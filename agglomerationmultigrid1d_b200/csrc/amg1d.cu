// libamg1d: C ABI (include/amg1d.h) + host-side driver of the B200 V-cycle.
//
// The V-cycle structure follows src/solvers.jl:19-50 of the reference; what each kernel computes is
// documented next to it in kernels_generic.cuh / kernels_fused.cuh.  Nothing here falls back to the
// CPU: every numerical operation is a kernel launch on the handle's stream.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#ifdef AMG1D_WITH_NCCL
#include <dlfcn.h>
#include <nccl.h>   // types and prototypes only: the library is dlopen'ed, never linked
#endif

#include "../../include/amg1d.h"
#include "kernels_generic.cuh"
#include "kernels_fused.cuh"
#include "kernels_multi.cuh"
#include "kernels_rows.cuh"
#include "direct_bcr.cuh"
#include "device_setup.cuh"
#include "halo_p2p.cuh"

#define AMG1D_VERSION 100
#define PAD_FRONT 64  // doubles in front of element 0 (ghost elements live at the end of them)
#define PAD_BACK 64
#define MULTI_SLOTS 8  // device scalars per column of the multi-column set (slot 0: ||b - A x||, 2: ||b||; the CG_*
                       // slots of amg1d_dev_pcg_multi up to CG_RZ_NEW = 7)
static_assert(MULTI_MAX_COLS == AMG1D_MAX_COLS, "kernels_multi.cuh and amg1d.h disagree on the column limit");

namespace {

std::string g_create_error;

struct DVec {
    double* raw = nullptr;
    double* p = nullptr;  // element 0
    int64_t len = 0;      // n * m
    bool in_arena = false;   // carved out of the handle's peer-mapped arena (halo_p2p.cuh): not freed on its own
};

// Scratch device allocation that is released on every exit path of an upload / download routine.
struct DevBuf {
    double* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(int64_t doubles) { return cudaMalloc((void**)&p, (size_t)(doubles > 0 ? doubles : 1) * 8); }
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
};

struct Level {
    bool set = false;
    int64_t n = 0;       // elements held by this rank (== n_glob unless the level is sharded)
    int64_t n_glob = 0;  // elements of the whole level
    int64_t start = 0;   // global index of local element 0
    int gl = 0, gr = 0;  // ghost elements on the left / right slab edge (sharded levels only)
    bool sharded = false;  // split into contiguous element slabs, one per rank
    bool present = true;   // this rank holds the level's operator (sharded, or rank 0)
    bool proxy = false;    // vectors only: a non-root rank's slab of the first gathered level
    double* mat_alloc = nullptr;
    int m = 0;
    int diag = 0;
    int K = 0;           // == md.K
    MatDesc md = {};     // structure class and tile-row offsets (layout.cuh)
    int64_t base_n = 0;  // sharded: elements per rank (the last rank also holds n_glob % nranks)
    // optional block-tridiagonal smoother operator S (overlapping Schwarz smoothers of CG levels,
    // src/smoother.jl:1-46): z = S r instead of z = Dinv r; stored like a level operator
    // flux operators G, D, C of the level as element-block arrays on the device (lo, di, up each), kept
    // between amg1d_set_level_flux / amg1d_coarsen_level and amg1d_finalize (device-side set-up)
    double* flux[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool smooth_tri = false;
    int dv_rec = 0;        // != 0: the stored Dinv is the device's own Gauss-Jordan inverse of A_di (adopt_device_dinv),
                           // the fused legs may recompute it in registers instead of streaming it; 2: no element
                           // of the level ever pivots (the legs skip the compare-and-swap chain)
    double* smat_alloc = nullptr;
    double* smat = nullptr;
    MatDesc smd = {};
    int64_t n_host = 0;  // reference vector length
    double* mat = nullptr;
    int64_t* perm = nullptr;  // device, n*m entries, or null
    // host copy of the blocks, kept only for small levels (coarsest-level factorisation)
    std::vector<double> h_lo, h_di, h_up;
    int64_t mat_bytes = 0;
    // translation-invariant level (amg1d_set_level_pattern): its n_head + 1 + n_tail distinct block sets
    // as a table tab[set][k] on the device, for the pattern-resident fused legs (PatOp, kernels_fused.cuh)
    double* pat = nullptr;
    int pat_head = 0, pat_tail = 0;
    std::vector<double> pat_host;   // host copy of the table (its interior row is the ParamOp of f_down_c / f_up_c)
};

struct Transfer {
    bool set = false;
    int64_t n_fine = 0, n_coarse = 0;
    int mf = 0, mc = 0;
    int64_t* parent = nullptr;  // device or null
    int64_t* cp = nullptr;      // device or null
    std::vector<int64_t> h_parent;  // host copy until finalize builds the child pointers
    int ratio = 1, shift = 0, base = 0, period = 0, n_head = 0, n_tail = 0;
    double* P0 = nullptr;
    double* P1 = nullptr;
    int64_t nblk = 0;
    bool single_parent_uniform = false;  // parent[e] = e / ratio, no P1
    bool closed = false;     // parent[e] = (e + shift) / ratio + base for every e (pattern or detected)
    bool fusable = false;    // closed, and every coarse element has a first P0-child (f_down's gather rule)
    int64_t p_first = 0;     // explicit blocks of a sharded level: global fine element of the first block kept
    int reach = 0;           // sharded two-parent transfers: fine ghost elements the restriction reads
    int64_t cover_extra = 0; // sharded: ghost elements right of the slab that own coarse elements of this rank
};

// One problem on the hierarchy: the resident problem, or one column of the multi-column set.  Every operation that
// reads or writes a vector, a buffer parity, a scalar slot or the reduction scratch is given the column it works on.
struct Column {
    struct Vecs { DVec x[2], b; int cur = 0; };   // x[cur]: the current iterate, x[1 - cur]: the other ping-pong buffer
    std::vector<Vecs> lv;          // [level]; a level this rank does not hold has none (column_alloc)
    double* scal = nullptr;        // device scalars (slot 0: ||b - A x||, 1: error, 2: ||b||, CG_* slots of the PCG)
    double* partial = nullptr;     // reduction scratch: partial_cap first-stage partial sums + 256 second-stage ones
    struct { DVec x, p, ap; } cg;  // level 0: CG solution, search direction, A p - allocated at the first CG call
};

// An instantiated V-cycle graph, keyed by the cycle parameters and the active columns (the resident cycle: mask 1)
struct GraphEntry {
    cudaGraphExec_t exec = nullptr;
    int pre = -1, post = -1, norm = -1, zero0 = -1;
    double alpha = 0.0;
    unsigned mask = 0;
    int64_t launches = 0;
    uint64_t stamp = 0;
};

}  // namespace

struct amg1d {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int n_levels = 0;
    std::vector<Level> L;
    std::vector<Transfer> T;
    bool finalized = false;
    std::string err;
    // work
    DVec scratch;          // residual scratch, max level size
    double* stage = nullptr;  // host-ordered staging for permuted levels
    int64_t stage_len = 0;
    int64_t partial_cap = 0;
    Column res;                // the resident problem (its 64 device scalars are its own allocation)
    bool norm_valid = false;   // res.scal[0] holds ||b - A x|| of the current level-0 iterate
    bool dev_problem = true;   // level 0's b / x still hold the device-resident problem (amg1d_dev_set_problem);
                               // cleared by the calls that stage through them (level-0 residual / smoother
                               // solve, amg1d_pcg) - the amg1d_dev_* calls then refuse to run on stale data
    double* h_scal = nullptr;  // pinned host scalars
    double* coarse_fac = nullptr;
    // options
    int opt_fused = 1, opt_graph = 1;
    int64_t opt_coarse_cta = 1024;
    int opt_compress = 1;         // drop structural zeros of the off-diagonal blocks (layout.cuh)
    int opt_pdl = 1;              // programmatic dependent launch between the fused kernels
    int opt_rows = 64;            // window of the row-per-thread fused legs (kernels_rows.cuh): 32, 64; 0 = off
    int opt_rows_rpt = 0;         // block rows per thread of those legs: 1, 2, 3; 0 = auto (rows_rpt() below)
    int opt_dvrec = 4;            // block-Jacobi inverses recomputed inside the fused legs of levels with blocks of at
                                  // least this size and at most 4 x 4 (0 = never; see adopt_device_dinv, leg_rec)
    int opt_dvrec_max = 4;        // ... and at most this size (option recompute_dinv_max, <= 5)
    int opt_dvreg = 0;            // 1: 4 x 4 DG legs keep the recomputed inverse in registers (f_down_dv / f_up_dv, 4 CTAs
                                  // per SM); 2: the 2 x 2 levels too
    int opt_pipe = 1;             // 1: 4 x 4 DG legs run as persistent CTAs that prefetch their next window with TMA bulk
                                  // copies (f_down_pp / f_up_pp, kernels_fused.cuh); 2: the 2 x 2 levels too; needs
                                  // recompute_dinv > 0
    int64_t opt_pipe_min = 500000;   // ... on levels with at least this many elements on this rank (option leg_pipeline_min;
                                  // measured, profiles/r03a_sweep_sizes.jsonl: 3 - 12 % per cycle from 2^20 elements up,
                                  // -2 % at 2^18, where the two ordinary stream dependencies around a persistent leg
                                  // cost more than the pipeline gains)
    int opt_pattern = 0;          // 1: levels given as patterns read their operator from the pattern table;
                                  // 2: and the interior CTAs of f_down / f_up take it as constant-bank operands
    // single-CTA coarse tail (f_tail): levels [tail_start, n_levels)
    int tail_start = -1;
    TailLevel* d_tail = nullptr;
    TailPlan tail_plan_ = {};
    std::vector<TailLevel> tail_host;   // d_tail without the vectors, which fill_tail patches in per column
    uint64_t tail_gen = 0;              // bumped by every build_tail
    GraphEntry graphs[4];               // graph cache of the resident problem's V-cycle
    uint64_t graph_clock = 0;
    int64_t launches_per_cycle = 0;
    // block-cyclic-reduction direct solvers: coarsest level (when it has more than AMG1D_BCR_MIN
    // elements) and, built on demand, any level asked for through amg1d_direct_solve
    BcrSolver coarse_bcr;
    std::vector<BcrSolver> direct;
    int64_t launch_counter = 0;
    int64_t device_bytes = 0;
    // per-kernel event profiling (option "profile"): one (start, stop) pair per launch of a leg
    int opt_profile = 0;
    struct Prof { std::vector<cudaEvent_t> ev; };
    std::vector<Prof> prof;   // index = level * 2 + leg (0 = down, 1 = up)
    // distributed (contiguous element slabs; SURVEY 8e)
    int rank = 0, nranks = 1;
    int ghost_depth = 4;          // elements per slab edge = max(nPre, nPost) + 1
    int64_t shard_min = 8192;     // a level is sharded while it has >= nranks * shard_min elements
    int gather_level = -1;        // first level that lives on rank 0 only (-1: single GPU)
#ifdef AMG1D_WITH_NCCL
    ncclComm_t comm = nullptr;
#endif
    // amg1d_vcycle_batch: copy-in / copy-out streams, double-buffered device staging of level-0 vectors, events
    struct Pipe {
        cudaStream_t s_in = nullptr, s_out = nullptr;
        double* st_b[2] = {nullptr, nullptr};
        double* st_x[2] = {nullptr, nullptr};
        double* st_o[2] = {nullptr, nullptr};
        cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_used[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr},
                    ev_out[2] = {nullptr, nullptr};
        int64_t len = 0;
    } pipe;
    // peer-memory halo exchange (halo_p2p.cuh): the vectors of the sharded levels and the receive counters live
    // in one arena that both slab neighbours map with CUDA IPC
    int opt_p2p = 1;
    struct P2P {
        bool on = false;
        char* arena = nullptr;
        int64_t bytes = 0, used = 0;
        char* peer[2] = {nullptr, nullptr};          // the arenas of rank - 1 / rank + 1, mapped here
        int n_ch = 0;                                // channels: 2 per sharded level
        unsigned long long* flags = nullptr;         // [side][channel] receive counters, at the start of the arena
        unsigned long long* epoch = nullptr;         // V-cycles enqueued so far (device)
        int* err = nullptr;                          // device: a spin timed out
        struct Nb { int64_t off[3] = {0, 0, 0}; int64_t n = 0; };   // byte offsets of x[0].p, x[1].p, b.p; owned n
        std::vector<Nb> nb[2];                       // per level, for the left / right neighbour
    } p2p;
    // multi-column resident problems (amg1d_dev_set_problems ...): columns of their own, apart from the resident problem
    struct Multi {
        std::vector<Column> col;                   // grown on demand, never shrunk
        int k = 0;                                 // columns of the current set (0: none)
        double* d_scal = nullptr;                  // MULTI_MAX_COLS x MULTI_SLOTS device scalars: col[c].scal is window c
        double* h_scal = nullptr;                  // pinned host copy
        TailLevel* d_tail = nullptr;               // MULTI_MAX_COLS x TAIL_MAXL descriptors of the single-CTA tail
        uint64_t tail_synced = ~0ull;              // tail_gen that d_tail was filled for
        bool norm_valid = false;                   // d_scal slot 0 of every column holds ||b - A x|| of its iterate
        bool rhs_consumed = false;                 // amg1d_dev_pcg_multi turned the right-hand sides into CG residuals
        int64_t launches_per_cycle = 0;
        int64_t pcg_launches = 0;                  // launches of the last PCG iteration outside the V-cycle
        GraphEntry graphs[4];
    } multi;
};

namespace {

int fail(amg1d* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(h, e_ == cudaErrorMemoryAllocation ? AMG1D_ERR_NOMEM : AMG1D_ERR_CUDA, \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

#define RET(expr)                \
    do {                         \
        int rc_ = (expr);        \
        if (rc_ != AMG1D_OK) return rc_; \
    } while (0)

int dev_alloc(amg1d* h, void** p, int64_t bytes) {
    if (bytes <= 0) bytes = 8;
    CK(cudaMalloc(p, (size_t)bytes));
    h->device_bytes += bytes;
    return AMG1D_OK;
}

int vec_alloc(amg1d* h, DVec& v, int64_t n, int m) {
    v.len = n * m;
    const int64_t total = PAD_FRONT + v.len + PAD_BACK;
    RET(dev_alloc(h, (void**)&v.raw, total * 8));
    CK(cudaMemsetAsync(v.raw, 0, (size_t)total * 8, h->stream));
    v.p = v.raw + PAD_FRONT;
    return AMG1D_OK;
}

void vec_free(DVec& v) {
    if (v.raw && !v.in_arena) cudaFree(v.raw);
    v.raw = v.p = nullptr;
}

inline int64_t arena_round(int64_t bytes) { return (bytes + 255) / 256 * 256; }

// a vector of a sharded level: carved out of the peer-mapped arena (zero-filled at allocation)
int vec_from_arena(amg1d* h, DVec& v, int64_t n, int m) {
    v.len = n * m;
    const int64_t bytes = arena_round((PAD_FRONT + v.len + PAD_BACK) * 8);
    if (h->p2p.used + bytes > h->p2p.bytes) return fail(h, AMG1D_ERR_STATE, "internal: halo arena overflow");
    v.raw = reinterpret_cast<double*>(h->p2p.arena + h->p2p.used);
    v.p = v.raw + PAD_FRONT;
    v.in_arena = true;
    h->p2p.used += bytes;
    return AMG1D_OK;
}

int64_t vec_bytes(const DVec& v) { return (PAD_FRONT + v.len + PAD_BACK) * 8; }

void vec_release(amg1d* h, DVec& v) {
    if (v.raw && !v.in_arena) h->device_bytes -= vec_bytes(v);
    vec_free(v);
}

// everything column_alloc gave col (not its scalars, which belong to their owner)
void column_free(amg1d* h, Column& col) {
    for (auto& v : col.lv) { vec_release(h, v.x[0]); vec_release(h, v.x[1]); vec_release(h, v.b); }
    col.lv.clear();
    if (col.partial) { cudaFree(col.partial); h->device_bytes -= (h->partial_cap + 256) * 8; col.partial = nullptr; }
    vec_release(h, col.cg.x); vec_release(h, col.cg.p); vec_release(h, col.cg.ap);
}

// What col still lacks: its vectors on every level this rank holds, with its reduction scratch, and with cg its level-0
// CG vectors.  Vectors of sharded levels come from the peer-mapped arena (in the order x[0], b, x[1] its neighbours
// expect); a proxy level holds no x[1].  A failure releases what this call took and clears the sticky CUDA error.
int column_alloc(amg1d* h, Column& col, bool cg) {
    const bool levels = col.lv.empty();
    int rc = AMG1D_OK;
    if (levels) {
        col.lv.resize((size_t)h->n_levels);
        for (int l = 0; l < h->n_levels && rc == AMG1D_OK; ++l) {
            const Level& lv = h->L[l];
            Column::Vecs& v = col.lv[(size_t)l];
            if (!lv.present && !lv.proxy) continue;
            const bool arena = lv.sharded && h->p2p.arena;
            for (DVec* d : {&v.x[0], &v.b, &v.x[1]})
                if (rc == AMG1D_OK && (d != &v.x[1] || lv.present))
                    rc = arena ? vec_from_arena(h, *d, lv.n, lv.m) : vec_alloc(h, *d, lv.n, lv.m);
        }
        if (rc == AMG1D_OK) rc = dev_alloc(h, (void**)&col.partial, (h->partial_cap + 256) * 8);
    }
    if (rc == AMG1D_OK && cg && !col.cg.x.raw)
        for (DVec* d : {&col.cg.x, &col.cg.p, &col.cg.ap})
            if (rc == AMG1D_OK) rc = vec_alloc(h, *d, h->L[0].n, h->L[0].m);
    if (rc != AMG1D_OK) {
        if (levels) column_free(h, col);
        else { vec_release(h, col.cg.x); vec_release(h, col.cg.p); vec_release(h, col.cg.ap); }
        cudaGetLastError();                      // an out-of-memory status must not surface at the next launch check
    }
    return rc;
}

inline dim3 gblock(int m) {
    int z = 256 / (AMG1D_TILE * m);
    if (z < 1) z = 1;
    return dim3(AMG1D_TILE, m, z);
}
inline unsigned ggrid(int64_t n, int m) {
    const int z = gblock(m).z;
    return (unsigned)((amg1d_tiles(n) + z - 1) / z);
}

#define LAUNCH_CHECK() CK(cudaGetLastError())

bool valid_level(amg1d* h, int l) { return h && l >= 0 && l < h->n_levels; }

TransferMap make_map(const Transfer& t) {
    TransferMap tm;
    tm.parent = t.parent;
    tm.cp = t.cp;
    tm.n_fine = t.n_fine;
    tm.n_coarse = t.n_coarse;
    tm.ratio = t.ratio;
    tm.shift = t.shift;
    tm.base = t.base;
    tm.period = t.period;
    tm.n_head = t.n_head;
    tm.n_tail = t.n_tail;
    return tm;
}

// closed-form version (no parent / child-pointer arrays): what the fused kernels take
TransferMap make_map_closed(const Transfer& t) {
    TransferMap tm = make_map(t);
    tm.parent = nullptr;
    tm.cp = nullptr;
    return tm;
}

// Transfer blocks as the kernels index them: by pattern position, or - explicit blocks - by GLOBAL fine element;
// a sharded level keeps only the blocks of its slab (p_first = first one kept), hence the bias.
inline const double* tp0(const Transfer& t) { return t.P0 ? t.P0 - t.p_first * (int64_t)(t.mf * t.mc) : nullptr; }
inline const double* tp1(const Transfer& t) { return t.P1 ? t.P1 - t.p_first * (int64_t)(t.mf * t.mc) : nullptr; }

// slab of rank r of a level with n_glob elements split over nranks: [start, start + n)
inline int64_t slab_start(int64_t n_glob, int nranks, int r) { return (n_glob / nranks) * r; }
inline int64_t slab_size(int64_t n_glob, int nranks, int r) {
    return n_glob / nranks + (r == nranks - 1 ? n_glob % nranks : 0);
}

#ifdef AMG1D_WITH_NCCL
// NCCL is resolved at run time (dlopen by SONAME) when a multi-GPU handle is created, so that a
// process that already loaded an NCCL (e.g. the one bundled with PyTorch) keeps using exactly that
// one, and single-GPU use never loads NCCL at all.  $AMG1D_NCCL_LIB overrides the library path.
struct NcclApi {
    void* lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclSend) Send = nullptr;
    decltype(&ncclRecv) Recv = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
};
NcclApi g_nccl;

const char* load_nccl() {
    if (g_nccl.lib) return nullptr;
    const char* env = getenv("AMG1D_NCCL_LIB");
    void* lib = env ? dlopen(env, RTLD_NOW | RTLD_LOCAL) : nullptr;
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
    if (!lib) return "cannot dlopen libnccl.so.2";
#define NSYM(field, name)                                                    \
    g_nccl.field = reinterpret_cast<decltype(g_nccl.field)>(dlsym(lib, name)); \
    if (!g_nccl.field) return "libnccl lacks " name;
    NSYM(GetUniqueId, "ncclGetUniqueId") NSYM(CommInitRank, "ncclCommInitRank")
    NSYM(CommDestroy, "ncclCommDestroy") NSYM(Send, "ncclSend") NSYM(Recv, "ncclRecv")
    NSYM(AllReduce, "ncclAllReduce") NSYM(AllGather, "ncclAllGather") NSYM(GroupStart, "ncclGroupStart") NSYM(GroupEnd, "ncclGroupEnd")
    NSYM(GetErrorString, "ncclGetErrorString")
#undef NSYM
    g_nccl.lib = lib;
    return nullptr;
}
#endif

// Block rows per thread of the row-per-thread legs on level l.  Measured on B200 (P8, 2^23 elements of 9 x 9
// blocks, profiles/r01d_*): with the operator streamed from HBM one row per thread (1152 resident threads
// per SM) is fastest - 3.72 / 3.87 ms per leg against 4.13 / 3.66 ms for three rows; with pattern-resident
// operators nothing waits for HBM any more and three rows per thread (fewer shared-memory reads per row)
// win: 3.16 / 2.84 ms against 3.39 / 3.55 ms.
int rows_rpt(const amg1d* h, int l) {
    if (h->opt_rows_rpt) return h->opt_rows_rpt;
    return h->opt_pattern && h->L[l].pat ? 3 : 1;
}

// 0: the fused legs of this level stream the stored inverse; 1 / 2: they invert A_di in registers (with / without pivots)
int leg_rec(const amg1d* h, const Level& lv, int mc = 0) {
    // measured on B200 (profiles/r02c_sweep_dvrec_*.jsonl): 4 x 4 DG blocks gain 4-5 % per leg (T level 0: 4.63 / 4.31
    // -> 4.43 / 4.12 ms); 5 x 5 blocks lose 10 % (the inversion's registers cost a resident CTA), 2 x 2 lose 5 %
    // bits 0-1: invert A_di in registers (1: with the pivot chain, 2: the level never pivots); bit 3: keep the inverse
    // in registers (option dinv_registers); bit 4: pipelined persistent leg (option leg_pipeline)
    int rec = (h->opt_dvrec > 0 && lv.dv_rec && lv.m >= h->opt_dvrec && lv.m <= h->opt_dvrec_max)
                  ? (lv.dv_rec | (h->opt_dvreg ? 8 : 0) | ((h->opt_pipe && lv.n >= h->opt_pipe_min) ? 16 : 0)) : 0;
    // option dinv_registers = 2: the 2 x 2 levels too, through the legs that keep the inverse in registers
    if (!rec && h->opt_dvrec > 0 && h->opt_dvreg >= 2 && lv.dv_rec && lv.m == 2 && fused_has_dv(lv.m, mc, lv.md.st, lv.diag))
        rec = lv.dv_rec | 8;
    // option leg_pipeline = 2: the 2 x 2 levels through the pipelined legs (which invert in registers as well)
    if (h->opt_dvrec > 0 && h->opt_pipe >= 2 && lv.n >= h->opt_pipe_min && lv.dv_rec && lv.m == 2 &&
        fused_has_pp(lv.m, mc, lv.md.st, lv.diag))
        rec = (rec & 8) | lv.dv_rec | 16;
    return rec;
}

// pattern-resident operator of level l (option pattern_resident = 1 and the level was given as a pattern)
PatOp make_pat(const amg1d* h, int l) {
    const Level& lv = h->L[l];
    PatOp po;
    po.tab = h->opt_pattern ? lv.pat : nullptr;
    po.n_glob = lv.n_glob;
    po.n_head = lv.pat_head;
    po.n_tail = lv.pat_tail;
    po.host_interior = (h->opt_pattern == 2 && lv.pat && !lv.pat_host.empty())
                           ? lv.pat_host.data() + (size_t)lv.pat_head * lv.K : nullptr;
    return po;
}

Slab make_slab(amg1d* h, int l) {
    Slab sl;
    const Level& lv = h->L[l];
    sl.gl = lv.gl;
    sl.gr = lv.gr;
    sl.e_off = lv.start;
    sl.c_off = 0;
    sl.nc = 0;
    if (l + 1 < h->n_levels) {
        const Level& lc = h->L[l + 1];
        // the coarse level is sharded too, or it is the gather level (slabs of its rhs are gathered to
        // rank 0 afterwards; on a single GPU this is simply the whole level)
        sl.c_off = lv.sharded ? slab_start(lc.n_glob, h->nranks, h->rank) : 0;
        sl.nc = lv.sharded ? slab_size(lc.n_glob, h->nranks, h->rank) : lc.n_glob;
    }
    return sl;
}

#ifdef AMG1D_WITH_NCCL
#define NCK(call)                                                                              \
    do {                                                                                       \
        ncclResult_t r_ = (call);                                                              \
        if (r_ != ncclSuccess)                                                                 \
            return fail(h, AMG1D_ERR_NCCL, "%s failed: %s (%s:%d)", #call, g_nccl.GetErrorString(r_), \
                        __FILE__, __LINE__);                                                   \
    } while (0)

// Exchange ghost_depth edge elements of a slab vector with both neighbour ranks.
// v points at local element 0; n = owned elements; m = block size.  A second vector (v2 != nullptr)
// travels in the same NCCL group: one communication kernel instead of two (the exchanges are latency
// bound: 4 x m doubles each way).
int op_halo(amg1d* h, double* v, int64_t n, int m, double* v2 = nullptr, int64_t n2 = 0, int m2 = 0) {
    NCK(g_nccl.GroupStart());
    for (int k = 0; k < 2; ++k) {
        double* p = k == 0 ? v : v2;
        if (!p) continue;
        const int64_t nn = k == 0 ? n : n2;
        const int mm = k == 0 ? m : m2;
        const int64_t cnt = (int64_t)h->ghost_depth * mm;
        if (h->rank > 0) {
            NCK(g_nccl.Send(p, cnt, ncclDouble, h->rank - 1, h->comm, h->stream));
            NCK(g_nccl.Recv(p - cnt, cnt, ncclDouble, h->rank - 1, h->comm, h->stream));
        }
        if (h->rank < h->nranks - 1) {
            NCK(g_nccl.Send(p + (nn - h->ghost_depth) * mm, cnt, ncclDouble, h->rank + 1, h->comm, h->stream));
            NCK(g_nccl.Recv(p + nn * mm, cnt, ncclDouble, h->rank + 1, h->comm, h->stream));
        }
    }
    NCK(g_nccl.GroupEnd());
    h->launch_counter++;
    return AMG1D_OK;
}

// rank r's slab of the gather level's right-hand side -> rank 0 (which owns the whole level)
int op_gather_rhs(amg1d* h, Column& col, int g) {
    Level& lg = h->L[g];
    double* b = col.lv[(size_t)g].b.p;
    NCK(g_nccl.GroupStart());
    if (h->rank == 0) {
        for (int r = 1; r < h->nranks; ++r)
            NCK(g_nccl.Recv(b + slab_start(lg.n_glob, h->nranks, r) * lg.m,
                            slab_size(lg.n_glob, h->nranks, r) * lg.m, ncclDouble, r, h->comm, h->stream));
    } else {
        NCK(g_nccl.Send(b, slab_size(lg.n_glob, h->nranks, h->rank) * lg.m, ncclDouble, 0, h->comm,
                        h->stream));
    }
    NCK(g_nccl.GroupEnd());
    h->launch_counter++;
    return AMG1D_OK;
}

// rank 0's solution of the gather level -> every rank's slab (with ghost elements)
int op_scatter_sol(amg1d* h, Column& col, int g) {
    Level& lg = h->L[g];
    Column::Vecs& v = col.lv[(size_t)g];
    const int gd = h->ghost_depth;
    NCK(g_nccl.GroupStart());
    if (h->rank == 0) {
        const double* x = v.x[v.cur].p;
        for (int r = 1; r < h->nranks; ++r) {
            const int64_t e0 = slab_start(lg.n_glob, h->nranks, r) - gd;
            const int64_t e1 = slab_start(lg.n_glob, h->nranks, r) + slab_size(lg.n_glob, h->nranks, r) +
                               (r < h->nranks - 1 ? gd : 0);
            NCK(g_nccl.Send(x + e0 * lg.m, (e1 - e0) * lg.m, ncclDouble, r, h->comm, h->stream));
        }
    } else {
        const int64_t cnt = (slab_size(lg.n_glob, h->nranks, h->rank) + gd +
                             (h->rank < h->nranks - 1 ? gd : 0)) * lg.m;
        NCK(g_nccl.Recv(v.x[0].p - (int64_t)gd * lg.m, cnt, ncclDouble, 0, h->comm, h->stream));
    }
    NCK(g_nccl.GroupEnd());
    h->launch_counter++;
    return AMG1D_OK;
}

// col.scal[slot] currently holds a local sum (of squares with take_sqrt): make it the global sum (2-norm)
__global__ void k_sqrt_inplace(double* v, int slot) { v[slot] = sqrt(v[slot]); }
int op_allreduce_max(amg1d* h, double* dptr, int count) {
    NCK(g_nccl.AllReduce(dptr, dptr, (size_t)count, ncclDouble, ncclMax, h->comm, h->stream));
    return AMG1D_OK;
}
int op_allreduce_norm(amg1d* h, Column& col, int slot, bool take_sqrt) {
    NCK(g_nccl.AllReduce(col.scal + slot, col.scal + slot, 1, ncclDouble, ncclSum, h->comm, h->stream));
    h->launch_counter++;
    if (!take_sqrt) return AMG1D_OK;
    k_sqrt_inplace<<<1, 1, 0, h->stream>>>(col.scal, slot);
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

// ---- peer-memory halo exchange (halo_p2p.cuh) ------------------------------------------------------------
#define AMG1D_P2P_MAXL 48
struct P2PXchg {                 // what every rank publishes about its arena
    cudaIpcMemHandle_t hnd;
    int32_t ok, n_sharded;
    int64_t off[AMG1D_P2P_MAXL][3];
    int64_t n[AMG1D_P2P_MAXL];
};

// all-gather of a small host struct through NCCL (device staging)
int nccl_allgather_host(amg1d* h, const void* mine, void* all, size_t bytes) {
    DevBuf snd, rcv;
    CK(snd.alloc((int64_t)(bytes + 7) / 8));
    CK(rcv.alloc((int64_t)(bytes * h->nranks + 7) / 8));
    CK(cudaMemcpyAsync(snd.p, mine, bytes, cudaMemcpyHostToDevice, h->stream));
    NCK(g_nccl.AllGather(snd.p, rcv.p, bytes, ncclChar, h->comm, h->stream));
    CK(cudaMemcpyAsync(all, rcv.p, bytes * h->nranks, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AMG1D_OK;
}

// one arena for the receive counters and the vectors of every sharded level (amg1d_finalize, before the vectors)
int p2p_alloc_arena(amg1d* h) {
    amg1d::P2P& P = h->p2p;
    int n_sh = 0;
    int64_t total = 0;
    for (int l = 0; l < h->n_levels; ++l) {
        const Level& lv = h->L[l];
        if (!lv.sharded) continue;
        ++n_sh;
        total += 3 * arena_round((PAD_FRONT + lv.n * lv.m + PAD_BACK) * 8);
    }
    if (n_sh == 0 || n_sh > AMG1D_P2P_MAXL) return AMG1D_OK;
    P.n_ch = 2 * n_sh;
    const int64_t flag_bytes = arena_round((int64_t)2 * P.n_ch * 8);
    total += flag_bytes;
    if (cudaMalloc((void**)&P.arena, (size_t)total) != cudaSuccess) { cudaGetLastError(); P.arena = nullptr; return AMG1D_OK; }
    CK(cudaMemsetAsync(P.arena, 0, (size_t)total, h->stream));
    h->device_bytes += total;
    P.bytes = total;
    P.used = flag_bytes;
    P.flags = reinterpret_cast<unsigned long long*>(P.arena);
    return AMG1D_OK;
}

void p2p_close(amg1d* h) {
    amg1d::P2P& P = h->p2p;
    for (int s = 0; s < 2; ++s)
        if (P.peer[s]) { cudaIpcCloseMemHandle(P.peer[s]); P.peer[s] = nullptr; }
    P.on = false;
}

// exchange the arena handles and map both neighbours' arenas; every rank takes the same decision
int p2p_connect(amg1d* h, Column& col) {
    amg1d::P2P& P = h->p2p;
    if (!P.arena) return AMG1D_OK;
    P2PXchg mine;
    memset(&mine, 0, sizeof mine);
    mine.ok = cudaIpcGetMemHandle(&mine.hnd, P.arena) == cudaSuccess ? 1 : 0;
    if (!mine.ok) cudaGetLastError();
    for (int l = 0; l < h->n_levels && l < AMG1D_P2P_MAXL; ++l) {
        const Level& lv = h->L[l];
        if (!lv.sharded) continue;
        ++mine.n_sharded;
        const Column::Vecs& cv = col.lv[(size_t)l];
        const DVec* v[3] = {&cv.x[0], &cv.x[1], &cv.b};
        for (int k = 0; k < 3; ++k) {
            if (!v[k]->in_arena) mine.ok = 0;
            mine.off[l][k] = reinterpret_cast<const char*>(v[k]->p) - P.arena;
        }
        mine.n[l] = lv.n;
    }
    std::vector<P2PXchg> all((size_t)h->nranks);
    RET(nccl_allgather_host(h, &mine, all.data(), sizeof mine));
    int good = 1;
    for (const auto& x : all) good = good && x.ok && x.n_sharded == mine.n_sharded;
    const int nbr[2] = {h->rank - 1, h->rank + 1};
    if (good)
        for (int s = 0; s < 2; ++s) {
            if (nbr[s] < 0 || nbr[s] >= h->nranks) continue;
            void* ptr = nullptr;
            if (cudaIpcOpenMemHandle(&ptr, all[(size_t)nbr[s]].hnd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                good = 0;
                break;
            }
            P.peer[s] = static_cast<char*>(ptr);
            P.nb[s].assign((size_t)h->n_levels, amg1d::P2P::Nb());
            for (int l = 0; l < h->n_levels && l < AMG1D_P2P_MAXL; ++l) {
                for (int k = 0; k < 3; ++k) P.nb[s][(size_t)l].off[k] = all[(size_t)nbr[s]].off[l][k];
                P.nb[s][(size_t)l].n = all[(size_t)nbr[s]].n[l];
            }
        }
    std::vector<int32_t> votes((size_t)h->nranks);
    const int32_t vote = good;
    RET(nccl_allgather_host(h, &vote, votes.data(), sizeof vote));
    for (int32_t v : votes) good = good && v;
    if (!good) { p2p_close(h); return AMG1D_OK; }            // the NCCL halo path keeps working on the same vectors
    DevBuf tmp;
    if (!P.epoch) {
        RET(dev_alloc(h, (void**)&P.epoch, 64));
        CK(cudaMemsetAsync(P.epoch, 0, 64, h->stream));
        P.err = reinterpret_cast<int*>(P.epoch + 4);
    }
    P.on = true;
    return AMG1D_OK;
}

unsigned long long* p2p_my_flag(amg1d* h, int side, int ch) {
    const int nbr = side == 0 ? h->rank - 1 : h->rank + 1;
    return (nbr < 0 || nbr >= h->nranks) ? nullptr : h->p2p.flags + side * h->p2p.n_ch + ch;
}

// push the edges of col's vector `vec` (0 / 1: x buffers, 2: b) on level l - and optionally of its vector vec2 on level
// l2 - on channel ch
int op_p2p_push(amg1d* h, Column& col, int ch, int l, int vec, int l2 = -1, int vec2 = 0) {
    amg1d::P2P& P = h->p2p;
    HaloPush a;
    memset(&a, 0, sizeof a);
    a.gd = h->ghost_depth;
    const int lv_[2] = {l, l2}, vc_[2] = {vec, vec2};
    for (int p = 0; p < 2; ++p) {
        if (lv_[p] < 0) continue;
        Level& lv = h->L[lv_[p]];
        const Column::Vecs& cv = col.lv[(size_t)lv_[p]];
        const DVec& v = vc_[p] == 2 ? cv.b : cv.x[vc_[p]];
        a.src[p] = v.p;
        a.n[p] = lv.n;
        a.m[p] = lv.m;
        if (P.peer[0]) {
            const amg1d::P2P::Nb& nb = P.nb[0][(size_t)lv_[p]];
            a.dst_left[p] = reinterpret_cast<double*>(P.peer[0] + nb.off[vc_[p]]) + nb.n * lv.m;
        }
        if (P.peer[1]) {
            const amg1d::P2P::Nb& nb = P.nb[1][(size_t)lv_[p]];
            a.dst_right[p] = reinterpret_cast<double*>(P.peer[1] + nb.off[vc_[p]]) - (int64_t)a.gd * lv.m;
        }
    }
    // I am the RIGHT neighbour of rank - 1 (its counters of side 1) and the LEFT neighbour of rank + 1 (side 0)
    if (P.peer[0]) a.flag_left = reinterpret_cast<unsigned long long*>(P.peer[0]) + 1 * P.n_ch + ch;
    if (P.peer[1]) a.flag_right = reinterpret_cast<unsigned long long*>(P.peer[1]) + 0 * P.n_ch + ch;
    k_halo_push<<<1, 128, 0, h->stream>>>(a);
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

// elements a channel receives per cycle and side: ghost_depth of the iterate (+ ghost_depth of the coarse rhs on a
// down-leg channel whose coarse level is sharded too)
unsigned long long p2p_quantum(const amg1d* h, int ch) {
    const int l = ch / 2;
    const bool down = (ch & 1) == 0;
    return (unsigned long long)h->ghost_depth * ((down && l + 1 < h->n_levels && h->L[l + 1].sharded) ? 2 : 1);
}

int op_p2p_begin_cycle(amg1d* h) {
    amg1d::P2P& P = h->p2p;
    k_epoch_wait<<<1, 1, 0, h->stream>>>(P.epoch, p2p_my_flag(h, 0, 1), p2p_my_flag(h, 1, 1), p2p_quantum(h, 1),
                                         P.err);                                                    // channel 1 = U_0
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

// neighbour-side addresses of a level's vector: slot of MY element 0 in the left neighbour (its right ghosts) and of
// MY element n - gd in the right neighbour (its left ghosts)
void p2p_peer_slots(amg1d* h, int level, int vec, double** left, double** right) {
    amg1d::P2P& P = h->p2p;
    const Level& lv = h->L[level];
    *left = *right = nullptr;
    if (P.peer[0]) {
        const amg1d::P2P::Nb& nb = P.nb[0][(size_t)level];
        *left = reinterpret_cast<double*>(P.peer[0] + nb.off[vec]) + nb.n * lv.m;
    }
    if (P.peer[1]) {
        const amg1d::P2P::Nb& nb = P.nb[1][(size_t)level];
        *right = reinterpret_cast<double*>(P.peer[1] + nb.off[vec]) - (int64_t)h->ghost_depth * lv.m;
    }
}

// The exchange of one leg of sharded level l as the fused kernels perform it themselves (halo_p2p.cuh: HaloLeg).
// out_vec: the x buffer the leg writes (its edges go to the neighbours) or -1: no push from inside the kernel.
HaloLeg make_halo_leg(amg1d* h, int l, bool down, int out_vec) {
    HaloLeg hl;
    memset(&hl, 0, sizeof hl);
    amg1d::P2P& P = h->p2p;
    if (!P.on || !h->L[l].sharded) return hl;
    hl.on = 1;
    hl.gd = h->ghost_depth;
    hl.epoch = P.epoch;
    hl.err = P.err;
    const bool coarse_sharded = l + 1 < h->n_levels && h->L[l + 1].sharded;
    int wch[2] = {-1, -1};
    if (down) { if (l > 0) wch[0] = 2 * (l - 1); }               // rhs ghosts: the finer level's down-leg channel
    else { wch[0] = 2 * l; if (coarse_sharded) wch[1] = 2 * (l + 1) + 1; }   // pre-smoothed ghosts; coarse correction
    for (int i = 0; i < 2; ++i) {
        if (wch[i] < 0) continue;
        hl.w_left[i] = p2p_my_flag(h, 0, wch[i]);
        hl.w_right[i] = p2p_my_flag(h, 1, wch[i]);
        hl.wq[i] = p2p_quantum(h, wch[i]);
        hl.wlag[i] = 0;
    }
    if (out_vec >= 0) {
        const int ch = down ? 2 * l : 2 * l + 1;
        p2p_peer_slots(h, l, out_vec, &hl.x_left, &hl.x_right);
        if (down && coarse_sharded) p2p_peer_slots(h, l + 1, 2, &hl.c_left, &hl.c_right);
        if (P.peer[0]) hl.f_left = reinterpret_cast<unsigned long long*>(P.peer[0]) + 1 * P.n_ch + ch;
        if (P.peer[1]) hl.f_right = reinterpret_cast<unsigned long long*>(P.peer[1]) + 0 * P.n_ch + ch;
        hl.nc = make_slab(h, l).nc;
    }
    return hl;
}

// the same waits as stand-alone kernels (legs that are not f_down / f_up)
int op_p2p_wait_for(amg1d* h, const HaloLeg& hl) {
    for (int i = 0; i < 2; ++i) {
        if (!hl.w_left[i] && !hl.w_right[i]) continue;
        k_halo_wait<<<1, 1, 0, h->stream>>>(hl.w_left[i], hl.w_right[i], hl.epoch, hl.wlag[i], hl.wq[i], hl.err);
        h->launch_counter++;
        LAUNCH_CHECK();
    }
    return AMG1D_OK;
}
#else
int op_p2p_push(amg1d* h, Column&, int, int, int, int = -1, int = 0) { return fail(h, AMG1D_ERR_UNSUPPORTED, "built without NCCL"); }
int op_p2p_begin_cycle(amg1d* h) { return fail(h, AMG1D_ERR_UNSUPPORTED, "built without NCCL"); }
HaloLeg make_halo_leg(amg1d*, int, bool, int) { HaloLeg hl; memset(&hl, 0, sizeof hl); return hl; }
int op_p2p_wait_for(amg1d* h, const HaloLeg&) { return fail(h, AMG1D_ERR_UNSUPPORTED, "built without NCCL"); }
int op_halo(amg1d* h, double*, int64_t, int, double* = nullptr, int64_t = 0, int = 0) { return fail(h, AMG1D_ERR_UNSUPPORTED, "built without NCCL"); }
int op_gather_rhs(amg1d* h, Column&, int) { return fail(h, AMG1D_ERR_UNSUPPORTED, "built without NCCL"); }
int op_scatter_sol(amg1d* h, Column&, int) { return fail(h, AMG1D_ERR_UNSUPPORTED, "built without NCCL"); }
int op_allreduce_norm(amg1d* h, Column&, int, bool) { return fail(h, AMG1D_ERR_UNSUPPORTED, "built without NCCL"); }
int op_allreduce_max(amg1d* h, double*, int) { return fail(h, AMG1D_ERR_UNSUPPORTED, "built without NCCL"); }
#endif

// ---- elementary enqueued operations ---------------------------------------------------------------
int op_apply(amg1d* h, int l, const double* b, const double* x, double* out, int mode);

int op_sweep(amg1d* h, int l, const double* b, const double* xin, double* xout, double alpha,
             int zero_guess) {
    Level& lv = h->L[l];
    if (lv.smooth_tri) {
        // r = b - A x into the scratch vector (its ghost elements stay zero), then x + alpha S r
        if (zero_guess) CK(cudaMemcpyAsync(h->scratch.p, b, (size_t)lv.n * lv.m * 8, cudaMemcpyDeviceToDevice, h->stream));
        else RET(op_apply(h, l, b, xin, h->scratch.p, 1));
        g_apply_tri_smoother<<<ggrid(lv.n, lv.m), gblock(lv.m), 0, h->stream>>>(
            lv.smat, lv.smd, h->scratch.p, zero_guess ? nullptr : xin, xout, lv.n, alpha);
        h->launch_counter++;
        LAUNCH_CHECK();
        return AMG1D_OK;
    }
    if (h->opt_fused && fused_sweep(lv.md, lv.mat, b, xin, xout, lv.n, alpha, zero_guess, h->stream)) {
        h->launch_counter++;
        LAUNCH_CHECK();
        return AMG1D_OK;
    }
    const dim3 blk = gblock(lv.m);
    const size_t sm = (size_t)blk.z * lv.m * AMG1D_TILE * sizeof(double);
    g_sweep<<<ggrid(lv.n, lv.m), blk, sm, h->stream>>>(lv.mat, lv.md, b, xin, xout, lv.n, alpha,
                                                        zero_guess);
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

int op_apply(amg1d* h, int l, const double* b, const double* x, double* out, int mode) {
    Level& lv = h->L[l];
    g_apply<<<ggrid(lv.n, lv.m), gblock(lv.m), 0, h->stream>>>(lv.mat, lv.md, b, x, out, lv.n, mode);
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

int op_restrict(amg1d* h, int l, const double* rf, double* rc) {
    Transfer& t = h->T[l];
    const int64_t total = t.n_coarse * t.mc;
    g_restrict<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(make_map(t), t.mf, t.mc, t.P0,
                                                                       t.P1, rf, rc);
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

int op_prolong(amg1d* h, int l, const double* xc, double* xf, int add) {
    Transfer& t = h->T[l];
    const int64_t total = t.n_fine * t.mf;
    g_prolong<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(make_map(t), t.mf, t.mc, t.P0,
                                                                      t.P1, xc, xf, add);
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

int op_coarse(amg1d* h, const double* b, double* x) {
    Level& lv = h->L[h->n_levels - 1];
    if (h->coarse_bcr.ready()) {             // parallel cyclic reduction (direct_bcr.cuh)
        CK(h->coarse_bcr.solve(b, x, h->stream, &h->launch_counter));
        return AMG1D_OK;
    }
    g_coarse_solve<<<1, 32, 2 * lv.m * sizeof(double), h->stream>>>(h->coarse_fac, lv.m, lv.n, b, x);
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

// col's slot <- || a - c ||_2 (c may be null)
int op_norm(amg1d* h, Column& col, const double* a, const double* c, int64_t n, int slot) {
    int nb = (int)std::min<int64_t>(AMG1D_RED_BLOCKS, (n + AMG1D_RED_THREADS - 1) / AMG1D_RED_THREADS);
    if (nb < 1) nb = 1;
    k_sqdiff_partial<<<nb, AMG1D_RED_THREADS, 0, h->stream>>>(a, c, n, col.partial);
    k_reduce_final<<<1, AMG1D_RED_THREADS, 0, h->stream>>>(col.partial, nb, col.scal, slot,
                                                           h->nranks > 1 ? 0 : 1);
    h->launch_counter += 2;
    LAUNCH_CHECK();
    if (h->nranks > 1) RET(op_allreduce_norm(h, col, slot, true));
    return AMG1D_OK;
}

// col's slot <- sum col.partial[0..np), square-rooted with take_sqrt, summed over the ranks in the sharded case; long
// arrays go through a second stage of 256 partial sums
int op_reduce_partials(amg1d* h, Column& col, int64_t np, int slot, bool take_sqrt) {
    const double* src = col.partial;
    if (np > 8192) {
        double* stage2 = col.partial + h->partial_cap;   // 256 extra slots behind the first stage
        k_sum_partial<<<256, AMG1D_RED_THREADS, 0, h->stream>>>(col.partial, np, stage2);
        h->launch_counter++;
        src = stage2;
        np = 256;
    }
    k_reduce_final<<<1, AMG1D_RED_THREADS, 0, h->stream>>>(src, (int)np, col.scal, slot,
                                                           take_sqrt && h->nranks == 1 ? 1 : 0);
    h->launch_counter++;
    LAUNCH_CHECK();
    if (h->nranks > 1) RET(op_allreduce_norm(h, col, slot, take_sqrt));
    return AMG1D_OK;
}

// || b - A x ||_2 of col on level l into its slot
int op_resnorm(amg1d* h, Column& col, int l, int slot) {
    Level& lv = h->L[l];
    Column::Vecs& v = col.lv[(size_t)l];
    if (lv.sharded) RET(op_halo(h, v.x[v.cur].p, lv.n, lv.m));
    if (h->opt_fused) {
        int nb = 0;
        if (fused_resnorm(lv.md, lv.mat, v.b.p, v.x[v.cur].p, lv.n, col.partial, h->partial_cap, &nb,
                          h->stream)) {
            h->launch_counter++;
            LAUNCH_CHECK();
            return op_reduce_partials(h, col, nb, slot, true);
        }
    }
    RET(op_apply(h, l, v.b.p, v.x[v.cur].p, h->scratch.p, 1));
    return op_norm(h, col, h->scratch.p, nullptr, lv.n * lv.m, slot);
}

// col's slot <- a . c over the owned entries
int op_dot(amg1d* h, Column& col, const double* a, const double* c, int64_t n, int slot) {
    int nb = (int)std::min<int64_t>(AMG1D_RED_BLOCKS, (n + AMG1D_RED_THREADS - 1) / AMG1D_RED_THREADS);
    if (nb < 1) nb = 1;
    k_dot_partial<<<nb, AMG1D_RED_THREADS, 0, h->stream>>>(a, c, n, col.partial);
    h->launch_counter++;
    LAUNCH_CHECK();
    return op_reduce_partials(h, col, nb, slot, false);
}

// y = A x on level l (x must carry valid ghost elements), col's slot <- x . y when slot >= 0
int op_matvec_dot(amg1d* h, Column& col, int l, double* x, double* y, int slot) {
    Level& lv = h->L[l];
    if (lv.sharded) RET(op_halo(h, x, lv.n, lv.m));
    int nb = 0;
    if (h->opt_fused && fused_matvec_dot(lv.md, lv.mat, x, y, lv.n, slot >= 0 ? col.partial : nullptr,
                                         h->partial_cap, &nb, h->stream)) {
        h->launch_counter++;
        LAUNCH_CHECK();
        return slot >= 0 ? op_reduce_partials(h, col, nb, slot, false) : AMG1D_OK;
    }
    RET(op_apply(h, l, nullptr, x, y, 0));
    return slot >= 0 ? op_dot(h, col, x, y, lv.n * lv.m, slot) : AMG1D_OK;
}

int prof_mark(amg1d* h, int level, int leg) {
    if (!h->opt_profile) return AMG1D_OK;
    if (h->prof.size() < (size_t)h->n_levels * 2) h->prof.resize((size_t)h->n_levels * 2);
    cudaEvent_t ev;
    CK(cudaEventCreate(&ev));
    CK(cudaEventRecord(ev, h->stream));
    h->prof[level * 2 + leg].ev.push_back(ev);
    return AMG1D_OK;
}

// ---- the V-cycle (src/solvers.jl:19-50) ------------------------------------------------------------
// Down leg of level l: nPre sweeps (zero guess on l > 0), residual, restriction into level l+1's rhs.
int leg_down(amg1d* h, Column& col, int l, int nPre, double alpha, bool zero0) {
    Level& lv = h->L[l];
    Transfer& t = h->T[l];
    Level& lc = h->L[l + 1];
    Column::Vecs& v = col.lv[(size_t)l];
    Column::Vecs& vc = col.lv[(size_t)l + 1];
    const bool zero = l > 0 || zero0;         // zero0: level 0 starts from a zero guess too (ldiv!, PCG)
    if (zero) v.cur = 0;
    RET(prof_mark(h, l, 0));
    // ghosts of the incoming iterate (peer-memory mode: they arrived with the last up leg's push, or with
    // amg1d_dev_set_problem's exchange)
    if (lv.sharded && !zero && !h->p2p.on) RET(op_halo(h, v.x[v.cur].p, lv.n, lv.m));
    // fused: nPre sweeps + residual + restriction in one pass over the operator
    if (h->opt_fused && t.fusable && !lv.smooth_tri) {
        const int ob = zero ? 0 : 1 - v.cur;
        cudaError_t le = cudaSuccess;
        const bool p2p = h->p2p.on && lv.sharded;
        // peer-memory exchange done by the leg itself: wait for the rhs ghosts, push the pre-smoothed edges + coarse rhs
        const HaloLeg hl = p2p ? make_halo_leg(h, l, true, ob) : HaloLeg();
        int fr = fused_down(lv.md, t.mc, make_map_closed(t), nPre, zero, lv.mat, make_pat(h, l), v.b.p, v.x[v.cur].p,
                            v.x[ob].p, tp0(t), tp1(t), vc.b.p, lv.n, lv.n + (lv.gr ? t.cover_extra : 0),
                            alpha, make_slab(h, l), h->stream, h->opt_pdl != 0, &le, leg_rec(h, lv, t.mc), hl);
        if (fr == FUSED_NA && h->opt_rows) {    // large blocks: one thread per block row; exchange by stand-alone kernels
            if (p2p) RET(op_p2p_wait_for(h, hl));
            fr = rows_down(lv.md, t.mc, make_map_closed(t), nPre, zero, lv.mat, make_pat(h, l), v.b.p, v.x[v.cur].p,
                           v.x[ob].p, tp0(t), tp1(t), vc.b.p, lv.n, lv.n + (lv.gr ? t.cover_extra : 0), alpha,
                           make_slab(h, l), h->opt_rows, rows_rpt(h, l), h->stream, h->opt_pdl != 0, &le);
            if (fr == FUSED_OK && p2p) {
                if (lc.sharded) RET(op_p2p_push(h, col, 2 * l, l, ob, l + 1, 2));
                else RET(op_p2p_push(h, col, 2 * l, l, ob));
            }
        }
        if (fr == FUSED_ERR) return fail(h, AMG1D_ERR_CUDA, "f_down launch failed on level %d: %s", l, cudaGetErrorString(le));
        if (fr == FUSED_OK) {
            v.cur = ob;
            h->launch_counter++;
            LAUNCH_CHECK();
            RET(prof_mark(h, l, 0));
            return AMG1D_OK;
        }
    }
    if (lv.sharded)
        return fail(h, AMG1D_ERR_UNSUPPORTED, "level %d: sharded levels need the fused kernels "
                    "(a block size / transfer with a fused leg, closed-form transfer, option fused = 1)", l);
    if (zero && nPre == 0) CK(cudaMemsetAsync(v.x[0].p, 0, (size_t)v.x[0].len * 8, h->stream));
    for (int s = 0; s < nPre; ++s) {
        if (zero && s == 0) {
            RET(op_sweep(h, l, v.b.p, v.x[0].p, v.x[0].p, alpha, 1));  // x = alpha Dinv b
        } else {
            RET(op_sweep(h, l, v.b.p, v.x[v.cur].p, v.x[1 - v.cur].p, alpha, 0));
            v.cur = 1 - v.cur;
        }
    }
    if (h->opt_fused && t.single_parent_uniform &&
        fused_residual_restrict(lv.md, t.mc, make_map_closed(t), lv.mat, v.b.p, v.x[v.cur].p, t.P0,
                                vc.b.p, lv.n, h->stream)) {
        h->launch_counter++;
        LAUNCH_CHECK();
    } else {
        RET(op_apply(h, l, v.b.p, v.x[v.cur].p, h->scratch.p, 1));
        RET(op_restrict(h, l, h->scratch.p, vc.b.p));
    }
    return prof_mark(h, l, 0);
}

// Up leg of level l: x += L x_c, nPost sweeps; optionally ||b - A x|| of the result (level 0).
int leg_up(amg1d* h, Column& col, int l, int nPost, double alpha, bool fuse_norm, bool* norm_done, bool* halo_pushed) {
    *halo_pushed = false;
    Level& lv = h->L[l];
    Transfer& t = h->T[l];
    Column::Vecs& v = col.lv[(size_t)l];
    Column::Vecs& vc = col.lv[(size_t)l + 1];
    RET(prof_mark(h, l, 1));
    if (h->opt_fused && t.fusable && !lv.smooth_tri) {
        int nb = 0;
        cudaError_t le = cudaSuccess;
        const bool p2p = h->p2p.on && lv.sharded;
        // Level 0's edges are pushed from inside the kernel only if the leg writes buffer 0, where the next cycle
        // reads them (a zero-guess cycle ends in buffer 1 and is copied over: enqueue_vcycle pushes after that copy)
        const int ob = 1 - v.cur;
        const bool push_inside = l > 0 || ob == 0;
        const HaloLeg hl = p2p ? make_halo_leg(h, l, false, push_inside ? ob : -1) : HaloLeg();
        int fr = fused_up(lv.md, t.mc, make_map_closed(t), nPost, lv.mat, make_pat(h, l), v.b.p, v.x[v.cur].p,
                          v.x[1 - v.cur].p, tp0(t), tp1(t), vc.x[vc.cur].p, lv.n, alpha,
                          fuse_norm ? col.partial : nullptr, h->partial_cap, &nb, make_slab(h, l),
                          h->stream, h->opt_pdl != 0, &le, leg_rec(h, lv, t.mc), hl);
        if (fr == FUSED_OK && p2p && push_inside) *halo_pushed = true;
        if (fr == FUSED_NA && h->opt_rows) {
            if (p2p) RET(op_p2p_wait_for(h, hl));
            fr = rows_up(lv.md, t.mc, make_map_closed(t), nPost, lv.mat, make_pat(h, l), v.b.p, v.x[v.cur].p,
                         v.x[1 - v.cur].p, tp0(t), tp1(t), vc.x[vc.cur].p, lv.n, alpha,
                         fuse_norm ? col.partial : nullptr, h->partial_cap, &nb, make_slab(h, l), h->opt_rows,
                         rows_rpt(h, l), h->stream, h->opt_pdl != 0, &le);
        }
        if (fr == FUSED_ERR) return fail(h, AMG1D_ERR_CUDA, "f_up launch failed on level %d: %s", l, cudaGetErrorString(le));
        if (fr == FUSED_OK) {
            v.cur = 1 - v.cur;
            h->launch_counter++;
            LAUNCH_CHECK();
            RET(prof_mark(h, l, 1));
            if (fuse_norm) {
                RET(op_reduce_partials(h, col, nb, 0, true));
                *norm_done = true;
            }
            return AMG1D_OK;
        }
    }
    if (lv.sharded)
        return fail(h, AMG1D_ERR_UNSUPPORTED, "level %d: sharded levels need the fused kernels", l);
    RET(op_prolong(h, l, vc.x[vc.cur].p, v.x[v.cur].p, 1));
    for (int s = 0; s < nPost; ++s) {
        RET(op_sweep(h, l, v.b.p, v.x[v.cur].p, v.x[1 - v.cur].p, alpha, 0));
        v.cur = 1 - v.cur;
    }
    return prof_mark(h, l, 1);
}

int enqueue_vcycle(amg1d* h, Column& col, int nPre, int nPost, double alpha, bool want_norm, bool zero0) {
    const int nl = h->n_levels;
    const int g = h->gather_level;          // -1 on a single GPU: every level is local
    bool norm_done = false;
    if (g >= 0) {
        int need = std::max(nPre, nPost) + 1;         // one halo exchange serves a whole fused leg
        for (int l = 0; l < nl - 1; ++l)
            if (h->L[l].sharded) need = std::max(need, std::max(nPre, nPost) + 1 + h->T[l].reach);
        if (need > h->ghost_depth)
            return fail(h, AMG1D_ERR_ARG, "nPre / nPost need ghost_depth >= %d (option \"ghost_depth\", "
                        "before the first level is set)", need);
    }
    // levels [ts, nl) run inside the single-CTA tail kernel (rank 0 holds them; ts > gather level)
    const int ts = (h->tail_start > 0 && h->L[h->tail_start].present) ? h->tail_start : nl;
    const bool p2p = g >= 0 && h->p2p.on;       // slab edges through peer memory (halo_p2p.cuh) instead of NCCL
    bool u0_pushed = false;
    if (p2p) RET(op_p2p_begin_cycle(h));
    // ---- down ----
    for (int l = 0; l < nl - 1 && l < ts; ++l) {
        Level& lv = h->L[l];
        if (!lv.present) break;                       // ranks > 0 stop at the gather level
        RET(leg_down(h, col, l, nPre, alpha, zero0));
        if (lv.sharded) {
            Level& lc = h->L[l + 1];
            Column::Vecs& v = col.lv[(size_t)l];
            // ghosts of the pre-smoothed iterate (for the up leg) and of the coarse rhs, in one exchange
            if (p2p) {                    // the leg exchanged its edges itself (leg_down)
                if (!lc.sharded) RET(op_gather_rhs(h, col, l + 1));        // slabs -> rank 0
            } else if (lc.sharded) RET(op_halo(h, v.x[v.cur].p, lv.n, lv.m, col.lv[(size_t)l + 1].b.p, lc.n, lc.m));
            else {
                RET(op_halo(h, v.x[v.cur].p, lv.n, lv.m));
                RET(op_gather_rhs(h, col, l + 1));                         // slabs -> rank 0
            }
        }
    }
    // ---- coarse tail in one CTA, or just the coarsest level: exact solve (src/solvers.jl:39) ----
    if (ts < nl) {
        for (int l = ts; l < nl; ++l) col.lv[(size_t)l].cur = 0;
        cudaError_t te = tail_launch(h->L[ts].m, h->d_tail, nl - ts, h->coarse_fac, nPre, nPost, alpha,
                                     h->tail_plan_, h->stream, h->opt_pdl != 0);
        if (te != cudaSuccess) return fail(h, AMG1D_ERR_CUDA, "f_tail launch failed: %s", cudaGetErrorString(te));
        h->launch_counter++;
    } else if (h->L[nl - 1].present) {
        Column::Vecs& v = col.lv[(size_t)nl - 1];
        if (nl > 1 || zero0) v.cur = 0;
        RET(op_coarse(h, v.b.p, v.x[v.cur].p));   // single level: x = A \ b overwrites x
    }
    // ---- up ----
    for (int l = std::min(nl - 2, ts - 1); l >= 0; --l) {
        Level& lv = h->L[l];
        Level& lc = h->L[l + 1];
        Column::Vecs& v = col.lv[(size_t)l];
        if (!lv.present) continue;
        if (lv.sharded && !lc.sharded) RET(op_scatter_sol(h, col, l + 1));   // rank 0 -> slabs (+ ghosts)
        bool pushed = false;
        RET(leg_up(h, col, l, nPost, alpha, want_norm && l == 0, &norm_done, &pushed));
        if (p2p && lv.sharded) {
            if (l == 0) u0_pushed = pushed;
            else if (!pushed) RET(op_p2p_push(h, col, 2 * l + 1, l, v.cur));   // (a leg without the fused exchange)
        } else if (lv.sharded && l > 0) RET(op_halo(h, v.x[v.cur].p, lv.n, lv.m));   // for level l-1's prolongation
    }
    Column::Vecs& v0 = col.lv[0];
    if (v0.cur != 0) {
        CK(cudaMemcpyAsync(v0.x[0].p, v0.x[1].p, (size_t)v0.x[0].len * 8, cudaMemcpyDeviceToDevice,
                           h->stream));
        v0.cur = 0;
    }
    // level 0's corrected iterate: the incoming iterate of the next cycle, and the signal that this rank's up
    // leg no longer reads the ghosts which the neighbours' next down leg overwrites
    if (p2p && h->L[0].sharded && !u0_pushed) RET(op_p2p_push(h, col, 1, 0, 0));
    if (want_norm && !norm_done) RET(op_resnorm(h, col, 0, 0));
    return AMG1D_OK;
}

// One V-cycle through enqueue(): replayed from the cache's graph for key, which a miss captures and instantiates in the
// least recently used entry; enqueued directly with option graph off or profile on.  *launches: kernels of one cycle.
// parity0: the level-0 iterates of the cycled columns are in buffer 0, as a capture assumes.
template <class Enqueue>
int replay_vcycle(amg1d* h, GraphEntry (&cache)[4], const GraphEntry& key, bool parity0, int64_t* launches,
                  Enqueue enqueue) {
    if (!h->opt_graph || h->opt_profile) {
        const int64_t c0 = h->launch_counter;
        RET(enqueue());
        *launches = h->launch_counter - c0;
        return AMG1D_OK;
    }
    GraphEntry* ge = nullptr;
    for (auto& g : cache)
        if (g.exec && g.mask == key.mask && g.pre == key.pre && g.post == key.post && g.alpha == key.alpha &&
            g.norm == key.norm && g.zero0 == key.zero0)
            ge = &g;
    if (!ge) {
        ge = &cache[0];                                   // free slot, else the least recently used one
        for (auto& g : cache) if (!g.exec) { ge = &g; break; } else if (g.stamp < ge->stamp) ge = &g;
        if (ge->exec) { cudaGraphExecDestroy(ge->exec); ge->exec = nullptr; }
        if (!parity0) return fail(h, AMG1D_ERR_STATE, "internal: level-0 buffer parity");
        cudaGraph_t g = nullptr;
        const int64_t c0 = h->launch_counter;
        CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue();
        cudaError_t ce = cudaStreamEndCapture(h->stream, &g);
        if (rc != AMG1D_OK) { if (g) cudaGraphDestroy(g); return rc; }
        if (ce != cudaSuccess) return fail(h, AMG1D_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(ce));
        const int64_t n = h->launch_counter - c0;
        h->launch_counter = c0;
        cudaGraphExec_t exec = nullptr;
        ce = cudaGraphInstantiate(&exec, g, 0);
        cudaGraphDestroy(g);
        if (ce != cudaSuccess) return fail(h, AMG1D_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(ce));
        *ge = key;
        ge->exec = exec;
        ge->launches = n;
    }
    ge->stamp = ++h->graph_clock;
    CK(cudaGraphLaunch(ge->exec, h->stream));
    *launches = ge->launches;
    h->launch_counter += ge->launches;
    return AMG1D_OK;
}

// V-cycle of the resident problem (col is h->res: the tail descriptors d_tail and the graph cache graphs[] hold its
// vectors)
int run_vcycle(amg1d* h, Column& col, int nPre, int nPost, double alpha, bool want_norm, bool zero0 = false) {
    if (nPre < 0 || nPost < 0) return fail(h, AMG1D_ERR_ARG, "nPre and nPost must be >= 0");
    GraphEntry key;
    key.pre = nPre; key.post = nPost; key.alpha = alpha; key.norm = (int)want_norm; key.zero0 = (int)zero0; key.mask = 1;
    RET(replay_vcycle(h, h->graphs, key, col.lv[0].cur == 0, &h->launches_per_cycle,
                      [&] { return enqueue_vcycle(h, col, nPre, nPost, alpha, want_norm, zero0); }));
    h->norm_valid = want_norm;
    return AMG1D_OK;
}

void release_graphs(GraphEntry (&cache)[4]) {
    for (auto& g : cache) {
        if (g.exec) cudaGraphExecDestroy(g.exec);
        g = GraphEntry();
    }
}

void invalidate_graph(amg1d* h) {
    release_graphs(h->graphs);
    release_graphs(h->multi.graphs);
    h->norm_valid = false;
    h->multi.norm_valid = false;
}

int p2p_check(amg1d* h) {                     // after a stream synchronisation: did a peer-memory wait time out?
    if (!h->p2p.on) return AMG1D_OK;
    int e = 0;
    CK(cudaMemcpy(&e, h->p2p.err, sizeof e, cudaMemcpyDeviceToHost));
    if (e) return fail(h, AMG1D_ERR_NCCL, "peer-memory halo exchange timed out: a neighbour rank did not reach the "
                       "same V-cycle (crashed or out of step)");
    return AMG1D_OK;
}

// ---- host <-> device vector movement (reference ordering <-> device block ordering) --------------
int ensure_stage(amg1d* h, int64_t len) {
    if (h->stage_len >= len) return AMG1D_OK;
    if (h->stage) { cudaFree(h->stage); h->device_bytes -= h->stage_len * 8; }
    h->stage = nullptr; h->stage_len = 0;
    RET(dev_alloc(h, (void**)&h->stage, len * 8));
    h->stage_len = len;
    return AMG1D_OK;
}

int to_device(amg1d* h, int l, const double* host, double* dev) {
    Level& lv = h->L[l];
    if (!lv.perm) {
        CK(cudaMemcpyAsync(dev, host, (size_t)lv.n_host * 8, cudaMemcpyHostToDevice, h->stream));
        return AMG1D_OK;
    }
    RET(ensure_stage(h, lv.n_host));
    CK(cudaMemcpyAsync(h->stage, host, (size_t)lv.n_host * 8, cudaMemcpyHostToDevice, h->stream));
    const int64_t ns = lv.n * lv.m;
    k_gather_perm<<<(unsigned)((ns + 255) / 256), 256, 0, h->stream>>>(lv.perm, h->stage, dev, ns);
    LAUNCH_CHECK();
    return AMG1D_OK;
}

int to_host(amg1d* h, int l, const double* dev, double* host) {
    Level& lv = h->L[l];
    if (!lv.perm) {
        CK(cudaMemcpyAsync(host, dev, (size_t)lv.n_host * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return p2p_check(h);
    }
    RET(ensure_stage(h, lv.n_host));
    const int64_t ns = lv.n * lv.m;
    k_scatter_perm<<<(unsigned)((ns + 255) / 256), 256, 0, h->stream>>>(lv.perm, dev, h->stage, ns);
    LAUNCH_CHECK();
    CK(cudaMemcpyAsync(host, h->stage, (size_t)lv.n_host * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AMG1D_OK;
}

int read_scalars(amg1d* h, Column& col, int count) {
    CK(cudaMemcpyAsync(h->h_scal, col.scal, sizeof(double) * count, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return p2p_check(h);
}

// multigrid() (src/solvers.jl) on the resident problem: V-cycles until ||b - A x|| < tol ||b|| or maxiter; with d_exact
// also err[i] = ||x - u_exact|| of every iterate (NaN without it)
int multigrid_run(amg1d* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters, double* res,
                  double* err, const double* d_exact) {
    Column::Vecs& v0 = h->res.lv[0];
    int rc = op_norm(h, h->res, v0.b.p, nullptr, v0.b.len, 2);
    int it = 0;
    for (int i = 0; i < maxiter && rc == AMG1D_OK; ++i) {
        rc = run_vcycle(h, h->res, nPre, nPost, alpha, true);
        if (rc != AMG1D_OK) break;
        if (d_exact) {
            rc = op_norm(h, h->res, v0.x[v0.cur].p, d_exact, v0.x[0].len, 1);
            if (rc != AMG1D_OK) break;
        }
        rc = read_scalars(h, h->res, 3);
        if (rc != AMG1D_OK) break;
        res[i] = h->h_scal[0];
        if (err) err[i] = d_exact ? h->h_scal[1] : NAN;
        it = i + 1;
        if (res[i] < tol * h->h_scal[2]) break;
    }
    RET(rc);
    *iters = it;
    return AMG1D_OK;
}

// dense m x m inverse with partial pivoting (Gauss-Jordan), column-major; returns false if singular
bool invert_block(const double* A, double* Ainv, int m) {
    std::vector<double> a(A, A + m * m);
    for (int j = 0; j < m; ++j)
        for (int i = 0; i < m; ++i) Ainv[j * m + i] = (i == j) ? 1.0 : 0.0;
    for (int c = 0; c < m; ++c) {
        int piv = c;
        double best = std::fabs(a[c * m + c]);
        for (int r = c + 1; r < m; ++r)
            if (std::fabs(a[c * m + r]) > best) { best = std::fabs(a[c * m + r]); piv = r; }
        if (best == 0.0) return false;
        if (piv != c)
            for (int j = 0; j < m; ++j) {
                std::swap(a[j * m + c], a[j * m + piv]);
                std::swap(Ainv[j * m + c], Ainv[j * m + piv]);
            }
        const double d = 1.0 / a[c * m + c];
        for (int j = 0; j < m; ++j) { a[j * m + c] *= d; Ainv[j * m + c] *= d; }
        for (int r = 0; r < m; ++r) {
            if (r == c) continue;
            const double f = a[c * m + r];
            if (f == 0.0) continue;
            for (int j = 0; j < m; ++j) {
                a[j * m + r] -= f * a[j * m + c];
                Ainv[j * m + r] -= f * Ainv[j * m + c];
            }
        }
    }
    return true;
}

void matmul_cm(const double* A, const double* B, double* C, int m) {  // C = A B, column-major
    for (int j = 0; j < m; ++j)
        for (int i = 0; i < m; ++i) {
            double s = 0.0;
            for (int k = 0; k < m; ++k) s += A[k * m + i] * B[j * m + k];
            C[j * m + i] = s;
        }
}

int bcr_factor(amg1d* h, BcrSolver& S, int level) {
    Level& lv = h->L[level];
    if (lv.m > AMG1D_BCR_MAXM) return fail(h, AMG1D_ERR_UNSUPPORTED, "block size %d too large for the direct solver", lv.m);
    bool singular = false;
    const cudaError_t e = S.factor(lv.mat, lv.md, lv.n, h->stream, &singular);
    if (e != cudaSuccess) {
        S.release();
        return fail(h, e == cudaErrorMemoryAllocation ? AMG1D_ERR_NOMEM : AMG1D_ERR_CUDA,
                    "direct solver factorisation of level %d failed: %s", level, cudaGetErrorString(e));
    }
    if (singular) { S.release(); return fail(h, AMG1D_ERR_ARG, "level %d is singular (cyclic reduction hit a singular block)", level); }
    h->device_bytes += S.bytes;
    return AMG1D_OK;
}

int factor_coarsest(amg1d* h) {
    Level& lv = h->L[h->n_levels - 1];
    if (lv.n > AMG1D_BCR_MIN) return bcr_factor(h, h->coarse_bcr, h->n_levels - 1);
    if (lv.h_di.empty())
        return fail(h, AMG1D_ERR_STATE, "internal: host copy of the coarsest level is missing");
    const int m = lv.m, mm = m * m;
    std::vector<double> fac((size_t)lv.n * 3 * mm, 0.0), S(mm), tmp(mm), Sinv_prev(mm);
    for (int64_t k = 0; k < lv.n; ++k) {
        double* W = &fac[(size_t)k * 3 * mm];
        double* Sinv = W + mm;
        double* U = W + 2 * mm;
        std::copy(&lv.h_di[(size_t)k * mm], &lv.h_di[(size_t)k * mm] + mm, S.begin());
        if (k > 0) {
            matmul_cm(&lv.h_lo[(size_t)k * mm], Sinv_prev.data(), W, m);       // W = L_k Sinv_{k-1}
            matmul_cm(W, &lv.h_up[(size_t)(k - 1) * mm], tmp.data(), m);        // W U_{k-1}
            for (int q = 0; q < mm; ++q) S[q] -= tmp[q];
        }
        if (!invert_block(S.data(), Sinv, m))
            return fail(h, AMG1D_ERR_ARG, "coarsest level is singular at element %lld", (long long)k);
        std::copy(&lv.h_up[(size_t)k * mm], &lv.h_up[(size_t)k * mm] + mm, U);
        std::copy(Sinv, Sinv + mm, Sinv_prev.begin());
    }
    RET(dev_alloc(h, (void**)&h->coarse_fac, (int64_t)fac.size() * 8));
    CK(cudaMemcpy(h->coarse_fac, fac.data(), fac.size() * 8, cudaMemcpyHostToDevice));
    return AMG1D_OK;
}

// tail_host with col's x[0] and b: the descriptors f_tail reads for that column (tail_host covers [n_levels - size, n_levels))
void fill_tail(const amg1d* h, const Column& col, TailLevel* out) {
    const size_t ts = (size_t)h->n_levels - h->tail_host.size();
    for (size_t i = 0; i < h->tail_host.size(); ++i) {
        out[i] = h->tail_host[i];
        out[i].x = col.lv[ts + i].x[0].p;
        out[i].b = col.lv[ts + i].b.p;
    }
}

// Single-CTA coarse tail (kernels_fused.cuh, f_tail): the longest suffix of levels [ts, n_levels) that
// are unsharded, have at most min(coarse_cta_elems, TAIL_B) elements, share one block size, use block
// smoothers and single-parent closed-form transfers, and whose operators + vectors fit the CTA's
// shared memory.  Level 0 never joins (it carries the caller's initial guess), and a tail of the
// coarsest level alone stays with g_coarse_solve.
int build_tail(amg1d* h) {
    h->tail_start = -1;
    h->tail_host.clear();
    h->tail_gen++;
    if (h->d_tail) { cudaFree(h->d_tail); h->d_tail = nullptr; }
    const int nl = h->n_levels;
    if (nl < 3 || h->opt_coarse_cta < 1 || !h->L[nl - 1].present || h->coarse_bcr.ready()) return AMG1D_OK;
    const int m = h->L[nl - 1].m;
    if (!tail_supported(m)) return AMG1D_OK;
    const int64_t cap = std::min<int64_t>(h->opt_coarse_cta, TAIL_B);
    int ts = nl;
    int op_total = 0, vec_total = 0, p_total = 0;
    for (int l = nl - 1; l >= 1 && nl - l < TAIL_MAXL; --l) {
        const Level& lv = h->L[l];
        if (lv.sharded || !lv.present || lv.m != m || lv.n_glob > cap) break;
        int p_len = 0;
        if (l < nl - 1) {
            const Transfer& t = h->T[l];
            if (lv.diag || lv.smooth_tri || !t.single_parent_uniform || t.P1) break;
            p_len = (int)(t.nblk * m * m);
        }
        const int op_len = (int)(amg1d_tiles(lv.n) * lv.K * AMG1D_TILE);
        const TailPlan trial = tail_plan(m, op_total + op_len, vec_total + (int)lv.n * m, p_total + p_len);
        if ((size_t)trial.total * 8 > TAIL_SMEM_MAX) break;
        op_total += op_len; vec_total += (int)lv.n * m; p_total += p_len;
        ts = l;
    }
    if (ts > nl - 2) return AMG1D_OK;
    std::vector<TailLevel> tl((size_t)(nl - ts));
    int op_off = 0, vec_off = 0, p_off = 0;
    for (int l = ts; l < nl; ++l) {
        const Level& lv = h->L[l];
        TailLevel& d = tl[(size_t)(l - ts)];
        memset(&d, 0, sizeof d);
        d.md = lv.md;
        d.mat = lv.mat;
        d.n = lv.n;
        d.op_off = op_off; d.op_len = (int)(amg1d_tiles(lv.n) * lv.K * AMG1D_TILE);
        d.vec_off = vec_off;
        d.p_off = p_off; d.p_len = 0;
        if (l < nl - 1) {
            d.tm = make_map_closed(h->T[l]);
            d.P0 = h->T[l].P0;
            d.p_len = (int)(h->T[l].nblk * m * m);
        }
        op_off += d.op_len; vec_off += (int)lv.n * m; p_off += d.p_len;
    }
    h->tail_plan_ = tail_plan(m, op_off, vec_off, p_off);
    cudaError_t e = tail_configure(m, (size_t)h->tail_plan_.total * 8);
    if (e != cudaSuccess) return fail(h, AMG1D_ERR_CUDA, "f_tail configuration failed: %s", cudaGetErrorString(e));
    h->tail_host = tl;
    fill_tail(h, h->res, tl.data());
    RET(dev_alloc(h, (void**)&h->d_tail, (int64_t)(tl.size() * sizeof(TailLevel))));
    CK(cudaMemcpy(h->d_tail, tl.data(), tl.size() * sizeof(TailLevel), cudaMemcpyHostToDevice));
    h->tail_start = ts;
    return AMG1D_OK;
}

int check_ready(amg1d* h) {
    if (!h) return AMG1D_ERR_ARG;
    if (!h->finalized) return fail(h, AMG1D_ERR_STATE, "hierarchy not finalized (call amg1d_finalize)");
    CK(cudaSetDevice(h->device));
    return AMG1D_OK;
}

int check_dev_problem(amg1d* h) {
    RET(check_ready(h));
    if (!h->dev_problem)
        return fail(h, AMG1D_ERR_STATE, "the device-resident problem was overwritten by a per-level host operation "
                    "(amg1d_residual / amg1d_smoother_solve on level 0, amg1d_pcg); call amg1d_dev_set_problem again");
    return AMG1D_OK;
}

// ---- multi-column resident problems (amg1d_dev_set_problems ...) ----------------------------------------------------
// Each column of the set has its own vectors on every level.  Levels whose legs have a fused multi-column kernel
// (kernels_multi.cuh) run one launch for all active columns; every other operation of the cycle - the row-per-thread and
// generic tiers, the single-CTA tail, the coarse solve - runs its single-column code once per column, so per column it
// is exactly the single-column cycle.

// storage for k columns: the set only grows; a failed allocation releases what it took and leaves the rest as it was
int multi_alloc(amg1d* h, int k) {
    amg1d::Multi& M = h->multi;
    if (!M.d_scal) RET(dev_alloc(h, (void**)&M.d_scal, MULTI_MAX_COLS * MULTI_SLOTS * 8));
    if (!M.h_scal) CK(cudaMallocHost(&M.h_scal, MULTI_MAX_COLS * MULTI_SLOTS * 8));
    if (!M.d_tail) RET(dev_alloc(h, (void**)&M.d_tail, (int64_t)(MULTI_MAX_COLS * TAIL_MAXL * sizeof(TailLevel))));
    while ((int)M.col.size() < k) {
        Column col;
        col.scal = M.d_scal + M.col.size() * MULTI_SLOTS;
        const int rc = column_alloc(h, col, false);
        if (rc != AMG1D_OK) return fail(h, rc, "column %d of the multi-column set: %s", (int)M.col.size(), h->err.c_str());
        M.col.push_back(std::move(col));
        M.tail_synced = ~0ull;
    }
    return AMG1D_OK;
}

// descriptors of the single-CTA tail for every column (before capture)
int multi_sync_tail(amg1d* h) {
    amg1d::Multi& M = h->multi;
    if (h->tail_start <= 0 || M.tail_synced == h->tail_gen) return AMG1D_OK;
    std::vector<TailLevel> all((size_t)MULTI_MAX_COLS * TAIL_MAXL);
    for (size_t c = 0; c < M.col.size(); ++c) fill_tail(h, M.col[c], &all[c * TAIL_MAXL]);
    CK(cudaMemcpyAsync(M.d_tail, all.data(), all.size() * sizeof(TailLevel), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    M.tail_synced = h->tail_gen;
    return AMG1D_OK;
}

// the fused multi-column kernels serve level l (the test of leg_down / leg_up plus a kernel for the combination)
bool multi_leg_level(const amg1d* h, int l) {
    const Level& lv = h->L[l];
    const Transfer& t = h->T[l];
    return h->opt_fused && t.fusable && !lv.smooth_tri && fused_multi_available(lv.md, t.mc);
}

int prof_unmark(amg1d* h, int level, int leg) {      // drop the opening bracket of a leg that did not launch
    if (!h->opt_profile) return AMG1D_OK;
    auto& ev = h->prof[level * 2 + leg].ev;
    cudaEventDestroy(ev.back());
    ev.pop_back();
    return AMG1D_OK;
}

int leg_down_multi(amg1d* h, int l, const int* act, int na, int nPre, double alpha, bool zero0) {
    Level& lv = h->L[l];
    Transfer& t = h->T[l];
    amg1d::Multi& M = h->multi;
    const bool zero = l > 0 || zero0;
    if (multi_leg_level(h, l)) {
        MultiCols mc = {};
        int ob[MULTI_MAX_COLS];
        for (int i = 0; i < na; ++i) {
            Column& col = M.col[(size_t)act[i]];
            Column::Vecs& v = col.lv[(size_t)l];
            if (zero) v.cur = 0;
            ob[i] = zero ? 0 : 1 - v.cur;
            mc.b[i] = v.b.p;
            mc.xin[i] = v.x[v.cur].p;
            mc.xout[i] = v.x[ob[i]].p;
            mc.xc[i] = col.lv[(size_t)l + 1].b.p;
        }
        RET(prof_mark(h, l, 0));
        cudaError_t le = cudaSuccess;
        const int fr = fused_down_multi(lv.md, t.mc, make_map_closed(t), nPre, zero, lv.mat, make_pat(h, l), mc, na,
                                        tp0(t), tp1(t), lv.n, alpha, make_slab(h, l), h->stream, h->opt_pdl != 0, &le,
                                        leg_rec(h, lv, t.mc));
        if (fr == FUSED_ERR) return fail(h, AMG1D_ERR_CUDA, "f_down_multi launch failed on level %d: %s", l, cudaGetErrorString(le));
        if (fr == FUSED_OK) {
            for (int i = 0; i < na; ++i) M.col[(size_t)act[i]].lv[(size_t)l].cur = ob[i];
            h->launch_counter++;
            LAUNCH_CHECK();
            return prof_mark(h, l, 0);
        }
        RET(prof_unmark(h, l, 0));
    }
    for (int i = 0; i < na; ++i) RET(leg_down(h, M.col[(size_t)act[i]], l, nPre, alpha, zero0));
    return AMG1D_OK;
}

// norm: level 0 of a cycle that leaves ||b - A x|| in slot 0 of every column (done[i]: already there)
int leg_up_multi(amg1d* h, int l, const int* act, int na, int nPost, double alpha, bool norm, bool* done) {
    Level& lv = h->L[l];
    Transfer& t = h->T[l];
    amg1d::Multi& M = h->multi;
    if (multi_leg_level(h, l)) {
        MultiCols mc = {};
        for (int i = 0; i < na; ++i) {
            Column& col = M.col[(size_t)act[i]];
            Column::Vecs& v = col.lv[(size_t)l];
            Column::Vecs& vc = col.lv[(size_t)l + 1];
            mc.b[i] = v.b.p;
            mc.xin[i] = v.x[v.cur].p;
            mc.xout[i] = v.x[1 - v.cur].p;
            mc.xc[i] = vc.x[vc.cur].p;
            mc.partial[i] = norm ? col.partial : nullptr;
        }
        RET(prof_mark(h, l, 1));
        cudaError_t le = cudaSuccess;
        int nb = 0;
        const int fr = fused_up_multi(lv.md, t.mc, make_map_closed(t), nPost, lv.mat, make_pat(h, l), mc, na, tp0(t),
                                      tp1(t), lv.n, alpha, norm, h->partial_cap, &nb, make_slab(h, l), h->stream,
                                      h->opt_pdl != 0, &le, leg_rec(h, lv, t.mc));
        if (fr == FUSED_ERR) return fail(h, AMG1D_ERR_CUDA, "f_up_multi launch failed on level %d: %s", l, cudaGetErrorString(le));
        if (fr == FUSED_OK) {
            for (int i = 0; i < na; ++i) { auto& v = M.col[(size_t)act[i]].lv[(size_t)l]; v.cur = 1 - v.cur; }
            h->launch_counter++;
            LAUNCH_CHECK();
            RET(prof_mark(h, l, 1));
            if (norm)
                for (int i = 0; i < na; ++i) {
                    RET(op_reduce_partials(h, M.col[(size_t)act[i]], nb, 0, true));
                    done[i] = true;
                }
            return AMG1D_OK;
        }
        RET(prof_unmark(h, l, 1));
    }
    for (int i = 0; i < na; ++i) {
        bool pushed = false;
        RET(leg_up(h, M.col[(size_t)act[i]], l, nPost, alpha, norm, &done[i], &pushed));
    }
    return AMG1D_OK;
}

// enqueue_vcycle for the active columns act[0..na) of the multi-column set (single GPU)
int enqueue_vcycle_multi(amg1d* h, const int* act, int na, int nPre, int nPost, double alpha, bool want_norm,
                         bool zero0) {
    const int nl = h->n_levels;
    const int ts = h->tail_start > 0 ? h->tail_start : nl;
    amg1d::Multi& M = h->multi;
    bool done[MULTI_MAX_COLS] = {};
    for (int l = 0; l < nl - 1 && l < ts; ++l) RET(leg_down_multi(h, l, act, na, nPre, alpha, zero0));
    if (ts < nl) {
        for (int i = 0; i < na; ++i) {
            for (int l = ts; l < nl; ++l) M.col[(size_t)act[i]].lv[(size_t)l].cur = 0;
            cudaError_t te = tail_launch(h->L[ts].m, M.d_tail + (size_t)act[i] * TAIL_MAXL, nl - ts, h->coarse_fac,
                                         nPre, nPost, alpha, h->tail_plan_, h->stream, h->opt_pdl != 0);
            if (te != cudaSuccess) return fail(h, AMG1D_ERR_CUDA, "f_tail launch failed: %s", cudaGetErrorString(te));
            h->launch_counter++;
        }
    } else {
        for (int i = 0; i < na; ++i) {
            Column::Vecs& v = M.col[(size_t)act[i]].lv[(size_t)nl - 1];
            if (nl > 1 || zero0) v.cur = 0;
            RET(op_coarse(h, v.b.p, v.x[v.cur].p));
        }
    }
    for (int l = std::min(nl - 2, ts - 1); l >= 0; --l)
        RET(leg_up_multi(h, l, act, na, nPost, alpha, want_norm && l == 0, done));
    for (int i = 0; i < na; ++i) {
        Column& col = M.col[(size_t)act[i]];
        auto& v = col.lv[0];
        if (v.cur != 0) {
            CK(cudaMemcpyAsync(v.x[0].p, v.x[1].p, (size_t)v.x[0].len * 8, cudaMemcpyDeviceToDevice, h->stream));
            v.cur = 0;
        }
        if (want_norm && !done[i]) RET(op_resnorm(h, col, 0, 0));
    }
    return AMG1D_OK;
}

// run_vcycle for the multi-column set: graph replay keyed by the cycle parameters and the active columns
int run_vcycle_multi(amg1d* h, const int* act, int na, int nPre, int nPost, double alpha, bool want_norm, bool zero0) {
    if (nPre < 0 || nPost < 0) return fail(h, AMG1D_ERR_ARG, "nPre and nPost must be >= 0");
    amg1d::Multi& M = h->multi;
    RET(multi_sync_tail(h));
    GraphEntry key;
    key.pre = nPre; key.post = nPost; key.alpha = alpha; key.norm = (int)want_norm; key.zero0 = (int)zero0;
    bool parity0 = true;
    for (int i = 0; i < na; ++i) {
        key.mask |= 1u << act[i];
        parity0 = parity0 && M.col[(size_t)act[i]].lv[0].cur == 0;
    }
    return replay_vcycle(h, M.graphs, key, parity0, &M.launches_per_cycle,
                         [&] { return enqueue_vcycle_multi(h, act, na, nPre, nPost, alpha, want_norm, zero0); });
}

// need_rhs: the call reads the set's right-hand sides, which amg1d_dev_pcg_multi consumes
int check_multi(amg1d* h, bool need_set, bool need_rhs = true) {
    RET(check_ready(h));
    if (h->nranks > 1)
        return fail(h, AMG1D_ERR_UNSUPPORTED, "multi-column problems run on a single GPU (this handle has %d ranks)",
                    h->nranks);
    if (need_set && h->multi.k == 0)
        return fail(h, AMG1D_ERR_STATE, "no multi-column problem set (amg1d_dev_set_problems / amg1d_dev_fill_rhs_random_multi)");
    if (need_set && need_rhs && h->multi.rhs_consumed)
        return fail(h, AMG1D_ERR_STATE, "the multi-column right-hand sides became CG residuals in amg1d_dev_pcg_multi; "
                    "install a set again (amg1d_dev_set_problems / amg1d_dev_fill_rhs_random_multi)");
    return AMG1D_OK;
}

int check_cols(amg1d* h, int k) {
    if (k < 1 || k > MULTI_MAX_COLS) return fail(h, AMG1D_ERR_ARG, "column count %d outside [1, %d]", k, MULTI_MAX_COLS);
    return AMG1D_OK;
}

int read_multi_scalars(amg1d* h) {
    CK(cudaMemcpyAsync(h->multi.h_scal, h->multi.d_scal, MULTI_MAX_COLS * MULTI_SLOTS * 8, cudaMemcpyDeviceToHost,
                       h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AMG1D_OK;
}

// Structure class of a level (layout.cuh) from `nb` uploaded off-diagonal block sets.
void detect_structure(const double* lo, const double* up, int64_t nb, int m, int* st, int* ilo, int* iup) {
    *st = AMG1D_ST_DENSE; *ilo = 0; *iup = 0;
    if (m < 2) return;
    const int mm = m * m;
    std::vector<char> lo_col(m, 0), lo_row(m, 0), up_col(m, 0), up_row(m, 0);
    for (int64_t e = 0; e < nb; ++e)
        for (int j = 0; j < m; ++j)
            for (int i = 0; i < m; ++i) {
                if (lo[e * mm + j * m + i] != 0.0) { lo_col[j] = 1; lo_row[i] = 1; }
                if (up[e * mm + j * m + i] != 0.0) { up_col[j] = 1; up_row[i] = 1; }
            }
    auto single = [m](const std::vector<char>& mask, int* idx) {
        int cnt = 0;
        *idx = 0;
        for (int q = 0; q < m; ++q) if (mask[q]) { ++cnt; *idx = q; }
        return cnt <= 1;
    };
    int a, b;
    if (single(lo_col, &a) && single(up_row, &b)) { *st = AMG1D_ST_COLROW; *ilo = a; *iup = b; return; }
    if (single(lo_row, &a) && single(up_col, &b)) { *st = AMG1D_ST_ROWCOL; *ilo = a; *iup = b; return; }
}

// A level upload failed after alloc_level_common succeeded: give back what it took (operator tiles,
// permutation, pattern table, the byte accounting and the gather-level decision) so that the level stays
// cleanly unset and the same call can be retried.
void undo_level_alloc(amg1d* h, int level) {
    Level& lv = h->L[level];
    if (lv.mat_alloc) { cudaFree(lv.mat_alloc); h->device_bytes -= lv.mat_bytes; }
    if (lv.perm) { cudaFree(lv.perm); h->device_bytes -= lv.n_glob * lv.m * 8; }
    if (lv.pat) { cudaFree(lv.pat); h->device_bytes -= (int64_t)lv.pat_host.size() * 8; }
    lv.mat_alloc = lv.mat = nullptr; lv.perm = nullptr; lv.pat = nullptr; lv.mat_bytes = 0;
    lv.pat_host.clear(); lv.h_lo.clear(); lv.h_di.clear(); lv.h_up.clear();
    if (h->gather_level == level) h->gather_level = -1;
    lv.set = false;
}

int alloc_level_common(amg1d* h, int level, int64_t n_elem, int m, int diag, const int64_t* perm,
                       int64_t n_dof_host, int st, int ilo, int iup) {
    if (!valid_level(h, level)) return fail(h, AMG1D_ERR_ARG, "level %d out of range", level);
    if (h->finalized) return fail(h, AMG1D_ERR_STATE, "hierarchy already finalized");
    if (n_elem < 1 || m < 1 || m > 32) return fail(h, AMG1D_ERR_ARG, "need n_elem >= 1 and 1 <= m <= 32");
    Level& lv = h->L[level];
    if (lv.set) return fail(h, AMG1D_ERR_STATE, "level %d already set", level);
    CK(cudaSetDevice(h->device));
    lv.m = m; lv.diag = diag ? 1 : 0;
    lv.md = amg1d_desc(m, lv.diag, st, ilo, iup);
    lv.K = lv.md.K;
    lv.n_glob = n_elem;
    if (!perm && n_dof_host != n_elem * m)
        return fail(h, AMG1D_ERR_ARG, "n_dof_host must equal n_elem*m when perm is NULL");
    // slab decision (SURVEY 8e): shard while the level is large, otherwise it lives on rank 0
    // (a remainder of one element - the closing vertex group of a CG level, n + 1 groups - goes to
    // the last rank)
    lv.sharded = h->nranks > 1 && !perm && n_elem % h->nranks <= 1 &&
                 n_elem / h->nranks >= h->shard_min &&
                 (level == 0 || h->L[level - 1].sharded);
    if (h->nranks > 1 && level == 0 && !lv.sharded)
        return fail(h, AMG1D_ERR_UNSUPPORTED, "multi-GPU: the finest level must be shardable (DG-type, "
                    "n_elem divisible by the rank count, >= %lld elements per rank)", (long long)h->shard_min);
    if (lv.sharded) {
        lv.base_n = n_elem / h->nranks;
        lv.n = slab_size(n_elem, h->nranks, h->rank);
        lv.start = slab_start(n_elem, h->nranks, h->rank);
        lv.gl = h->rank > 0 ? h->ghost_depth : 0;
        lv.gr = h->rank < h->nranks - 1 ? h->ghost_depth : 0;
        lv.present = true;
        n_dof_host = lv.n * m;                    // host vectors are the rank's slab
    } else {
        lv.n = n_elem; lv.start = 0; lv.gl = lv.gr = 0;
        lv.present = h->rank == 0;
        if (h->nranks > 1 && h->gather_level < 0) h->gather_level = level;
    }
    lv.n_host = n_dof_host;
    if (perm)                                     // validated before anything is allocated
        for (int64_t s = 0; s < n_elem * m; ++s)
            if (perm[s] < -1 || perm[s] >= n_dof_host) {
                if (h->gather_level == level) h->gather_level = -1;
                return fail(h, AMG1D_ERR_ARG, "perm[%lld] out of range", (long long)s);
            }
    if (!lv.present) return AMG1D_OK;             // ranks > 0 hold nothing of gathered levels
    // one spare tile in front of element 0 (ghost elements have negative local indices)
    lv.mat_bytes = (amg1d_tiles(lv.n + lv.gr) + 1) * (int64_t)lv.K * AMG1D_TILE * 8;
    int rc = dev_alloc(h, (void**)&lv.mat_alloc, lv.mat_bytes);
    if (rc != AMG1D_OK) { lv.mat_alloc = nullptr; undo_level_alloc(h, level); return rc; }
    lv.mat = lv.mat_alloc + (int64_t)lv.K * AMG1D_TILE;
    cudaError_t ce = cudaMemsetAsync(lv.mat_alloc, 0, (size_t)lv.K * AMG1D_TILE * 8, h->stream);
    if (ce == cudaSuccess && perm) {
        const int64_t ns = n_elem * m;
        rc = dev_alloc(h, (void**)&lv.perm, ns * 8);
        if (rc != AMG1D_OK) { lv.perm = nullptr; undo_level_alloc(h, level); return rc; }
        ce = cudaMemcpy(lv.perm, perm, (size_t)ns * 8, cudaMemcpyHostToDevice);
    }
    if (ce != cudaSuccess) {
        undo_level_alloc(h, level);
        return fail(h, AMG1D_ERR_CUDA, "level %d allocation failed: %s", level, cudaGetErrorString(ce));
    }
    return AMG1D_OK;
}

void free_flux(amg1d* h, Level& lv) {
    for (double*& p : lv.flux)
        if (p) { cudaFree(p); p = nullptr; h->device_bytes -= lv.n * lv.m * lv.m * 8; }
}

// Option "recompute_dinv" (default on): replace the uploaded block-Jacobi inverses of a level by the device's own
// Gauss-Jordan inverse of the stored diagonal blocks - provided the upload agrees with it to 1e-8, i.e.
// really is inv(A_di) (src/smoother.jl:154-164) and not some other smoother block.  Afterwards every kernel that
// reads the stored inverse and the fused legs that recompute it in registers (reg_invert; 16 of the 40 stored
// doubles of a 4 x 4 DG element never leave HBM) produce the same bits.  Point-Jacobi levels keep their diagonal.
// The elimination is unpivoted when the level does not need its pivots (k_dinv_recompute: no element swaps rows, or
// every element that does gets the same inverse to 1e-12 without), else it keeps the partial-pivoting chain.  On a
// sharded level the verdict is reduced over the ranks, so that all slabs - and the single-GPU run, whose level is
// the union of the slabs - use the same elimination.
int adopt_device_dinv(amg1d* h, int level) {
    Level& lv = h->L[level];
    lv.dv_rec = 0;
    if (!h->opt_dvrec || lv.diag || lv.m > AMG1D_DVREC_MAXM) return AMG1D_OK;
    const bool collective = h->nranks > 1 && lv.sharded;
    if (!lv.present && !collective) return AMG1D_OK;
    DevBuf sc;
    CK(sc.alloc(4));
    CK(cudaMemsetAsync(sc.p, 0, 32, h->stream));
    unsigned long long* d_dev = reinterpret_cast<unsigned long long*>(sc.p);
    int* d_flag = reinterpret_cast<int*>(sc.p + 1);
    const int64_t e0 = -(int64_t)lv.gl, e1 = lv.n + lv.gr;
    const unsigned grid = (unsigned)((e1 - e0 + 127) / 128);
    if (lv.present)
        launch_dinv_recompute(grid, h->stream, lv.mat, lv.md, e0, e1, AMG1D_TILE, 2, d_dev, d_flag);   // one pass
    double host[4] = {0.0, 0.0, 0.0, 0.0};
    CK(cudaMemcpyAsync(host, sc.p, 16, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    int flag;
    memcpy(&flag, &host[1], sizeof flag);
    if (collective) {                              // max over the ranks of (deviation, singular, swaps, needs pivots)
        const double v[4] = {host[0], (flag & 1) ? 1.0 : 0.0, (flag & 2) ? 1.0 : 0.0, (flag & 4) ? 1.0 : 0.0};
        CK(cudaMemcpyAsync(sc.p, v, 32, cudaMemcpyHostToDevice, h->stream));
        RET(op_allreduce_max(h, sc.p, 4));
        CK(cudaMemcpyAsync(host, sc.p, 32, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        flag = (host[1] != 0.0 ? 1 : 0) | (host[2] != 0.0 ? 2 : 0) | (host[3] != 0.0 ? 4 : 0);
    }
    if ((flag & 1) || !(host[0] <= 1e-8)) return AMG1D_OK;    // not the inverse of A_di: keep what was uploaded
    const bool unpivot = (flag & 2) && !(flag & 4);           // rows swap somewhere, but no element needs it
    if (unpivot && lv.present)
        launch_dinv_recompute(grid, h->stream, lv.mat, lv.md, e0, e1, AMG1D_TILE, 3, d_dev, d_flag);
    if (lv.pat) {                                             // the pattern table's Dinv rows as well
        const int ns = lv.pat_head + 1 + lv.pat_tail;
        launch_dinv_recompute(1, h->stream, lv.pat, lv.md, 0, ns, 1, unpivot ? 3 : 1, d_dev, d_flag);
        CK(cudaMemcpyAsync(lv.pat_host.data(), lv.pat, lv.pat_host.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    lv.dv_rec = (flag & 4) ? 1 : 2;
    return AMG1D_OK;
}

// Installs a level whose operator blocks A_lo / A_di / A_up already sit on the device as element-block
// arrays dA[0..2] (n blocks of m x m): smoother inverses (block-Jacobi inverses of the diagonal blocks,
// src/smoother.jl:154-164, or the reciprocal diagonal, :92-98), structure detection, tile layout - the
// state amg1d_set_level leaves.  perm / n_dof_host as in amg1d_set_level; padding slots of a regrouped
// level get the identity on the diagonal.  dA[1] is modified (padding) and stays owned by the caller.
int install_from_blocks(amg1d* h, int level, int64_t n, int m, double* const* dA, int diag,
                        const int64_t* perm, int64_t n_dof_host) {
    const int mm = m * m;
    const int dsz = diag ? m : mm;
    DevBuf dDinv, dints;                           // dints: 4 m structure masks + 1 singular flag (ints)
    CK(dDinv.alloc((int64_t)n * dsz));
    CK(dints.alloc(2 * m + 1));
    int* dmask = reinterpret_cast<int*>(dints.p);
    int* dflag = dmask + 4 * m;
    CK(cudaMemsetAsync(dints.p, 0, (size_t)(2 * m + 1) * 8, h->stream));
    const unsigned grid = (unsigned)((n * mm + 127) / 128);
    k_structure_masks<<<grid, 128, 0, h->stream>>>(dA[0], dA[2], n, m, dmask);
    std::vector<int> mask(4 * (size_t)m, 0);
    CK(cudaMemcpyAsync(mask.data(), dmask, 4 * m * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    int st = AMG1D_ST_DENSE, ilo = 0, iup = 0;
    if (h->opt_compress && m >= 2) {
        auto single = [m](const int* mk, int* idx) {
            int cnt = 0;
            *idx = 0;
            for (int q = 0; q < m; ++q) if (mk[q]) { ++cnt; *idx = q; }
            return cnt <= 1;
        };
        int a, b;
        if (single(&mask[0], &a) && single(&mask[3 * m], &b)) { st = AMG1D_ST_COLROW; ilo = a; iup = b; }
        else if (single(&mask[m], &a) && single(&mask[2 * m], &b)) { st = AMG1D_ST_ROWCOL; ilo = a; iup = b; }
    }
    RET(alloc_level_common(h, level, n, m, diag, perm, n_dof_host, st, ilo, iup));
    Level& lv = h->L[level];
    auto undo = [&]() { undo_level_alloc(h, level); };   // the level stays unset
#define CKU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { undo(); \
        return fail(h, e_ == cudaErrorMemoryAllocation ? AMG1D_ERR_NOMEM : AMG1D_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); } } while (0)
    const unsigned gs = (unsigned)((n * m + 127) / 128);
    if (lv.perm) k_pad_identity<<<gs, 128, 0, h->stream>>>(dA[1], lv.perm, n, m);
    if (diag) {
        k_diag_reciprocal<<<gs, 128, 0, h->stream>>>(dA[1], n, m, dDinv.p, dflag);
    } else {
        CKU(cudaMemcpyAsync(dDinv.p, dA[1], (size_t)n * mm * 8, cudaMemcpyDeviceToDevice, h->stream));
        k_bcr_invert_odd<<<(unsigned)((n + 31) / 32), 32, 0, h->stream>>>(dDinv.p, m, n, 0, 1, dflag);
    }
    int flag = 0;
    CKU(cudaMemcpyAsync(&flag, dflag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CKU(cudaStreamSynchronize(h->stream));
    CKU(cudaGetLastError());
    if (flag) { undo(); return fail(h, AMG1D_ERR_ARG, "level %d: singular diagonal block", level); }
    const int64_t total = amg1d_tiles(n) * (int64_t)lv.K * AMG1D_TILE;
    k_repack<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(dA[0], dA[1], dA[2], dDinv.p, lv.md, 0, n, lv.mat);
    if (n <= AMG1D_BCR_MIN) {                      // host copy for the block-Thomas factorisation
        lv.h_lo.resize((size_t)n * mm); lv.h_di.resize((size_t)n * mm); lv.h_up.resize((size_t)n * mm);
        CKU(cudaMemcpyAsync(lv.h_lo.data(), dA[0], (size_t)n * mm * 8, cudaMemcpyDeviceToHost, h->stream));
        CKU(cudaMemcpyAsync(lv.h_di.data(), dA[1], (size_t)n * mm * 8, cudaMemcpyDeviceToHost, h->stream));
        CKU(cudaMemcpyAsync(lv.h_up.data(), dA[2], (size_t)n * mm * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    CKU(cudaStreamSynchronize(h->stream));
    CKU(cudaGetLastError());
#undef CKU
    lv.set = true;
    return adopt_device_dinv(h, level);
}

// Device-side set-up of one level from its flux operators (device_setup.cuh): A = C - D M^-1 G, then
// install_from_blocks with a block smoother.  flux: 9 element-block device arrays; d_minv: n blocks (or
// one when mi_const).
int install_from_flux(amg1d* h, int level, int64_t n, int m, double* const* flux, const double* d_minv,
                      int mi_const) {
    const int mm = m * m;
    DevBuf A[3], dband;
    for (auto& b : A) CK(b.alloc((int64_t)n * mm));
    CK(dband.alloc(2));
    CK(cudaMemsetAsync(dband.p, 0, 16, h->stream));
    const unsigned grid = (unsigned)((n * mm + 127) / 128);
    k_flux_operator<<<grid, 128, 0, h->stream>>>(flux[0], flux[1], flux[2], flux[3], flux[4], flux[5], flux[6],
                                                  flux[7], flux[8], d_minv, mi_const, n, m, A[0].p, A[1].p, A[2].p,
                                                  dband.p);
    double band[2] = {0.0, 0.0};
    CK(cudaMemcpyAsync(band, dband.p, 16, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    if (band[0] > 1e-11 * band[1])
        return fail(h, AMG1D_ERR_ARG, "level %d: C - D M^-1 G is not block tridiagonal (outer band %.3e vs "
                    "diagonal %.3e)", level, band[0], band[1]);
    double* dA[3] = {A[0].p, A[1].p, A[2].p};
    return install_from_blocks(h, level, n, m, dA, 0, nullptr, n * m);
}

}  // namespace

// =====================================================================================================
extern "C" {

int amg1d_version(void) { return AMG1D_VERSION; }

const char* amg1d_last_error(const amg1d_t* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int amg1d_create(amg1d_t** out, int n_levels, int device, void* stream) {
    amg1d* h = nullptr;
    if (!out) return fail(h, AMG1D_ERR_ARG, "null handle pointer");
    *out = nullptr;
    if (n_levels < 1) return fail(h, AMG1D_ERR_ARG, "At least one level required.");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(h, AMG1D_ERR_ARG, "device %d not available (%d visible)", device, ndev);
    CK(cudaSetDevice(device));
    amg1d* nh = new (std::nothrow) amg1d();
    if (!nh) return fail(h, AMG1D_ERR_NOMEM, "host allocation failed");
    nh->device = device;
    nh->n_levels = n_levels;
    nh->L.resize(n_levels);
    nh->T.resize(n_levels > 1 ? n_levels - 1 : 0);
    if (stream) {
        nh->stream = (cudaStream_t)stream;
    } else {
        cudaError_t e = cudaStreamCreateWithFlags(&nh->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete nh; return fail(h, AMG1D_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
        nh->own_stream = true;
    }
    *out = nh;
    return AMG1D_OK;
}

int amg1d_nccl_unique_id(void* id128) {
    amg1d* h = nullptr;
    if (!id128) return fail(h, AMG1D_ERR_ARG, "null id buffer");
#ifdef AMG1D_WITH_NCCL
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
    if (const char* e = load_nccl()) return fail(h, AMG1D_ERR_NCCL, "%s", e);
    ncclUniqueId id;
    NCK(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, sizeof id);
    return AMG1D_OK;
#else
    return fail(h, AMG1D_ERR_UNSUPPORTED, "libamg1d was built without NCCL");
#endif
}

int amg1d_create_dist(amg1d_t** out, int n_levels, int device, void* stream, int rank, int nranks,
                      const void* nccl_id) {
    if (nranks == 1 && rank == 0) return amg1d_create(out, n_levels, device, stream);
    amg1d* h = nullptr;
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(h, AMG1D_ERR_ARG, "bad rank / nranks");
    if (!nccl_id) return fail(h, AMG1D_ERR_ARG, "null NCCL id");
#ifdef AMG1D_WITH_NCCL
    if (const char* e = load_nccl()) return fail(h, AMG1D_ERR_NCCL, "%s", e);
    RET(amg1d_create(out, n_levels, device, stream));
    amg1d* nh = *out;
    nh->rank = rank;
    nh->nranks = nranks;
    ncclUniqueId id;
    memcpy(&id, nccl_id, sizeof id);
    ncclResult_t r = g_nccl.CommInitRank(&nh->comm, nranks, id, rank);
    if (r != ncclSuccess) {
        amg1d_destroy(nh);
        *out = nullptr;
        return fail(h, AMG1D_ERR_NCCL, "ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
    }
    return AMG1D_OK;
#else
    return fail(h, AMG1D_ERR_UNSUPPORTED, "libamg1d was built without NCCL");
#endif
}

int amg1d_destroy(amg1d_t* h) {
    if (!h) return AMG1D_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    release_graphs(h->graphs);
    release_graphs(h->multi.graphs);
    for (auto& col : h->multi.col) column_free(h, col);
    column_free(h, h->res);
    if (h->multi.d_scal) cudaFree(h->multi.d_scal);
    if (h->multi.h_scal) cudaFreeHost(h->multi.h_scal);
    if (h->multi.d_tail) cudaFree(h->multi.d_tail);
    if (h->res.scal) cudaFree(h->res.scal);
    for (auto& pr : h->prof) for (auto ev : pr.ev) cudaEventDestroy(ev);
    for (auto& lv : h->L) {
        if (lv.mat_alloc) cudaFree(lv.mat_alloc);
        if (lv.smat_alloc) cudaFree(lv.smat_alloc);
        if (lv.pat) cudaFree(lv.pat);
        free_flux(h, lv);
        if (lv.perm) cudaFree(lv.perm);
    }
    for (auto& t : h->T) {
        if (t.parent) cudaFree(t.parent);
        if (t.cp) cudaFree(t.cp);
        if (t.P0) cudaFree(t.P0);
        if (t.P1) cudaFree(t.P1);
    }
    vec_free(h->scratch);
    if (h->stage) cudaFree(h->stage);
    if (h->h_scal) cudaFreeHost(h->h_scal);
    if (h->coarse_fac) cudaFree(h->coarse_fac);
    if (h->d_tail) cudaFree(h->d_tail);
    h->coarse_bcr.release();
    for (auto& S : h->direct) S.release();
#ifdef AMG1D_WITH_NCCL
    p2p_close(h);
    if (h->comm) g_nccl.CommDestroy(h->comm);       // (a collective: no neighbour still writes into the arena after it)
#endif
    for (int k = 0; k < 2; ++k) {
        if (h->pipe.st_b[k]) cudaFree(h->pipe.st_b[k]);
        if (h->pipe.st_x[k]) cudaFree(h->pipe.st_x[k]);
        if (h->pipe.st_o[k]) cudaFree(h->pipe.st_o[k]);
        for (cudaEvent_t e : {h->pipe.ev_in[k], h->pipe.ev_used[k], h->pipe.ev_done[k], h->pipe.ev_out[k]})
            if (e) cudaEventDestroy(e);
    }
    if (h->pipe.s_in) cudaStreamDestroy(h->pipe.s_in);
    if (h->pipe.s_out) cudaStreamDestroy(h->pipe.s_out);
    if (h->p2p.epoch) cudaFree(h->p2p.epoch);
    if (h->p2p.arena) cudaFree(h->p2p.arena);
    if (h->own_stream) cudaStreamDestroy(h->stream);
    delete h;
    return AMG1D_OK;
}

int amg1d_set_level(amg1d_t* h, int level, int64_t n_elem, int m, const double* A_lo,
                    const double* A_di, const double* A_up, const double* Dinv,
                    int dinv_is_diagonal, const int64_t* perm, int64_t n_dof_host) {
    if (!h) return AMG1D_ERR_ARG;
    if (!A_lo || !A_di || !A_up || !Dinv) return fail(h, AMG1D_ERR_ARG, "null operator array");
    if (n_elem < 1 || m < 1 || m > 32) return fail(h, AMG1D_ERR_ARG, "need n_elem >= 1 and 1 <= m <= 32");
    const int mm = m * m;
    for (int q = 0; q < mm; ++q)
        if (A_lo[q] != 0.0 || A_up[(size_t)(n_elem - 1) * mm + q] != 0.0)
            return fail(h, AMG1D_ERR_ARG, "A_lo[0] and A_up[n-1] must be zero blocks");
    int st = 0, ilo = 0, iup = 0;
    if (h->opt_compress) detect_structure(A_lo, A_up, n_elem, m, &st, &ilo, &iup);
    RET(alloc_level_common(h, level, n_elem, m, dinv_is_diagonal, perm, n_dof_host, st, ilo, iup));
    Level& lv = h->L[level];
    const int dsz = lv.diag ? m : mm;
    if (!lv.present) { lv.set = true; return AMG1D_OK; }
    // local range of elements to store: [-gl, n + gr) in local indices = [g0, g1) in global ones
    const int64_t g0 = lv.start - lv.gl, g1 = lv.start + lv.n + lv.gr;
    const int64_t chunk = 1 << 18;  // elements per staging chunk (multiple of 32)
    const int64_t c = std::min(chunk, (lv.n + lv.gr + 63) / 32 * 32);
    DevBuf b_lo, b_di, b_up, b_dv;
    // from here on a failure must release what alloc_level_common took (undo_level_alloc)
#define CKU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { undo_level_alloc(h, level); \
        return fail(h, e_ == cudaErrorMemoryAllocation ? AMG1D_ERR_NOMEM : AMG1D_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); } } while (0)
    CKU(b_lo.alloc(c * mm));
    CKU(b_di.alloc(c * mm));
    CKU(b_up.alloc(c * mm));
    CKU(b_dv.alloc(c * dsz));
    double *d_lo = b_lo.p, *d_di = b_di.p, *d_up = b_up.p, *d_dv = b_dv.p;
    int rc = AMG1D_OK;
    // chunks are aligned to tiles of the local storage; the first one starts at local element -32 when
    // the slab has left ghosts (those tiles are zero-filled outside [g0, g1))
    const int64_t l_begin = lv.gl ? -AMG1D_TILE : 0;
    for (int64_t le0 = l_begin; le0 < lv.n + lv.gr && rc == AMG1D_OK; le0 += c) {
        const int64_t cnt = std::min<int64_t>(c, lv.n + lv.gr - le0);
        // global elements of this chunk that exist: [a, b)
        const int64_t a = std::max(g0, lv.start + le0), b = std::min(g1, lv.start + le0 + cnt);
        const int64_t off = a - (lv.start + le0);       // leading elements of the chunk left at zero
        CKU(cudaMemsetAsync(d_lo, 0, (size_t)cnt * mm * 8, h->stream));
        CKU(cudaMemsetAsync(d_di, 0, (size_t)cnt * mm * 8, h->stream));
        CKU(cudaMemsetAsync(d_up, 0, (size_t)cnt * mm * 8, h->stream));
        CKU(cudaMemsetAsync(d_dv, 0, (size_t)cnt * dsz * 8, h->stream));
        if (b > a) {
            CKU(cudaMemcpyAsync(d_lo + off * mm, A_lo + a * mm, (size_t)(b - a) * mm * 8, cudaMemcpyHostToDevice, h->stream));
            CKU(cudaMemcpyAsync(d_di + off * mm, A_di + a * mm, (size_t)(b - a) * mm * 8, cudaMemcpyHostToDevice, h->stream));
            CKU(cudaMemcpyAsync(d_up + off * mm, A_up + a * mm, (size_t)(b - a) * mm * 8, cudaMemcpyHostToDevice, h->stream));
            CKU(cudaMemcpyAsync(d_dv + off * dsz, Dinv + a * dsz, (size_t)(b - a) * dsz * 8, cudaMemcpyHostToDevice, h->stream));
        }
        const int64_t total = amg1d_tiles(cnt) * (int64_t)lv.K * AMG1D_TILE;
        k_repack<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(d_lo, d_di, d_up, d_dv, lv.md,
                                                                         le0, cnt, lv.mat);
        cudaError_t e = cudaStreamSynchronize(h->stream);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) rc = fail(h, AMG1D_ERR_CUDA, "level upload failed: %s", cudaGetErrorString(e));
    }
    if (rc != AMG1D_OK) { undo_level_alloc(h, level); return rc; }
    if (n_elem <= AMG1D_BCR_MIN && !lv.sharded) {   // host copy for the block-Thomas factorisation
        lv.h_lo.assign(A_lo, A_lo + (size_t)n_elem * mm);
        lv.h_di.assign(A_di, A_di + (size_t)n_elem * mm);
        lv.h_up.assign(A_up, A_up + (size_t)n_elem * mm);
    }
    lv.set = true;
    return adopt_device_dinv(h, level);
}

int amg1d_set_level_pattern(amg1d_t* h, int level, int64_t n_elem, int m, int n_head, int n_tail,
                            const double* A_lo, const double* A_di, const double* A_up,
                            const double* Dinv, int dinv_is_diagonal) {
    if (!h) return AMG1D_ERR_ARG;
    if (!A_lo || !A_di || !A_up || !Dinv) return fail(h, AMG1D_ERR_ARG, "null operator array");
    if (n_head < 0 || n_tail < 0 || (int64_t)n_head + n_tail > n_elem)
        return fail(h, AMG1D_ERR_ARG, "need n_head + n_tail <= n_elem");
    if (n_elem < 1 || m < 1 || m > 32) return fail(h, AMG1D_ERR_ARG, "need n_elem >= 1 and 1 <= m <= 32");
    const int mm = m * m;
    const int nb = n_head + 1 + n_tail;
    int st = 0, ilo = 0, iup = 0;
    if (h->opt_compress) detect_structure(A_lo, A_up, nb, m, &st, &ilo, &iup);
    RET(alloc_level_common(h, level, n_elem, m, dinv_is_diagonal, nullptr, n_elem * m, st, ilo, iup));
    Level& lv = h->L[level];
    const int dsz = lv.diag ? m : mm;
    if (!lv.present) { lv.set = true; return AMG1D_OK; }
    DevBuf b_lo, b_di, b_up, b_dv;
    CKU(b_lo.alloc((int64_t)nb * mm));
    CKU(b_di.alloc((int64_t)nb * mm));
    CKU(b_up.alloc((int64_t)nb * mm));
    CKU(b_dv.alloc((int64_t)nb * dsz));
    double *d_lo = b_lo.p, *d_di = b_di.p, *d_up = b_up.p, *d_dv = b_dv.p;
    CKU(cudaMemcpyAsync(d_lo, A_lo, (size_t)nb * mm * 8, cudaMemcpyHostToDevice, h->stream));
    CKU(cudaMemcpyAsync(d_di, A_di, (size_t)nb * mm * 8, cudaMemcpyHostToDevice, h->stream));
    CKU(cudaMemcpyAsync(d_up, A_up, (size_t)nb * mm * 8, cudaMemcpyHostToDevice, h->stream));
    CKU(cudaMemcpyAsync(d_dv, Dinv, (size_t)nb * dsz * 8, cudaMemcpyHostToDevice, h->stream));
    // fill every stored tile, including the spare front tile that holds the left ghost elements
    const int64_t ntiles = amg1d_tiles(lv.n + lv.gr) + 1;
    const int64_t total = ntiles * (int64_t)lv.K * AMG1D_TILE;
    k_fill_pattern<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(
        d_lo, d_di, d_up, d_dv, lv.md, n_elem, n_head, n_tail, lv.start, -(int64_t)lv.gl,
        lv.n + lv.gr, ntiles, lv.mat_alloc);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { undo_level_alloc(h, level); return fail(h, AMG1D_ERR_CUDA, "pattern fill failed: %s", cudaGetErrorString(e)); }
    {   // the distinct block sets as a table tab[set][k], k = tile row: what the pattern-resident legs read
        std::vector<double> tab((size_t)nb * lv.K);
        for (int sidx = 0; sidx < nb; ++sidx)
            for (int k = 0; k < lv.K; ++k) {
                int which, idx;
                amg1d_row_source(lv.md, k, &which, &idx);
                const double* src = which == 0 ? A_lo + (size_t)sidx * mm : which == 1 ? A_di + (size_t)sidx * mm
                                  : which == 2 ? A_up + (size_t)sidx * mm : Dinv + (size_t)sidx * dsz;
                tab[(size_t)sidx * lv.K + k] = src[idx];
            }
        lv.pat_host = std::move(tab);                       // (its size is what undo_level_alloc gives back)
        if (dev_alloc(h, (void**)&lv.pat, (int64_t)lv.pat_host.size() * 8) != AMG1D_OK) {
            lv.pat = nullptr;
            undo_level_alloc(h, level);
            return AMG1D_ERR_NOMEM;
        }
        CKU(cudaMemcpy(lv.pat, lv.pat_host.data(), lv.pat_host.size() * 8, cudaMemcpyHostToDevice));
        lv.pat_head = n_head;
        lv.pat_tail = n_tail;
    }
#undef CKU
    if (n_elem <= AMG1D_BCR_MIN && !lv.sharded) {   // host copy for the block-Thomas factorisation
        lv.h_lo.resize((size_t)n_elem * mm); lv.h_di.resize((size_t)n_elem * mm); lv.h_up.resize((size_t)n_elem * mm);
        for (int64_t el = 0; el < n_elem; ++el) {
            int64_t s = el < n_head ? el : (el >= n_elem - n_tail ? n_head + 1 + (el - (n_elem - n_tail)) : n_head);
            std::copy(A_lo + s * mm, A_lo + (s + 1) * mm, &lv.h_lo[(size_t)el * mm]);
            std::copy(A_di + s * mm, A_di + (s + 1) * mm, &lv.h_di[(size_t)el * mm]);
            std::copy(A_up + s * mm, A_up + (s + 1) * mm, &lv.h_up[(size_t)el * mm]);
        }
    }
    lv.set = true;
    return adopt_device_dinv(h, level);
}

int amg1d_set_level_smoother(amg1d_t* h, int level, const double* S_lo, const double* S_di,
                             const double* S_up) {
    if (!h) return AMG1D_ERR_ARG;
    if (!valid_level(h, level)) return fail(h, AMG1D_ERR_ARG, "level %d out of range", level);
    if (h->finalized) return fail(h, AMG1D_ERR_STATE, "hierarchy already finalized");
    if (!S_lo || !S_di || !S_up) return fail(h, AMG1D_ERR_ARG, "null smoother array");
    Level& lv = h->L[level];
    if (!lv.set) return fail(h, AMG1D_ERR_STATE, "level %d must be set before its smoother operator", level);
    if (lv.sharded || h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "block-tridiagonal smoothers are single-GPU only");
    if (lv.smooth_tri) return fail(h, AMG1D_ERR_STATE, "level %d already has a smoother operator", level);
    CK(cudaSetDevice(h->device));
    const int m = lv.m, mm = m * m;
    const int64_t n = lv.n;
    int st = 0, ilo = 0, iup = 0;
    if (h->opt_compress) detect_structure(S_lo, S_up, n, m, &st, &ilo, &iup);
    lv.smd = amg1d_desc(m, 1, st, ilo, iup);            // the "Dinv" rows of this tile are unused (zeros)
    const int64_t bytes = (amg1d_tiles(n) + 1) * (int64_t)lv.smd.K * AMG1D_TILE * 8;
    RET(dev_alloc(h, (void**)&lv.smat_alloc, bytes));
    CK(cudaMemsetAsync(lv.smat_alloc, 0, (size_t)bytes, h->stream));
    lv.smat = lv.smat_alloc + (int64_t)lv.smd.K * AMG1D_TILE;
    const int64_t c = std::min<int64_t>(1 << 18, (n + 31) / 32 * 32);
    DevBuf b_lo, b_di, b_up, b_dv;
    CK(b_lo.alloc(c * mm));
    CK(b_di.alloc(c * mm));
    CK(b_up.alloc(c * mm));
    CK(b_dv.alloc(c * m));
    double *d_lo = b_lo.p, *d_di = b_di.p, *d_up = b_up.p, *d_dv = b_dv.p;
    cudaMemsetAsync(d_dv, 0, (size_t)c * m * 8, h->stream);
    int rc = AMG1D_OK;
    for (int64_t e0 = 0; e0 < n && rc == AMG1D_OK; e0 += c) {
        const int64_t cnt = std::min<int64_t>(c, n - e0);
        cudaMemcpyAsync(d_lo, S_lo + e0 * mm, (size_t)cnt * mm * 8, cudaMemcpyHostToDevice, h->stream);
        cudaMemcpyAsync(d_di, S_di + e0 * mm, (size_t)cnt * mm * 8, cudaMemcpyHostToDevice, h->stream);
        cudaMemcpyAsync(d_up, S_up + e0 * mm, (size_t)cnt * mm * 8, cudaMemcpyHostToDevice, h->stream);
        const int64_t total = amg1d_tiles(cnt) * (int64_t)lv.smd.K * AMG1D_TILE;
        k_repack<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(d_lo, d_di, d_up, d_dv, lv.smd, e0, cnt, lv.smat);
        cudaError_t e = cudaStreamSynchronize(h->stream);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) rc = fail(h, AMG1D_ERR_CUDA, "smoother upload failed: %s", cudaGetErrorString(e));
    }
    RET(rc);
    lv.smooth_tri = true;
    return AMG1D_OK;
}

static int upload_blocks(amg1d* h, double** dst, const double* src, int64_t count) {
    CK(cudaMalloc((void**)dst, (size_t)std::max<int64_t>(count, 1) * 8));
    CK(cudaMemcpyAsync(*dst, src, (size_t)count * 8, cudaMemcpyHostToDevice, h->stream));
    return AMG1D_OK;
}

int amg1d_set_level_flux(amg1d_t* h, int level, int64_t n_elem, int m, const double* G_lo,
                         const double* G_di, const double* G_up, const double* D_lo, const double* D_di,
                         const double* D_up, const double* C_lo, const double* C_di, const double* C_up,
                         const double* Minv, int minv_is_constant) {
    if (!h) return AMG1D_ERR_ARG;
    const double* src[9] = {G_lo, G_di, G_up, D_lo, D_di, D_up, C_lo, C_di, C_up};
    for (const double* p : src) if (!p) return fail(h, AMG1D_ERR_ARG, "null flux operator array");
    if (!Minv) return fail(h, AMG1D_ERR_ARG, "null mass-matrix inverse");
    if (!valid_level(h, level)) return fail(h, AMG1D_ERR_ARG, "level %d out of range", level);
    if (h->finalized) return fail(h, AMG1D_ERR_STATE, "hierarchy already finalized");
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "device-side set-up is single-GPU only");
    if (n_elem < 1 || m < 1 || m > AMG1D_BCR_MAXM) return fail(h, AMG1D_ERR_ARG, "need n_elem >= 1 and 1 <= m <= 32");
    Level& lv = h->L[level];
    if (lv.set) return fail(h, AMG1D_ERR_STATE, "level %d already set", level);
    CK(cudaSetDevice(h->device));
    free_flux(h, lv);                              // left over from an earlier, failed attempt
    const int64_t cnt = n_elem * m * m;
    for (int k = 0; k < 9; ++k) {
        RET(upload_blocks(h, &lv.flux[k], src[k], cnt));
        h->device_bytes += cnt * 8;
    }
    DevBuf minv;
    RET(upload_blocks(h, &minv.p, Minv, minv_is_constant ? (int64_t)m * m : cnt));
    lv.n = n_elem; lv.m = m;                       // for free_flux if the installation fails
    return install_from_flux(h, level, n_elem, m, lv.flux, minv.p, minv_is_constant);
}

int amg1d_coarsen_level(amg1d_t* h, int level, const double* Minv_coarse, int minv_is_constant) {
    if (!h) return AMG1D_ERR_ARG;
    if (level < 0 || level >= h->n_levels - 1) return fail(h, AMG1D_ERR_ARG, "level %d has no coarser level", level);
    if (h->finalized) return fail(h, AMG1D_ERR_STATE, "hierarchy already finalized");
    if (!Minv_coarse) return fail(h, AMG1D_ERR_ARG, "null mass-matrix inverse");
    Level& lf = h->L[level];
    Level& lc = h->L[level + 1];
    Transfer& t = h->T[level];
    if (!lf.set || !lf.flux[0]) return fail(h, AMG1D_ERR_STATE, "level %d has no flux operators (amg1d_set_level_flux / amg1d_coarsen_level)", level);
    if (!t.set) return fail(h, AMG1D_ERR_STATE, "transfer %d must be set before amg1d_coarsen_level", level);
    if (lc.set) return fail(h, AMG1D_ERR_STATE, "level %d already set", level + 1);
    if (!t.single_parent_uniform)
        return fail(h, AMG1D_ERR_UNSUPPORTED, "device-side coarsening needs a single-parent transfer with parent[e] = e / ratio");
    if (t.n_fine != lf.n || t.mf != lf.m) return fail(h, AMG1D_ERR_ARG, "transfer %d does not match level %d", level, level);
    CK(cudaSetDevice(h->device));
    const int mc = t.mc;
    const int64_t nc = t.n_coarse, cnt = nc * mc * mc;
    free_flux(h, lc);
    lc.n = nc; lc.m = mc;
    for (int k = 0; k < 9; ++k) {
        CK(cudaMalloc((void**)&lc.flux[k], (size_t)cnt * 8));
        h->device_bytes += cnt * 8;
    }
    const TransferMap tm = make_map_closed(t);
    const unsigned grid = (unsigned)((cnt + 127) / 128);
    for (int k = 0; k < 3; ++k)
        k_galerkin_tri<<<grid, 128, 0, h->stream>>>(lf.flux[3 * k], lf.flux[3 * k + 1], lf.flux[3 * k + 2], t.P0, tm,
                                                     t.mf, mc, lc.flux[3 * k], lc.flux[3 * k + 1], lc.flux[3 * k + 2]);
    LAUNCH_CHECK();
    DevBuf minv;
    RET(upload_blocks(h, &minv.p, Minv_coarse, minv_is_constant ? (int64_t)mc * mc : cnt));
    return install_from_flux(h, level + 1, nc, mc, lc.flux, minv.p, minv_is_constant);
}

int amg1d_coarsen_level_galerkin(amg1d_t* h, int level, int64_t n_coarse_elem, int dinv_is_diagonal,
                                 const int64_t* perm_coarse, int64_t n_dof_host_coarse) {
    if (!h) return AMG1D_ERR_ARG;
    if (level < 0 || level >= h->n_levels - 1) return fail(h, AMG1D_ERR_ARG, "level %d has no coarser level", level);
    if (h->finalized) return fail(h, AMG1D_ERR_STATE, "hierarchy already finalized");
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "device-side set-up is single-GPU only");
    Level& lf = h->L[level];
    Level& lc = h->L[level + 1];
    Transfer& t = h->T[level];
    if (!lf.set) return fail(h, AMG1D_ERR_STATE, "level %d must be set before amg1d_coarsen_level_galerkin", level);
    if (!t.set) return fail(h, AMG1D_ERR_STATE, "transfer %d must be set before amg1d_coarsen_level_galerkin", level);
    if (lc.set) return fail(h, AMG1D_ERR_STATE, "level %d already set", level + 1);
    if (lf.smooth_tri) return fail(h, AMG1D_ERR_UNSUPPORTED, "level %d carries a tridiagonal smoother operator", level);
    if (t.n_fine != lf.n || t.mf != lf.m) return fail(h, AMG1D_ERR_ARG, "transfer %d does not match level %d", level, level);
    const int mc = t.mc, mf = t.mf;
    const int64_t nc = n_coarse_elem;
    if (mc > AMG1D_BCR_MAXM) return fail(h, AMG1D_ERR_ARG, "coarse block size %d too large", mc);
    if (nc < t.n_coarse || nc > t.n_coarse + (t.P1 ? 1 : 0))
        return fail(h, AMG1D_ERR_ARG, "transfer %d reaches coarse element %lld but n_coarse_elem is %lld", level,
                    (long long)t.n_coarse - 1, (long long)nc);
    CK(cudaSetDevice(h->device));
    // fine operator as element-block arrays, coarse result, child pointers of an explicit parent map
    DevBuf F[3], C[3], dband, dcp;
    const int64_t fcnt = lf.n * mf * mf, ccnt = nc * mc * mc;
    for (auto& b : F) CK(b.alloc(fcnt));
    for (auto& b : C) CK(b.alloc(ccnt));
    CK(dband.alloc(2));
    CK(cudaMemsetAsync(dband.p, 0, 16, h->stream));
    k_bcr_extract<<<(unsigned)((fcnt + 255) / 256), 256, 0, h->stream>>>(lf.mat, lf.md, lf.n, F[0].p, F[1].p, F[2].p);
    TransferMap tm = make_map(t);
    tm.n_coarse = nc;
    tm.cp = nullptr;
    if (!t.closed) {
        if (t.h_parent.size() != (size_t)t.n_fine) return fail(h, AMG1D_ERR_STATE, "transfer %d has no parent map", level);
        std::vector<int64_t> cp((size_t)nc + 2);
        int64_t e = 0;
        for (int64_t q = 0; q < nc + 2; ++q) {
            while (e < t.n_fine && t.h_parent[(size_t)e] < q - 1) ++e;
            cp[(size_t)q] = e;
        }
        CK(dcp.alloc((int64_t)cp.size()));
        CK(cudaMemcpyAsync(dcp.p, cp.data(), cp.size() * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));         // cp is a local vector
        tm.cp = reinterpret_cast<const int64_t*>(dcp.p);
    } else {
        tm.parent = nullptr;
    }
    k_galerkin_general<<<(unsigned)((ccnt + 127) / 128), 128, 0, h->stream>>>(F[0].p, F[1].p, F[2].p, t.P0, t.P1, tm, mf,
                                                                               mc, nc, C[0].p, C[1].p, C[2].p, dband.p);
    double band[2] = {0.0, 0.0};
    CK(cudaMemcpyAsync(band, dband.p, 16, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    if (band[0] > 1e-11 * band[1])
        return fail(h, AMG1D_ERR_ARG, "level %d: L' A L is not block tridiagonal (outer band %.3e vs diagonal %.3e)",
                    level + 1, band[0], band[1]);
    double* dA[3] = {C[0].p, C[1].p, C[2].p};
    return install_from_blocks(h, level + 1, nc, mc, dA, dinv_is_diagonal, perm_coarse,
                               perm_coarse ? n_dof_host_coarse : nc * mc);
}

int amg1d_get_level(amg1d_t* h, int level, double* A_lo, double* A_di, double* A_up, double* Dinv) {
    if (!h) return AMG1D_ERR_ARG;
    if (!valid_level(h, level) || !h->L[level].set) return fail(h, AMG1D_ERR_ARG, "level %d is not set", level);
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "per-level host operations are single-GPU only");
    if (!A_lo || !A_di || !A_up || !Dinv) return fail(h, AMG1D_ERR_ARG, "null output array");
    Level& lv = h->L[level];
    CK(cudaSetDevice(h->device));
    const int64_t cnt = lv.n * lv.m * lv.m, dcnt = lv.n * (lv.diag ? lv.m : lv.m * lv.m);
    DevBuf d[3], dv;
    for (auto& b : d) CK(b.alloc(cnt));
    CK(dv.alloc(dcnt));
    k_bcr_extract<<<(unsigned)((cnt + 255) / 256), 256, 0, h->stream>>>(lv.mat, lv.md, lv.n, d[0].p, d[1].p, d[2].p);
    k_extract_dinv<<<(unsigned)((dcnt + 255) / 256), 256, 0, h->stream>>>(lv.mat, lv.md, lv.n, dv.p);
    LAUNCH_CHECK();
    double* out[3] = {A_lo, A_di, A_up};
    for (int k = 0; k < 3; ++k) CK(cudaMemcpyAsync(out[k], d[k].p, (size_t)cnt * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(Dinv, dv.p, (size_t)dcnt * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AMG1D_OK;
}

static int transfer_common(amg1d_t* h, int level, int64_t n_fine, int mf, int mc) {
    if (!h) return AMG1D_ERR_ARG;
    if (level < 0 || level >= h->n_levels - 1) return fail(h, AMG1D_ERR_ARG, "transfer %d out of range", level);
    if (h->finalized) return fail(h, AMG1D_ERR_STATE, "hierarchy already finalized");
    if (h->T[level].set) return fail(h, AMG1D_ERR_STATE, "transfer %d already set", level);
    if (n_fine < 1 || mf < 1 || mc < 1 || mf > 32 || mc > 32) return fail(h, AMG1D_ERR_ARG, "bad transfer shape");
    CK(cudaSetDevice(h->device));
    return AMG1D_OK;
}

int amg1d_set_transfer(amg1d_t* h, int level, int64_t n_fine_elem, int m_f, int m_c,
                       const int64_t* parent, const double* P0, const double* P1) {
    RET(transfer_common(h, level, n_fine_elem, m_f, m_c));
    if (!parent || !P0) return fail(h, AMG1D_ERR_ARG, "null transfer array");
    if (h->nranks > 1 && !h->L[level].set)
        return fail(h, AMG1D_ERR_STATE, "multi-GPU: level %d must be set before its transfer", level);
    const bool slab = h->L[level].set && h->L[level].sharded;   // keep this rank's slab of blocks only (below)
    Transfer& t = h->T[level];
    t.n_fine = n_fine_elem; t.mf = m_f; t.mc = m_c; t.period = 0;
    int64_t maxp = -1;
    for (int64_t e = 0; e < n_fine_elem; ++e) {
        if (parent[e] < -1 || (e > 0 && parent[e] < parent[e - 1]))
            return fail(h, AMG1D_ERR_ARG, "parent map must be non-decreasing and >= -1 (element %lld)", (long long)e);
        maxp = std::max(maxp, parent[e]);
    }
    t.n_coarse = maxp + 1;  // validated against the coarse level at finalize (P1 may reach maxp + 1)
    // closed-form detection: parent[e] = (e + shift) / ratio + base, with base = parent[0], the first
    // run of equal parents fixing the shift and the second run the ratio
    {
        const int64_t base = parent[0];
        int64_t c0 = 1;
        while (c0 < n_fine_elem && parent[c0] == base) ++c0;
        int64_t c1 = 0;
        while (c0 + c1 < n_fine_elem && parent[c0 + c1] == base + 1) ++c1;
        const bool second_run_complete = c0 + c1 < n_fine_elem;
        int64_t ratio = second_run_complete ? c1 : std::max(c0, c1);
        if (ratio < 1) ratio = 1;
        const int64_t shift = ratio - c0;
        bool closed = ratio <= 1024 && shift >= 0 && shift < ratio;
        for (int64_t e = 0; e < n_fine_elem && closed; ++e) closed = parent[e] == (e + shift) / ratio + base;
        t.closed = closed;
        t.ratio = closed ? (int)ratio : 1;
        t.shift = closed ? (int)shift : 0;
        t.base = closed ? (int)base : 0;
    }
    t.single_parent_uniform = t.closed && P1 == nullptr && t.shift == 0 && t.base == 0;
    const int bs = m_f * m_c;
    if (slab) {
        // A sharded level runs the fused legs only: they need the closed-form parent map (checked again at
        // amg1d_finalize) and index the blocks by global fine element.  This rank keeps the blocks its legs can
        // touch: its slab, the ghost elements and the children of the coarse elements next to them.
        if (!t.closed)
            return fail(h, AMG1D_ERR_UNSUPPORTED, "transfer %d: a sharded level needs parent[e] = (e + shift) / ratio + base", level);
        const Level& lf = h->L[level];
        const int64_t margin = h->ghost_depth + 2 * (int64_t)t.ratio + 2;
        const int64_t lo = std::max<int64_t>(0, lf.start - margin), hi = std::min<int64_t>(n_fine_elem, lf.start + lf.n + margin);
        t.p_first = lo;
        t.nblk = hi - lo;
        RET(dev_alloc(h, (void**)&t.P0, t.nblk * bs * 8));
        CK(cudaMemcpy(t.P0, P0 + lo * bs, (size_t)t.nblk * bs * 8, cudaMemcpyHostToDevice));
        if (P1) {
            RET(dev_alloc(h, (void**)&t.P1, t.nblk * bs * 8));
            CK(cudaMemcpy(t.P1, P1 + lo * bs, (size_t)t.nblk * bs * 8, cudaMemcpyHostToDevice));
        }
        t.set = true;
        return AMG1D_OK;
    }
    RET(dev_alloc(h, (void**)&t.P0, n_fine_elem * bs * 8));
    CK(cudaMemcpy(t.P0, P0, (size_t)n_fine_elem * bs * 8, cudaMemcpyHostToDevice));
    if (P1) {
        RET(dev_alloc(h, (void**)&t.P1, n_fine_elem * bs * 8));
        CK(cudaMemcpy(t.P1, P1, (size_t)n_fine_elem * bs * 8, cudaMemcpyHostToDevice));
    }
    t.nblk = n_fine_elem;
    RET(dev_alloc(h, (void**)&t.parent, n_fine_elem * 8));
    CK(cudaMemcpy(t.parent, parent, (size_t)n_fine_elem * 8, cudaMemcpyHostToDevice));
    t.set = true;
    // child pointers are built at finalize once the coarse element count is known
    t.h_parent.assign(parent, parent + n_fine_elem);
    return AMG1D_OK;
}

int amg1d_set_transfer_pattern(amg1d_t* h, int level, int64_t n_fine_elem, int m_f, int m_c,
                               int ratio, int shift, int base, int period, int n_head, int n_tail,
                               const double* P0_pat, const double* P1_pat) {
    RET(transfer_common(h, level, n_fine_elem, m_f, m_c));
    if (!P0_pat) return fail(h, AMG1D_ERR_ARG, "null transfer array");
    if (ratio < 1 || period < 1 || shift < 0 || shift >= ratio || n_head < 0 || n_tail < 0 ||
        (int64_t)n_head + n_tail > n_fine_elem)
        return fail(h, AMG1D_ERR_ARG, "bad transfer pattern");
    Transfer& t = h->T[level];
    t.n_fine = n_fine_elem; t.mf = m_f; t.mc = m_c;
    t.ratio = ratio; t.shift = shift; t.base = base; t.period = period; t.n_head = n_head; t.n_tail = n_tail;
    t.n_coarse = (n_fine_elem - 1 + shift) / ratio + base + 1;
    t.single_parent_uniform = (P1_pat == nullptr) && shift == 0 && base == 0;
    t.closed = true;
    const int bs = m_f * m_c;
    t.nblk = n_head + period + n_tail;
    RET(dev_alloc(h, (void**)&t.P0, t.nblk * bs * 8));
    CK(cudaMemcpy(t.P0, P0_pat, (size_t)t.nblk * bs * 8, cudaMemcpyHostToDevice));
    if (P1_pat) {
        RET(dev_alloc(h, (void**)&t.P1, t.nblk * bs * 8));
        CK(cudaMemcpy(t.P1, P1_pat, (size_t)t.nblk * bs * 8, cudaMemcpyHostToDevice));
    }
    t.set = true;
    return AMG1D_OK;
}

int amg1d_finalize(amg1d_t* h) {
    if (!h) return AMG1D_ERR_ARG;
    if (h->finalized) return fail(h, AMG1D_ERR_STATE, "hierarchy already finalized");
    CK(cudaSetDevice(h->device));
    for (int l = 0; l < h->n_levels; ++l)
        if (!h->L[l].set) return fail(h, AMG1D_ERR_STATE, "level %d was never set", l);
    if (h->nranks > 1 && h->gather_level < 0)
        return fail(h, AMG1D_ERR_UNSUPPORTED, "multi-GPU: the coarsest levels must fall below the shard "
                    "threshold (%lld elements per rank) so that they can be gathered", (long long)h->shard_min);
    int64_t maxlen = 0;
    for (int l = 0; l < h->n_levels - 1; ++l) {
        Transfer& t = h->T[l];
        if (!t.set) return fail(h, AMG1D_ERR_STATE, "transfer %d was never set", l);
        Level& lf = h->L[l];
        Level& lc = h->L[l + 1];
        if (t.n_fine != lf.n_glob || t.mf != lf.m || t.mc != lc.m)
            return fail(h, AMG1D_ERR_ARG, "transfer %d does not match its levels (n_fine %lld vs %lld, m_f %d vs %d, m_c %d vs %d)",
                        l, (long long)t.n_fine, (long long)lf.n_glob, t.mf, lf.m, t.mc, lc.m);
        const int64_t need = t.n_coarse + (t.P1 ? 1 : 0);
        if (t.n_coarse > lc.n_glob || need < lc.n_glob)
            return fail(h, AMG1D_ERR_ARG, "transfer %d reaches coarse element %lld but level %d has %lld elements",
                        l, (long long)t.n_coarse - 1, l + 1, (long long)lc.n_glob);
        t.n_coarse = lc.n_glob;
        // f_down gathers coarse element q in the thread of its first P0-child first(q) = (q - base) *
        // ratio - shift: that child must exist for every q, and first(0) must not be clamped
        t.fusable = t.closed && (-(int64_t)t.base * t.ratio - t.shift) >= 0 &&
                    ((lc.n_glob - 1 - t.base) * (int64_t)t.ratio - t.shift) < t.n_fine;
        if (lf.sharded) {
            if (!t.fusable)
                return fail(h, AMG1D_ERR_UNSUPPORTED, "transfer %d: sharded levels need a closed-form parent map "
                            "parent[e] = (e + shift) / ratio + base in which every coarse element has a first child", l);
            if (lf.n < 2 * h->ghost_depth)
                return fail(h, AMG1D_ERR_UNSUPPORTED, "transfer %d: slab of %lld elements is too small", l,
                            (long long)lf.n);
            // Every rank's coarse slab must be gathered from its own fine slab plus at most `reach`
            // ghost elements per edge (0 for single-parent transfers aligned to the agglomerates).
            int64_t reach = 0, extra = 0;
            for (int r = 0; r < h->nranks; ++r) {
                const int64_t f0 = slab_start(lf.n_glob, h->nranks, r), f1 = f0 + slab_size(lf.n_glob, h->nranks, r);
                const int64_t c0 = slab_start(lc.n_glob, h->nranks, r), c1 = c0 + slab_size(lc.n_glob, h->nranks, r);
                auto first = [&](int64_t q) {
                    int64_t v = (q - t.base) * (int64_t)t.ratio - t.shift;
                    return std::min<int64_t>(std::max<int64_t>(v, 0), t.n_fine);
                };
                const int64_t lo_child = first(t.P1 ? c0 - 1 : c0);   // first fine element rank r's coarse slab reads
                const int64_t hi_child = first(c1);                   // one past the last
                reach = std::max(reach, std::max(f0 - lo_child, hi_child - f1));
                extra = std::max(extra, first(c1 - 1) + 1 - f1);      // owners (first P0-children) right of the slab
                const bool plain = !t.P1 && t.shift == 0 && t.base == 0;   // window without extra halo
                if (plain ? (lo_child != f0 || hi_child != f1)
                          : (lo_child > f0 + t.ratio || hi_child < f1 - t.ratio || f0 - lo_child > t.ratio ||
                             hi_child - f1 > t.ratio))
                    return fail(h, AMG1D_ERR_UNSUPPORTED, "transfer %d: rank %d's slab of level %d [%lld, %lld) "
                                "is not aligned with its slab of level %d (children [%lld, %lld))", l, r, l,
                                (long long)f0, (long long)f1, l + 1, (long long)lo_child, (long long)hi_child);
            }
            if (reach < 0) reach = 0;
            if (extra < 0) extra = 0;
            if (reach > 64)
                return fail(h, AMG1D_ERR_UNSUPPORTED, "transfer %d: slabs of levels %d and %d are misaligned "
                            "by %lld elements", l, l, l + 1, (long long)reach);
            t.reach = (int)reach;
            t.cover_extra = extra;
        }
        if (t.parent) {  // build child pointers: cp[q] = first e with parent[e] >= q - 1, q = 0..n_coarse+1
            std::vector<int64_t> cp((size_t)lc.n_glob + 2);
            int64_t e = 0;
            for (int64_t q = 0; q < lc.n_glob + 2; ++q) {
                while (e < t.n_fine && t.h_parent[e] < q - 1) ++e;
                cp[q] = e;
            }
            t.h_parent.clear();
            t.h_parent.shrink_to_fit();
            RET(dev_alloc(h, (void**)&t.cp, (int64_t)cp.size() * 8));
            CK(cudaMemcpy(t.cp, cp.data(), cp.size() * 8, cudaMemcpyHostToDevice));
        }
    }
    // a non-root rank keeps only its slab of the first gathered level (vectors, no operator)
    if (h->nranks > 1 && h->rank > 0) {
        Level& lg = h->L[h->gather_level];
        lg.proxy = true;
        lg.n = slab_size(lg.n_glob, h->nranks, h->rank);
        lg.start = slab_start(lg.n_glob, h->nranks, h->rank);
    }
    h->partial_cap = AMG1D_RED_BLOCKS;
#ifdef AMG1D_WITH_NCCL
    if (h->nranks > 1 && h->opt_p2p) RET(p2p_alloc_arena(h));
#endif
    for (const Level& lv : h->L) {
        if (!lv.present && !lv.proxy) continue;
        maxlen = std::max(maxlen, lv.n * lv.m);
        h->partial_cap = std::max<int64_t>(h->partial_cap, lv.n / (lv.m > 5 ? 16 : FUSED_B / 2) + 16);
    }
    RET(column_alloc(h, h->res, false));
    RET(vec_alloc(h, h->scratch, maxlen, 1));
    RET(dev_alloc(h, (void**)&h->res.scal, 64 * 8));
    CK(cudaMallocHost(&h->h_scal, 64 * 8));
    if (h->L[h->n_levels - 1].present) RET(factor_coarsest(h));
    RET(build_tail(h));
    {
        const cudaError_t pe = pipe_configure_all();          // shared-memory limit of the pipelined legs (f_*_pp)
        if (pe != cudaSuccess) return fail(h, AMG1D_ERR_CUDA, "pipelined leg configuration failed: %s", cudaGetErrorString(pe));
    }
    // the row-per-thread legs of the large-block levels use > 48 KB of dynamic shared memory
    for (int l = 0; l + 1 < h->n_levels; ++l) {
        const Level& lv = h->L[l];
        if (!lv.present || !h->T[l].fusable) continue;
        bool have = false;
        cudaError_t e = rows_configure(lv.md, h->T[l].mc, &have);
        if (e != cudaSuccess)
            return fail(h, AMG1D_ERR_CUDA, "r_down / r_up configuration failed on level %d: %s", l, cudaGetErrorString(e));
    }
    for (auto& lv : h->L) free_flux(h, lv);
    CK(cudaStreamSynchronize(h->stream));
#ifdef AMG1D_WITH_NCCL
    if (h->nranks > 1) RET(p2p_connect(h, h->res));           // collective: every rank reaches this point or none does
#endif
    h->finalized = true;
    return AMG1D_OK;
}

// ---- hot path ----------------------------------------------------------------------------------------
int amg1d_dev_set_problem(amg1d_t* h, const double* x0, const double* b) {
    RET(check_ready(h));
    Level& l0 = h->L[0];
    Column::Vecs& v0 = h->res.lv[0];
    h->norm_valid = false;
    if (!b && !h->dev_problem)
        return fail(h, AMG1D_ERR_STATE, "amg1d_dev_set_problem: b == NULL keeps the resident right-hand side, but that "
                    "was overwritten by a per-level host operation");
    if (b) {
        RET(to_device(h, 0, b, v0.b.p));
        if (l0.sharded) RET(op_halo(h, v0.b.p, l0.n, l0.m));
        h->dev_problem = true;
    }
    if (v0.cur != 0) v0.cur = 0;
    if (x0) RET(to_device(h, 0, x0, v0.x[0].p));
    else CK(cudaMemsetAsync(v0.x[0].p, 0, (size_t)v0.x[0].len * 8, h->stream));
    // ghosts of the new iterate.  (The two-sided exchange also orders this call after the neighbours' last
    // peer-memory push of an earlier cycle, which targets the same ghost slots.)
    if (l0.sharded) RET(op_halo(h, v0.x[0].p, l0.n, l0.m));
    return AMG1D_OK;
}

int amg1d_dev_fill_rhs_random(amg1d_t* h, uint64_t seed) {
    RET(check_ready(h));
    Level& l0 = h->L[0];
    Column::Vecs& v0 = h->res.lv[0];
    if (l0.perm) return fail(h, AMG1D_ERR_UNSUPPORTED, "random rhs only for unpermuted (DG) fine levels");
    h->norm_valid = false;
    k_fill_random<<<1184, 256, 0, h->stream>>>(v0.b.p, v0.b.len, seed, l0.start * l0.m);
    LAUNCH_CHECK();
    h->dev_problem = true;
    v0.cur = 0;
    CK(cudaMemsetAsync(v0.x[0].p, 0, (size_t)v0.x[0].len * 8, h->stream));
    if (l0.sharded) RET(op_halo(h, v0.b.p, l0.n, l0.m, v0.x[0].p, l0.n, l0.m));
    return AMG1D_OK;
}

int amg1d_dev_assemble_rhs(amg1d_t* h, int kind, int nq, const double* xi, const double* W, int n_basis,
                           int n_terms, const double* terms, double xin, double xout, const double* vertices,
                           int n_fix, const int64_t* fix_slot, const double* fix_val, const int* fix_op) {
    RET(check_ready(h));
    Level& l0 = h->L[0];
    Column::Vecs& v0 = h->res.lv[0];
    if (kind < 0 || kind > 1) return fail(h, AMG1D_ERR_ARG, "kind must be 0 (DG-type level) or 1 (CG level in group form)");
    if (!xi || !W || !terms || nq < 1 || nq > AMG1D_RHS_MAXQ || n_basis < 1 || n_basis > AMG1D_RHS_MAXM ||
        n_terms < 1 || n_terms > AMG1D_RHS_MAXT)
        return fail(h, AMG1D_ERR_ARG, "need 1 <= nq <= %d, 1 <= n_basis <= %d, 1 <= n_terms <= %d", AMG1D_RHS_MAXQ,
                    AMG1D_RHS_MAXM, AMG1D_RHS_MAXT);
    if (n_fix < 0 || (n_fix > 0 && (!fix_slot || !fix_val || !fix_op))) return fail(h, AMG1D_ERR_ARG, "bad fix list");
    if (l0.perm) return fail(h, AMG1D_ERR_UNSUPPORTED, "device right-hand sides need level 0 in device order (no perm): "
                             "DG-type levels, or CG levels uploaded in group order");
    if ((kind == 0 && n_basis != l0.m) || (kind == 1 && n_basis != l0.m + 1))
        return fail(h, AMG1D_ERR_ARG, "n_basis %d does not match level 0 (block size %d)", n_basis, l0.m);
    for (int t = 0; t < n_terms; ++t) {
        const double k = terms[5 * t], pw = terms[5 * t + 2];
        if (!(k == 0.0 || k == 1.0 || k == 2.0 || k == 3.0) || !(pw >= 0.0 && pw <= 16.0 && pw == std::floor(pw)))
            return fail(h, AMG1D_ERR_ARG, "term %d: kind must be 0 (1), 1 (cos), 2 (sin), 3 (exp); pow an integer in [0, 16]", t);
    }
    RhsSpec sp = {};
    sp.kind = kind; sp.nq = nq; sp.m = n_basis; sp.n_terms = n_terms;
    for (int q = 0; q < nq; ++q) {
        sp.xi[q] = xi[q];
        for (int i = 0; i < n_basis; ++i) sp.W[q * AMG1D_RHS_MAXM + i] = W[q * n_basis + i];
    }
    memcpy(sp.terms, terms, sizeof(double) * 5 * n_terms);
    sp.xin = xin; sp.xout = xout;
    sp.n_glob = kind == 0 ? l0.n_glob : l0.n_glob - 1;        // CG: n + 1 vertex groups on n elements
    DevBuf dvert, dfs, dfv, dfo;
    if (vertices) {
        CK(dvert.alloc(sp.n_glob + 1));
        CK(cudaMemcpyAsync(dvert.p, vertices, (size_t)(sp.n_glob + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    }
    h->norm_valid = false;
    // the slab with its ghost elements (their right-hand side feeds the recomputed halo of the fused legs)
    const int64_t e0 = -(int64_t)l0.gl, e1 = l0.n + l0.gr;
    CK(cudaMemsetAsync(v0.b.p + e0 * l0.m, 0, (size_t)(e1 - e0) * l0.m * 8, h->stream));
    k_assemble_rhs<<<(unsigned)((e1 - e0 + 127) / 128), 128, 0, h->stream>>>(sp, dvert.p && vertices ? dvert.p : nullptr,
                                                                          l0.start, e0, e1, e1 * l0.m, v0.b.p, 0);
    h->launch_counter++;
    LAUNCH_CHECK();
    if (kind == 1 && l0.gl) {
        // the first ghost group's vertex also receives fe[1] of the element left of it, which no thread of this
        // rank visits: recompute that one element's contribution
        k_assemble_rhs<<<1, 1, 0, h->stream>>>(sp, dvert.p && vertices ? dvert.p : nullptr, l0.start, e0 - 1, e0,
                                               e1 * l0.m, v0.b.p, 1);
        h->launch_counter++;
        LAUNCH_CHECK();
    }
    if (n_fix) {
        CK(dfs.alloc(n_fix)); CK(dfv.alloc(n_fix)); CK(dfo.alloc(n_fix));
        CK(cudaMemcpyAsync(dfs.p, fix_slot, (size_t)n_fix * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(dfv.p, fix_val, (size_t)n_fix * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(dfo.p, fix_op, (size_t)n_fix * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        k_apply_fixes<<<1, 32, 0, h->stream>>>(v0.b.p, l0.start * l0.m, e0 * l0.m, e1 * l0.m, n_fix,
                                               reinterpret_cast<const int64_t*>(dfs.p), dfv.p,
                                               reinterpret_cast<const int*>(dfo.p));
        h->launch_counter++;
        LAUNCH_CHECK();
    }
    v0.cur = 0;
    CK(cudaMemsetAsync(v0.x[0].p, 0, (size_t)v0.x[0].len * 8, h->stream));
    if (l0.sharded) RET(op_halo(h, v0.x[0].p, l0.n, l0.m));      // (zero ghosts; orders this call after earlier pushes)
    CK(cudaStreamSynchronize(h->stream));         // the staging buffers above are released on return
    h->dev_problem = true;
    return AMG1D_OK;
}

int amg1d_dev_get_rhs(amg1d_t* h, double* b) {
    RET(check_dev_problem(h));
    if (!b) return fail(h, AMG1D_ERR_ARG, "null b");
    return to_host(h, 0, h->res.lv[0].b.p, b);
}

int amg1d_dev_solve(amg1d_t* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters, double* res) {
    RET(check_dev_problem(h));
    if (!res || !iters) return fail(h, AMG1D_ERR_ARG, "null argument");
    if (maxiter < 0) return fail(h, AMG1D_ERR_ARG, "maxiter must be >= 0");
    return multigrid_run(h, maxiter, tol, nPre, nPost, alpha, iters, res, nullptr, nullptr);
}

int amg1d_dev_vcycle(amg1d_t* h, int nPre, int nPost, double alpha, int with_residual_norm) {
    RET(check_dev_problem(h));
    return run_vcycle(h, h->res, nPre, nPost, alpha, with_residual_norm != 0);
}

int amg1d_dev_residual_norm(amg1d_t* h, double* res) {
    RET(check_dev_problem(h));
    if (!h->norm_valid) RET(op_resnorm(h, h->res, 0, 0));
    RET(read_scalars(h, h->res, 1));
    if (res) *res = h->h_scal[0];
    return AMG1D_OK;
}

int amg1d_dev_rhs_norm(amg1d_t* h, double* nb) {
    RET(check_dev_problem(h));
    // slot 2 (as amg1d_solve): slot 0 caches ||b - A x|| of a norm-fused V-cycle (norm_valid) and must survive
    Column::Vecs& v0 = h->res.lv[0];
    RET(op_norm(h, h->res, v0.b.p, nullptr, v0.b.len, 2));
    RET(read_scalars(h, h->res, 3));
    if (nb) *nb = h->h_scal[2];
    return AMG1D_OK;
}

int amg1d_dev_get_solution(amg1d_t* h, double* x) {
    RET(check_ready(h));
    if (!x) return fail(h, AMG1D_ERR_ARG, "null x");
    return to_host(h, 0, h->res.lv[0].x[h->res.lv[0].cur].p, x);
}

// ---- multi-column resident problems ----------------------------------------------------------------------------
int amg1d_dev_set_problems(amg1d_t* h, int k, const double* X0, const double* B) {
    RET(check_multi(h, false));
    RET(check_cols(h, k));
    if (!B) return fail(h, AMG1D_ERR_ARG, "null B");
    RET(multi_alloc(h, k));
    amg1d::Multi& M = h->multi;
    const int64_t nh = h->L[0].n_host;
    M.k = 0;
    M.norm_valid = false;
    for (int c = 0; c < k; ++c) {
        auto& v = M.col[(size_t)c].lv[0];
        RET(to_device(h, 0, B + c * nh, v.b.p));
        v.cur = 0;
        if (X0) RET(to_device(h, 0, X0 + c * nh, v.x[0].p));
        else CK(cudaMemsetAsync(v.x[0].p, 0, (size_t)v.x[0].len * 8, h->stream));
    }
    M.k = k;
    M.rhs_consumed = false;
    return AMG1D_OK;
}

int amg1d_dev_fill_rhs_random_multi(amg1d_t* h, int k, uint64_t seed) {
    RET(check_multi(h, false));
    RET(check_cols(h, k));
    Level& l0 = h->L[0];
    if (l0.perm) return fail(h, AMG1D_ERR_UNSUPPORTED, "random rhs only for unpermuted (DG) fine levels");
    RET(multi_alloc(h, k));
    amg1d::Multi& M = h->multi;
    M.norm_valid = false;
    for (int c = 0; c < k; ++c) {
        auto& v = M.col[(size_t)c].lv[0];
        k_fill_random<<<1184, 256, 0, h->stream>>>(v.b.p, v.b.len, seed + (uint64_t)c, l0.start * l0.m);
        LAUNCH_CHECK();
        v.cur = 0;
        CK(cudaMemsetAsync(v.x[0].p, 0, (size_t)v.x[0].len * 8, h->stream));
    }
    M.k = k;
    M.rhs_consumed = false;
    return AMG1D_OK;
}

int amg1d_dev_vcycle_multi(amg1d_t* h, int nPre, int nPost, double alpha, int zero_guess, int with_residual_norms) {
    RET(check_multi(h, true));
    amg1d::Multi& M = h->multi;
    int act[MULTI_MAX_COLS];
    for (int c = 0; c < M.k; ++c) act[c] = c;
    M.norm_valid = false;
    RET(run_vcycle_multi(h, act, M.k, nPre, nPost, alpha, with_residual_norms != 0, zero_guess != 0));
    M.norm_valid = with_residual_norms != 0;
    return AMG1D_OK;
}

int amg1d_dev_residual_norms(amg1d_t* h, double* res) {
    RET(check_multi(h, true));
    amg1d::Multi& M = h->multi;
    if (!M.norm_valid)
        for (int c = 0; c < M.k; ++c) RET(op_resnorm(h, M.col[(size_t)c], 0, 0));
    RET(read_multi_scalars(h));
    if (res)
        for (int c = 0; c < M.k; ++c) res[c] = M.h_scal[c * MULTI_SLOTS];
    return AMG1D_OK;
}

int amg1d_dev_solve_multi(amg1d_t* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters,
                          double* res) {
    RET(check_multi(h, true));
    if (!res || !iters) return fail(h, AMG1D_ERR_ARG, "null argument");
    if (maxiter < 0) return fail(h, AMG1D_ERR_ARG, "maxiter must be >= 0");
    amg1d::Multi& M = h->multi;
    const int k = M.k;
    for (int c = 0; c < k; ++c) {
        iters[c] = 0;
        Column& col = M.col[(size_t)c];
        RET(op_norm(h, col, col.lv[0].b.p, nullptr, col.lv[0].b.len, 2));
    }
    M.norm_valid = false;
    int act[MULTI_MAX_COLS];
    int na = k;
    for (int c = 0; c < k; ++c) act[c] = c;
    for (int i = 0; i < maxiter && na > 0; ++i) {
        RET(run_vcycle_multi(h, act, na, nPre, nPost, alpha, true, false));
        RET(read_multi_scalars(h));
        int keep = 0;
        for (int j = 0; j < na; ++j) {
            const int c = act[j];
            const double r = M.h_scal[c * MULTI_SLOTS];
            res[(int64_t)c * maxiter + i] = r;
            iters[c] = i + 1;
            if (!(r < tol * M.h_scal[c * MULTI_SLOTS + 2])) act[keep++] = c;   // multigrid()'s stop rule, per column
        }
        na = keep;
    }
    return AMG1D_OK;
}

int amg1d_dev_get_solutions(amg1d_t* h, double* X) {
    RET(check_multi(h, true, false));
    if (!X) return fail(h, AMG1D_ERR_ARG, "null X");
    const int64_t nh = h->L[0].n_host;
    for (int c = 0; c < h->multi.k; ++c) {
        auto& v = h->multi.col[(size_t)c].lv[0];
        RET(to_host(h, 0, v.x[v.cur].p, X + c * nh));
    }
    return AMG1D_OK;
}

int amg1d_synchronize(amg1d_t* h) {
    if (!h) return AMG1D_ERR_ARG;
    CK(cudaStreamSynchronize(h->stream));
    return p2p_check(h);
}

void* amg1d_stream(amg1d_t* h) { return h ? (void*)h->stream : nullptr; }

void* amg1d_dev_ptr(amg1d_t* h, int level, int which) {
    if (!valid_level(h, level) || !h->finalized) return nullptr;
    Column::Vecs& v = h->res.lv[(size_t)level];
    switch (which) {
        case AMG1D_VEC_X: return v.x[v.cur].p;
        case AMG1D_VEC_B: return v.b.p;
        case AMG1D_VEC_R: return h->scratch.p;
        default: return nullptr;
    }
}

int amg1d_vcycle(amg1d_t* h, double* x, const double* b, int nPre, int nPost, double alpha) {
    RET(check_ready(h));
    if (!x || !b) return fail(h, AMG1D_ERR_ARG, "null vector");
    RET(amg1d_dev_set_problem(h, x, b));
    RET(run_vcycle(h, h->res, nPre, nPost, alpha, false));
    return to_host(h, 0, h->res.lv[0].x[h->res.lv[0].cur].p, x);
}

int amg1d_solve(amg1d_t* h, double* x, const double* b, int maxiter, double tol, int nPre,
                int nPost, double alpha, int* iters, double* res, double* err,
                const double* u_exact) {
    RET(check_ready(h));
    if (!x || !b || !res || !iters) return fail(h, AMG1D_ERR_ARG, "null argument");
    if (maxiter < 0) return fail(h, AMG1D_ERR_ARG, "maxiter must be >= 0");
    Column::Vecs& v0 = h->res.lv[0];
    RET(amg1d_dev_set_problem(h, x, b));
    DevBuf exact;
    if (err && u_exact) {
        CK(exact.alloc(v0.x[0].len + 8));
        RET(to_device(h, 0, u_exact, exact.p));
    }
    RET(multigrid_run(h, maxiter, tol, nPre, nPost, alpha, iters, res, err, exact.p));
    return to_host(h, 0, v0.x[v0.cur].p, x);
}

int amg1d_ldiv(amg1d_t* h, double* y, const double* b, int nPre, int nPost, double alpha) {
    RET(check_ready(h));
    if (!y || !b) return fail(h, AMG1D_ERR_ARG, "null vector");
    Level& l0 = h->L[0];
    Column::Vecs& v0 = h->res.lv[0];
    h->norm_valid = false;
    RET(to_device(h, 0, b, v0.b.p));
    if (l0.sharded) RET(op_halo(h, v0.b.p, l0.n, l0.m));
    v0.cur = 0;
    RET(run_vcycle(h, h->res, nPre, nPost, alpha, false, true));      // zero guess: x0 is neither uploaded nor read
    return to_host(h, 0, v0.x[v0.cur].p, y);
}

// multigrid_v_cycle / ldiv! on `count` independent problems, software-pipelined over PCIe: while problem k runs its
// V-cycle on the compute stream, problem k + 1 travels host -> device on a copy-in stream and the iterate of
// problem k - 1 device -> host on a copy-out stream (PCIe is full duplex; with one problem per call the three
// phases are serial and the call is bound by 3 vector transfers).  Level-0 vectors are staged in two device
// buffers per direction; every problem runs exactly the kernels of amg1d_vcycle / amg1d_ldiv: same bits.
int amg1d_vcycle_batch(amg1d_t* h, int count, double* const* x, const double* const* b, int zero_guess, int nPre,
                       int nPost, double alpha) {
    RET(check_ready(h));
    if (count < 0 || (count > 0 && (!x || !b))) return fail(h, AMG1D_ERR_ARG, "bad arguments");
    for (int k = 0; k < count; ++k)
        if (!x[k] || !b[k]) return fail(h, AMG1D_ERR_ARG, "null vector %d", k);
    if (count == 0) return AMG1D_OK;
    Level& l0 = h->L[0];
    Column::Vecs& v0 = h->res.lv[0];
    amg1d::Pipe& P = h->pipe;
    if (!P.s_in) {
        CK(cudaStreamCreateWithFlags(&P.s_in, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&P.s_out, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            CK(cudaEventCreateWithFlags(&P.ev_in[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&P.ev_used[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&P.ev_done[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&P.ev_out[k], cudaEventDisableTiming));
            RET(dev_alloc(h, (void**)&P.st_b[k], l0.n_host * 8));
            RET(dev_alloc(h, (void**)&P.st_x[k], l0.n_host * 8));
            RET(dev_alloc(h, (void**)&P.st_o[k], l0.n_host * 8));
        }
        P.len = l0.n_host;
    }
    h->norm_valid = false;
    const size_t bytes = (size_t)l0.n_host * 8;
    const int64_t ns = l0.n * l0.m;
    const unsigned gp = (unsigned)((ns + 255) / 256);
    // the compute stream may still be busy with earlier work that the copy streams must not overtake
    CK(cudaEventRecord(P.ev_used[0], h->stream));
    CK(cudaStreamWaitEvent(P.s_in, P.ev_used[0], 0));
    for (int k = 0; k < count; ++k) {
        const int sl = k & 1;
        // ---- copy-in stream: stage slot sl is free once problem k - 2 has been moved into the level vectors
        if (k >= 2) {
            CK(cudaStreamWaitEvent(P.s_in, P.ev_used[sl], 0));
            CK(cudaStreamWaitEvent(P.s_in, P.ev_out[sl], 0));    // (a caller may pass problem k - 2's output array again)
        }
        CK(cudaMemcpyAsync(P.st_b[sl], b[k], bytes, cudaMemcpyHostToDevice, P.s_in));
        if (!zero_guess) CK(cudaMemcpyAsync(P.st_x[sl], x[k], bytes, cudaMemcpyHostToDevice, P.s_in));
        CK(cudaEventRecord(P.ev_in[sl], P.s_in));
        // ---- compute stream
        CK(cudaStreamWaitEvent(h->stream, P.ev_in[sl], 0));
        v0.cur = 0;
        if (l0.perm) {
            k_gather_perm<<<gp, 256, 0, h->stream>>>(l0.perm, P.st_b[sl], v0.b.p, ns);
            if (!zero_guess) k_gather_perm<<<gp, 256, 0, h->stream>>>(l0.perm, P.st_x[sl], v0.x[0].p, ns);
            LAUNCH_CHECK();
        } else {
            CK(cudaMemcpyAsync(v0.b.p, P.st_b[sl], bytes, cudaMemcpyDeviceToDevice, h->stream));
            if (!zero_guess) CK(cudaMemcpyAsync(v0.x[0].p, P.st_x[sl], bytes, cudaMemcpyDeviceToDevice, h->stream));
        }
        CK(cudaEventRecord(P.ev_used[sl], h->stream));
        if (l0.sharded) {
            if (zero_guess) RET(op_halo(h, v0.b.p, l0.n, l0.m));
            else RET(op_halo(h, v0.b.p, l0.n, l0.m, v0.x[0].p, l0.n, l0.m));
        }
        RET(run_vcycle(h, h->res, nPre, nPost, alpha, false, zero_guess != 0));
        if (k >= 2) CK(cudaStreamWaitEvent(h->stream, P.ev_out[sl], 0));      // the iterate of problem k - 2 has left
        if (l0.perm) {
            k_scatter_perm<<<gp, 256, 0, h->stream>>>(l0.perm, v0.x[v0.cur].p, P.st_o[sl], ns);
            LAUNCH_CHECK();
        } else {
            CK(cudaMemcpyAsync(P.st_o[sl], v0.x[v0.cur].p, bytes, cudaMemcpyDeviceToDevice, h->stream));
        }
        CK(cudaEventRecord(P.ev_done[sl], h->stream));
        // ---- copy-out stream
        CK(cudaStreamWaitEvent(P.s_out, P.ev_done[sl], 0));
        CK(cudaMemcpyAsync(x[k], P.st_o[sl], bytes, cudaMemcpyDeviceToHost, P.s_out));
        CK(cudaEventRecord(P.ev_out[sl], P.s_out));
    }
    CK(cudaStreamSynchronize(P.s_out));
    CK(cudaStreamSynchronize(h->stream));
    h->dev_problem = true;
    return p2p_check(h);
}

}  // extern "C"

namespace {
// Conjugate gradients preconditioned with one V-cycle (ldiv!(z, H, r)) on the resident problem col; expects the initial
// guess in col.cg.x and the right-hand side in its level-0 rhs buffer, which becomes the residual.  The solution is left
// in col.cg.x.
int pcg_run(amg1d* h, Column& col, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters, double* res) {
    Level& l0 = h->L[0];
    Column::Vecs& v0 = col.lv[0];
    const int64_t N = l0.n * l0.m;
    h->norm_valid = false;
    h->dev_problem = false;                   // level 0's rhs buffer becomes the CG residual
    double* X = col.cg.x.p;
    double* P = col.cg.p.p;
    double* AP = col.cg.ap.p;
    double* R = v0.b.p;                       // the residual lives in the level's rhs buffer: it IS the
                                              // right-hand side of every preconditioner application
    RET(op_norm(h, col, R, nullptr, N, CG_NB));                       // ||b||
    // r = b - A x0
    RET(op_matvec_dot(h, col, 0, X, AP, -1));
    {
        int nb = (int)std::min<int64_t>(AMG1D_RED_BLOCKS, (N + AMG1D_RED_THREADS - 1) / AMG1D_RED_THREADS);
        k_axpy<<<nb, AMG1D_RED_THREADS, 0, h->stream>>>(R, AP, N, -1.0);
        h->launch_counter++;
        LAUNCH_CHECK();
    }
    int it = 0, rc = AMG1D_OK;
    const int nbv = (int)std::max<int64_t>(1, std::min<int64_t>(AMG1D_RED_BLOCKS, (N + AMG1D_RED_THREADS - 1) / AMG1D_RED_THREADS));
    // the initial residual is tested first: b = 0 or an x0 that already solves the system returns x0 with
    // iters = 0 (r.z = p.Ap = 0 would otherwise make the first step 0 / 0)
    RET(op_norm(h, col, R, nullptr, N, CG_RES));
    RET(read_scalars(h, col, 3));
    if (!std::isfinite(h->h_scal[CG_RES]) || !std::isfinite(h->h_scal[CG_NB]))
        return fail(h, AMG1D_ERR_ARG, "amg1d_pcg: non-finite right-hand side or initial guess");
    *iters = 0;
    if (h->h_scal[CG_NB] == 0.0 || h->h_scal[CG_RES] <= tol * h->h_scal[CG_NB]) return AMG1D_OK;
    for (int i = 0; i < maxiter; ++i) {
        // z = M^-1 r: one V-cycle from a zero guess with rhs r (already in place); z = level-0 iterate
        if (l0.sharded) { rc = op_halo(h, R, l0.n, l0.m); if (rc) break; }
        v0.cur = 0;
        rc = run_vcycle(h, col, nPre, nPost, alpha, false, true);
        if (rc) break;
        double* Z = v0.x[v0.cur].p;
        rc = op_dot(h, col, R, Z, N, i == 0 ? CG_RZ : CG_RZ_NEW);
        if (rc) break;
        if (i > 0) { k_cg_beta<<<1, 1, 0, h->stream>>>(col.scal); h->launch_counter++; }
        k_cg_direction<<<nbv, AMG1D_RED_THREADS, 0, h->stream>>>(P, Z, N, col.scal, i == 0 ? 1 : 0);
        h->launch_counter++;
        rc = op_matvec_dot(h, col, 0, P, AP, CG_PAP);
        if (rc) break;
        k_cg_alpha<<<1, 1, 0, h->stream>>>(col.scal);
        k_cg_update<<<nbv, AMG1D_RED_THREADS, 0, h->stream>>>(X, R, P, AP, N, col.scal, col.partial);
        h->launch_counter += 2;
        { cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) { rc = fail(h, AMG1D_ERR_CUDA, "pcg kernels: %s", cudaGetErrorString(e_)); break; } }
        rc = op_reduce_partials(h, col, nbv, CG_RES, true);       // ||r||_2
        if (rc) break;
        rc = read_scalars(h, col, 3);
        if (rc) break;
        res[i] = h->h_scal[CG_RES];
        it = i + 1;
        if (!(res[i] >= tol * h->h_scal[CG_NB])) break;          // also stops on NaN
    }
    RET(rc);
    *iters = it;
    if (it > 0 && !std::isfinite(res[it - 1]))                   // never AMG1D_OK with NaNs in the caller's x
        return fail(h, AMG1D_ERR_ARG, "amg1d_pcg: breakdown at iteration %d (non-finite residual: the operator "
                    "or the V-cycle preconditioner is not symmetric positive definite)", it);
    return AMG1D_OK;
}

// ---- pcg_run on every column of the multi-column set (amg1d_dev_pcg_multi) --------------------------------------
// The vectors, reduction scratch and scalar windows of the active columns act[0..na), entry i for column act[i].
struct CgMultiVecs {
    ColVecs X, R, P, AP, Z, part, scal;
    CgMultiVecs(amg1d* h, const int* act, int na) : X(), R(), P(), AP(), Z(), part(), scal() {
        amg1d::Multi& M = h->multi;
        for (int i = 0; i < na; ++i) {
            Column& col = M.col[(size_t)act[i]];
            auto& v = col.lv[0];
            X.v[i] = col.cg.x.p;
            P.v[i] = col.cg.p.p;
            AP.v[i] = col.cg.ap.p;
            R.v[i] = v.b.p;                      // the residual lives in the column's level-0 rhs buffer, as in pcg_run
            Z.v[i] = v.x[v.cur].p;               // the preconditioned residual: the column's level-0 iterate
            part.v[i] = col.partial;
            scal.v[i] = col.scal;
        }
    }
};

// op_reduce_partials of every active column in one launch per stage
int reduce_partials_multi(amg1d* h, const CgMultiVecs& v, int na, int64_t np, int slot, int take_sqrt) {
    ColVecs src = v.part;
    if (np > 8192) {
        ColVecs st2 = {};
        for (int i = 0; i < na; ++i) st2.v[i] = v.part.v[i] + h->partial_cap;
        k_sum_partial_multi<<<dim3(256, na), AMG1D_RED_THREADS, 0, h->stream>>>(v.part, np, st2);
        h->launch_counter++;
        src = st2;
        np = 256;
    }
    k_reduce_final_multi<<<dim3(1, na), AMG1D_RED_THREADS, 0, h->stream>>>(src, (int)np, v.scal, slot, take_sqrt);
    h->launch_counter++;
    LAUNCH_CHECK();
    return AMG1D_OK;
}

// op_matvec_dot(h, col, 0, x_c, y_c, slot) for every active column: one launch that reads level 0's operator once where
// op_matvec_dot would take the fused kernel (the same predicate, hence the same partial sums), its own code per
// column elsewhere
int matvec_dot_multi(amg1d* h, const int* act, int na, const CgMultiVecs& v, const ColVecs& x, const ColVecs& y,
                     int slot) {
    Level& l0 = h->L[0];
    MatvecCols mc = {};
    for (int i = 0; i < na; ++i) {
        mc.x[i] = x.v[i];
        mc.y[i] = y.v[i];
        mc.partial[i] = slot >= 0 ? v.part.v[i] : nullptr;
    }
    int nb = 0;
    if (h->opt_fused && fused_matvec_dot_multi(l0.md, l0.mat, mc, na, l0.n, h->partial_cap, &nb, h->stream)) {
        h->launch_counter++;
        LAUNCH_CHECK();
        return slot >= 0 ? reduce_partials_multi(h, v, na, nb, slot, 0) : AMG1D_OK;
    }
    for (int i = 0; i < na; ++i) RET(op_matvec_dot(h, h->multi.col[(size_t)act[i]], 0, x.v[i], y.v[i], slot));
    return AMG1D_OK;
}

// pcg_run step for step on every column of the set, the columns that are still iterating batched into each launch.
// The initial guess is the column's resident iterate, the solution becomes it; the right-hand side becomes the residual.
int pcg_multi_run(amg1d* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters, double* res) {
    Level& l0 = h->L[0];
    amg1d::Multi& M = h->multi;
    const int k = M.k;
    const int64_t N = l0.n * l0.m;
    const size_t bytes = (size_t)M.col[0].lv[0].x[0].len * 8;
    for (int c = 0; c < k; ++c) {
        const int rc = column_alloc(h, M.col[(size_t)c], true);
        if (rc != AMG1D_OK) return fail(h, rc, "CG vectors of column %d of the multi-column set: %s", c, h->err.c_str());
    }
    int act[MULTI_MAX_COLS];
    int na = k;
    for (int c = 0; c < k; ++c) {
        act[c] = c;
        iters[c] = 0;
        auto& v = M.col[(size_t)c].lv[0];
        CK(cudaMemcpyAsync(M.col[(size_t)c].cg.x.p, v.x[v.cur].p, bytes, cudaMemcpyDeviceToDevice, h->stream));
    }
    M.norm_valid = false;
    M.rhs_consumed = true;
    const int nbv = (int)std::max<int64_t>(1, std::min<int64_t>(AMG1D_RED_BLOCKS, (N + AMG1D_RED_THREADS - 1) / AMG1D_RED_THREADS));
    const dim3 gv(nbv, na), gs(1, na);
    {
        const CgMultiVecs v(h, act, na);
        k_sqdiff_partial_multi<<<gv, AMG1D_RED_THREADS, 0, h->stream>>>(v.R, N, v.part);           // ||b||
        k_reduce_final_multi<<<gs, AMG1D_RED_THREADS, 0, h->stream>>>(v.part, nbv, v.scal, CG_NB, 1);
        h->launch_counter += 2;
        LAUNCH_CHECK();
        RET(matvec_dot_multi(h, act, na, v, v.X, v.AP, -1));                                       // r = b - A x0
        k_axpy_multi<<<gv, AMG1D_RED_THREADS, 0, h->stream>>>(v.R, v.AP, N, -1.0);
        k_sqdiff_partial_multi<<<gv, AMG1D_RED_THREADS, 0, h->stream>>>(v.R, N, v.part);
        k_reduce_final_multi<<<gs, AMG1D_RED_THREADS, 0, h->stream>>>(v.part, nbv, v.scal, CG_RES, 1);
        h->launch_counter += 3;
        LAUNCH_CHECK();
    }
    RET(read_multi_scalars(h));
    na = 0;
    for (int c = 0; c < k; ++c) {
        const double* s = M.h_scal + c * MULTI_SLOTS;
        if (!std::isfinite(s[CG_RES]) || !std::isfinite(s[CG_NB]))
            return fail(h, AMG1D_ERR_ARG, "amg1d_dev_pcg_multi: non-finite right-hand side or initial guess in column %d", c);
        if (!(s[CG_NB] == 0.0 || s[CG_RES] <= tol * s[CG_NB])) act[na++] = c;   // pcg_run's initial-residual test
    }
    for (int i = 0; i < maxiter && na > 0; ++i) {
        // z = M^-1 r: one multi-column V-cycle from a zero guess with right-hand sides r (already in place)
        RET(run_vcycle_multi(h, act, na, nPre, nPost, alpha, false, true));
        const int64_t c0 = h->launch_counter;
        const CgMultiVecs v(h, act, na);
        const dim3 g(nbv, na);
        k_dot_partial_multi<<<g, AMG1D_RED_THREADS, 0, h->stream>>>(v.R, v.Z, N, v.part);
        h->launch_counter++;
        LAUNCH_CHECK();
        RET(reduce_partials_multi(h, v, na, nbv, i == 0 ? CG_RZ : CG_RZ_NEW, 0));
        if (i > 0) { k_cg_beta_multi<<<1, na, 0, h->stream>>>(v.scal); h->launch_counter++; }
        k_cg_direction_multi<<<g, AMG1D_RED_THREADS, 0, h->stream>>>(v.P, v.Z, N, v.scal, i == 0 ? 1 : 0);
        h->launch_counter++;
        LAUNCH_CHECK();
        RET(matvec_dot_multi(h, act, na, v, v.P, v.AP, CG_PAP));
        k_cg_alpha_multi<<<1, na, 0, h->stream>>>(v.scal);
        k_cg_update_multi<<<g, AMG1D_RED_THREADS, 0, h->stream>>>(v.X, v.R, v.P, v.AP, N, v.scal, v.part);
        h->launch_counter += 2;
        LAUNCH_CHECK();
        RET(reduce_partials_multi(h, v, na, nbv, CG_RES, 1));                                  // ||r||_2
        M.pcg_launches = h->launch_counter - c0;
        RET(read_multi_scalars(h));
        int keep = 0;
        for (int j = 0; j < na; ++j) {
            const int c = act[j];
            const double r = M.h_scal[c * MULTI_SLOTS + CG_RES];
            res[(int64_t)c * maxiter + i] = r;
            iters[c] = i + 1;
            if (r >= tol * M.h_scal[c * MULTI_SLOTS + CG_NB]) act[keep++] = c;                   // also stops on NaN
        }
        na = keep;
    }
    for (int c = 0; c < k; ++c) {                                  // the solutions become the resident iterates
        auto& v = M.col[(size_t)c].lv[0];
        v.cur = 0;
        CK(cudaMemcpyAsync(v.x[0].p, M.col[(size_t)c].cg.x.p, bytes, cudaMemcpyDeviceToDevice, h->stream));
    }
    for (int c = 0; c < k; ++c)
        if (iters[c] > 0 && !std::isfinite(res[(int64_t)c * maxiter + iters[c] - 1]))
            return fail(h, AMG1D_ERR_ARG, "amg1d_dev_pcg_multi: breakdown in column %d at iteration %d (non-finite "
                        "residual: the operator or the V-cycle preconditioner is not symmetric positive definite)",
                        c, iters[c]);
    return AMG1D_OK;
}
}  // namespace

extern "C" {

int amg1d_pcg(amg1d_t* h, double* x, const double* b, int maxiter, double tol, int nPre, int nPost,
              double alpha, int* iters, double* res) {
    RET(check_ready(h));
    if (!x || !b || !res || !iters) return fail(h, AMG1D_ERR_ARG, "null argument");
    if (maxiter < 0) return fail(h, AMG1D_ERR_ARG, "maxiter must be >= 0");
    RET(column_alloc(h, h->res, true));
    RET(to_device(h, 0, b, h->res.lv[0].b.p));
    RET(to_device(h, 0, x, h->res.cg.x.p));
    RET(pcg_run(h, h->res, maxiter, tol, nPre, nPost, alpha, iters, res));
    return to_host(h, 0, h->res.cg.x.p, x);
}

int amg1d_dev_pcg(amg1d_t* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters, double* res) {
    RET(check_dev_problem(h));
    if (!res || !iters) return fail(h, AMG1D_ERR_ARG, "null argument");
    if (maxiter < 0) return fail(h, AMG1D_ERR_ARG, "maxiter must be >= 0");
    Column::Vecs& v0 = h->res.lv[0];
    RET(column_alloc(h, h->res, true));
    CK(cudaMemcpyAsync(h->res.cg.x.p, v0.x[v0.cur].p, (size_t)v0.x[0].len * 8, cudaMemcpyDeviceToDevice, h->stream));
    RET(pcg_run(h, h->res, maxiter, tol, nPre, nPost, alpha, iters, res));
    v0.cur = 0;                                                  // the solution becomes the resident iterate
    CK(cudaMemcpyAsync(v0.x[0].p, h->res.cg.x.p, (size_t)v0.x[0].len * 8, cudaMemcpyDeviceToDevice, h->stream));
    return AMG1D_OK;
}

int amg1d_dev_pcg_multi(amg1d_t* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters,
                        double* res) {
    RET(check_multi(h, true));
    if (!res || !iters) return fail(h, AMG1D_ERR_ARG, "null argument");
    if (maxiter < 0) return fail(h, AMG1D_ERR_ARG, "maxiter must be >= 0");
    return pcg_multi_run(h, maxiter, tol, nPre, nPost, alpha, iters, res);
}

int amg1d_apply_smoother(amg1d_t* h, int level, double* Y, const double* B, int64_t n_rhs,
                         double alpha) {
    RET(check_ready(h));
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "per-level host operations are single-GPU only");
    if (!valid_level(h, level)) return fail(h, AMG1D_ERR_ARG, "level %d out of range", level);
    if (!Y || !B || n_rhs < 1) return fail(h, AMG1D_ERR_ARG, "bad arguments");
    Level& lv = h->L[level];
    Column::Vecs& v = h->res.lv[(size_t)level];
    double* in = v.x[1 - v.cur].p;  // free ping-pong buffer as input staging
    for (int64_t c = 0; c < n_rhs; ++c) {
        RET(to_device(h, level, B + c * lv.n_host, in));
        if (lv.smooth_tri)
            g_apply_tri_smoother<<<ggrid(lv.n, lv.m), gblock(lv.m), 0, h->stream>>>(
                lv.smat, lv.smd, in, nullptr, h->scratch.p, lv.n, alpha);
        else
        g_apply_smoother<<<ggrid(lv.n, lv.m), gblock(lv.m), 0, h->stream>>>(
            lv.mat, lv.md, in, h->scratch.p, lv.n, alpha);
        LAUNCH_CHECK();
        RET(to_host(h, level, h->scratch.p, Y + c * lv.n_host));
    }
    return AMG1D_OK;
}

int amg1d_smoother_solve(amg1d_t* h, int level, double* x, const double* b, int maxiter, double tol,
                         double alpha, int* iters, double* res, double* err, const double* u_exact) {
    RET(check_ready(h));
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "per-level host operations are single-GPU only");
    if (!valid_level(h, level)) return fail(h, AMG1D_ERR_ARG, "level %d out of range", level);
    if (!x || !b || !res || !iters) return fail(h, AMG1D_ERR_ARG, "null argument");
    Level& lv = h->L[level];
    Column& col = h->res;
    Column::Vecs& v = col.lv[(size_t)level];
    invalidate_graph(h);
    if (level == 0) h->dev_problem = false;    // stages b and x in level 0's own vectors
    v.cur = 0;
    RET(to_device(h, level, b, v.b.p));
    RET(to_device(h, level, x, v.x[0].p));
    DevBuf exact;
    double* d_exact = nullptr;
    if (err && u_exact) {
        CK(exact.alloc(v.x[0].len + 8));
        d_exact = exact.p;
        RET(to_device(h, level, u_exact, d_exact));
    }
    int rc = op_norm(h, col, v.b.p, nullptr, v.b.len, 2);
    int it = 0;
    for (int i = 0; i < maxiter && rc == AMG1D_OK; ++i) {
        rc = op_sweep(h, level, v.b.p, v.x[v.cur].p, v.x[1 - v.cur].p, alpha, 0);
        if (rc != AMG1D_OK) break;
        v.cur = 1 - v.cur;
        rc = op_resnorm(h, col, level, 0);
        if (rc != AMG1D_OK) break;
        if (d_exact) {
            rc = op_norm(h, col, v.x[v.cur].p, d_exact, v.x[0].len, 1);
            if (rc != AMG1D_OK) break;
        }
        rc = read_scalars(h, col, 3);
        if (rc != AMG1D_OK) break;
        res[i] = h->h_scal[0];
        if (err) err[i] = d_exact ? h->h_scal[1] : NAN;
        it = i + 1;
        if (res[i] < tol * h->h_scal[2]) break;
    }
    RET(rc);
    *iters = it;
    rc = to_host(h, level, v.x[v.cur].p, x);
    if (v.cur != 0) {
        CK(cudaMemcpyAsync(v.x[0].p, v.x[1].p, (size_t)v.x[0].len * 8, cudaMemcpyDeviceToDevice, h->stream));
        v.cur = 0;
    }
    return rc;
}

static int apply_common(amg1d_t* h, int level, double* out, const double* x, const double* b, int mode) {
    RET(check_ready(h));
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "per-level host operations are single-GPU only");
    if (!valid_level(h, level)) return fail(h, AMG1D_ERR_ARG, "level %d out of range", level);
    if (!out || !x || (mode && !b)) return fail(h, AMG1D_ERR_ARG, "null vector");
    Column::Vecs& v = h->res.lv[(size_t)level];
    invalidate_graph(h);
    double* xin = v.x[1 - v.cur].p;
    RET(to_device(h, level, x, xin));
    double* bin = v.b.p;  // clobbers the level rhs: amg1d_vcycle / amg1d_solve re-upload it, the device-resident
    if (mode) {            // problem (level 0) is marked stale so that amg1d_dev_vcycle refuses to use it
        if (level == 0) h->dev_problem = false;
        RET(to_device(h, level, b, bin));
    }
    RET(op_apply(h, level, bin, xin, h->scratch.p, mode));
    return to_host(h, level, h->scratch.p, out);
}

int amg1d_matvec(amg1d_t* h, int level, double* y, const double* x) {
    return apply_common(h, level, y, x, nullptr, 0);
}

int amg1d_residual(amg1d_t* h, int level, double* r, const double* x, const double* b) {
    return apply_common(h, level, r, x, b, 1);
}

int amg1d_restrict(amg1d_t* h, int level, double* rc, const double* rf) {
    RET(check_ready(h));
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "per-level host operations are single-GPU only");
    if (level < 0 || level >= h->n_levels - 1) return fail(h, AMG1D_ERR_ARG, "transfer %d out of range", level);
    if (!rc || !rf) return fail(h, AMG1D_ERR_ARG, "null vector");
    invalidate_graph(h);
    Column::Vecs& vf = h->res.lv[(size_t)level];
    Column::Vecs& vc = h->res.lv[(size_t)level + 1];
    double* fin = vf.x[1 - vf.cur].p;
    RET(to_device(h, level, rf, fin));
    RET(op_restrict(h, level, fin, vc.b.p));
    return to_host(h, level + 1, vc.b.p, rc);
}

int amg1d_prolong(amg1d_t* h, int level, double* xf, const double* xc) {
    RET(check_ready(h));
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "per-level host operations are single-GPU only");
    if (level < 0 || level >= h->n_levels - 1) return fail(h, AMG1D_ERR_ARG, "transfer %d out of range", level);
    if (!xf || !xc) return fail(h, AMG1D_ERR_ARG, "null vector");
    invalidate_graph(h);
    Column::Vecs& vc = h->res.lv[(size_t)level + 1];
    double* cin = vc.x[1 - vc.cur].p;
    RET(to_device(h, level + 1, xc, cin));
    RET(op_prolong(h, level, cin, h->scratch.p, 0));
    return to_host(h, level, h->scratch.p, xf);
}

int amg1d_coarse_solve(amg1d_t* h, double* x, const double* b) {
    RET(check_ready(h));
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "per-level host operations are single-GPU only");
    if (!x || !b) return fail(h, AMG1D_ERR_ARG, "null vector");
    invalidate_graph(h);
    const int l = h->n_levels - 1;
    Column::Vecs& v = h->res.lv[(size_t)l];
    double* bin = v.x[1 - v.cur].p;
    RET(to_device(h, l, b, bin));
    RET(op_coarse(h, bin, h->scratch.p));
    return to_host(h, l, h->scratch.p, x);
}

int amg1d_direct_solve(amg1d_t* h, int level, double* x, const double* b) {
    RET(check_ready(h));
    if (h->nranks > 1) return fail(h, AMG1D_ERR_UNSUPPORTED, "per-level host operations are single-GPU only");
    if (!valid_level(h, level)) return fail(h, AMG1D_ERR_ARG, "level %d out of range", level);
    if (!x || !b) return fail(h, AMG1D_ERR_ARG, "null vector");
    if (h->direct.size() < (size_t)h->n_levels) h->direct.resize((size_t)h->n_levels);
    BcrSolver& S = h->direct[(size_t)level];
    if (!S.ready()) RET(bcr_factor(h, S, level));
    invalidate_graph(h);
    Column::Vecs& v = h->res.lv[(size_t)level];
    double* bin = v.x[1 - v.cur].p;              // free ping-pong buffer as input staging
    RET(to_device(h, level, b, bin));
    CK(S.solve(bin, h->scratch.p, h->stream, &h->launch_counter));
    return to_host(h, level, h->scratch.p, x);
}

int amg1d_set_option(amg1d_t* h, const char* key, int64_t value) {
    if (!h || !key) return AMG1D_ERR_ARG;
    invalidate_graph(h);
    if (!strcmp(key, "fused")) h->opt_fused = (int)value;
    else if (!strcmp(key, "graph")) h->opt_graph = (int)value;
    else if (!strcmp(key, "pdl")) h->opt_pdl = (int)value;
    else if (!strcmp(key, "rows_window")) {
        if (value != 0 && !rows_window_ok((int)value)) return fail(h, AMG1D_ERR_ARG, "rows_window must be 0, 32 or 64");
        h->opt_rows = (int)value;
    }
    else if (!strcmp(key, "pattern_resident")) {
        if (value < 0 || value > 2) return fail(h, AMG1D_ERR_ARG, "pattern_resident must be 0, 1 or 2");
        h->opt_pattern = (int)value;
    }
    else if (!strcmp(key, "p2p_halo")) {
        if (h->finalized) return fail(h, AMG1D_ERR_STATE, "'p2p_halo' must be set before amg1d_finalize");
        h->opt_p2p = value != 0;
    }
    else if (!strcmp(key, "dinv_registers")) h->opt_dvreg = (int)value;
    else if (!strcmp(key, "leg_pipeline_min")) {
        if (value < 0) return fail(h, AMG1D_ERR_ARG, "leg_pipeline_min must be >= 0");
        h->opt_pipe_min = value;
    }
    else if (!strcmp(key, "recompute_dinv_max")) {
        if (value < 1 || value > 5) return fail(h, AMG1D_ERR_ARG, "recompute_dinv_max must be in [1, 5]");
        h->opt_dvrec_max = (int)value;
    }
    else if (!strcmp(key, "leg_pipeline")) {
        if (value < 0 || value > 2) return fail(h, AMG1D_ERR_ARG, "leg_pipeline must be 0, 1 or 2");
        h->opt_pipe = (int)value;
    }
    else if (!strcmp(key, "recompute_dinv")) {
        // before the first level: whether uploaded inverses are replaced by the device's own (adopt_device_dinv);
        // afterwards: whether the fused legs recompute them or stream the stored ones (same bits either way)
        if (value < 0) return fail(h, AMG1D_ERR_ARG, "recompute_dinv must be >= 0");
        h->opt_dvrec = (int)value;
    }
    else if (!strcmp(key, "rows_per_thread")) {
        if (value != 0 && !rows_rpt_ok((int)value)) return fail(h, AMG1D_ERR_ARG, "rows_per_thread must be 0 (auto), 1, 2 or 3");
        h->opt_rows_rpt = (int)value;
    }
    else if (!strcmp(key, "coarse_cta_elems")) {
        h->opt_coarse_cta = value;
        if (h->finalized) { CK(cudaSetDevice(h->device)); CK(cudaStreamSynchronize(h->stream)); RET(build_tail(h)); }
    }
    else if (!strcmp(key, "ghost_depth") || !strcmp(key, "shard_min") || !strcmp(key, "compress")) {
        for (auto& lv : h->L)
            if (lv.set) return fail(h, AMG1D_ERR_STATE, "'%s' must be set before the first level", key);
        if (!strcmp(key, "compress")) { h->opt_compress = value != 0; return AMG1D_OK; }
        if (value < 1) return fail(h, AMG1D_ERR_ARG, "'%s' must be >= 1", key);
        if (!strcmp(key, "ghost_depth")) {
            if ((value + 2) * 8 > PAD_FRONT) return fail(h, AMG1D_ERR_ARG, "ghost_depth must be <= %d", PAD_FRONT / 8 - 2);
            h->ghost_depth = (int)value;
        } else h->shard_min = value;
    }
    else if (!strcmp(key, "profile")) {
        h->opt_profile = (int)value;
        for (auto& pr : h->prof) { for (auto ev : pr.ev) cudaEventDestroy(ev); pr.ev.clear(); }
    }
    else return fail(h, AMG1D_ERR_ARG, "unknown option '%s'", key);
    return AMG1D_OK;
}

int64_t amg1d_get_info(amg1d_t* h, const char* key) {
    if (!h || !key) return -1;
    if (!strcmp(key, "kernel_launches")) return h->launch_counter;
    if (!strcmp(key, "launches_per_cycle")) return h->launches_per_cycle;
    if (!strcmp(key, "device_bytes")) return h->device_bytes;
    if (!strcmp(key, "n_levels")) return h->n_levels;
    if (!strcmp(key, "local_elements")) return h->L[0].n;
    if (!strcmp(key, "local_dofs")) return h->L[0].n * h->L[0].m;
    if (!strcmp(key, "local_offset_dofs")) return h->L[0].start * h->L[0].m;
    if (!strcmp(key, "gather_level")) return h->gather_level;
    if (!strcmp(key, "tail_start")) return h->tail_start;
    if (!strcmp(key, "ghost_depth")) return h->ghost_depth;
    if (!strcmp(key, "rows_window")) return h->opt_rows;
    if (!strcmp(key, "rows_per_thread")) return h->opt_rows_rpt;
    if (!strcmp(key, "pattern_resident")) return h->opt_pattern;
    if (!strncmp(key, "pattern:", 8)) {                      // 1: level has a pattern table
        const int l = atoi(key + 8);
        return valid_level(h, l) && h->L[l].pat ? 1 : 0;
    }
    if (!strcmp(key, "recompute_dinv")) return h->opt_dvrec;
    if (!strcmp(key, "dinv_registers")) return h->opt_dvreg;
    if (!strcmp(key, "leg_pipeline")) return h->opt_pipe;
    if (!strcmp(key, "leg_pipeline_min")) return h->opt_pipe_min;
    if (!strncmp(key, "leg_pipeline:", 13)) {       // 1: the fused legs of this level are the pipelined persistent kernels
        const int l = atoi(key + 13);
        if (!valid_level(h, l) || !h->L[l].set || l + 1 >= h->n_levels || !h->T[l].fusable) return 0;
        if (h->opt_pattern && h->L[l].pat) return 0;
        const int rec = leg_rec(h, h->L[l], h->T[l].mc);
        return ((rec & 16) && (rec & 3) && fused_has_pp(h->L[l].m, h->T[l].mc, h->L[l].md.st, h->L[l].diag)) ? 1 : 0;
    }
    if (!strcmp(key, "p2p_halo")) return h->p2p.on ? 1 : 0;     // 1: slab edges travel through peer memory, 0: NCCL
    if (!strcmp(key, "halo_bytes_per_cycle")) {                  // algorithmic bytes this rank SENDS to its slab neighbours
        int64_t bytes = 0;                                       // per V-cycle: per sharded level the pre-smoothed edges, the
        const int sides = (h->rank > 0) + (h->rank < h->nranks - 1);   // coarse rhs edges and the corrected edges
        for (int l = 0; l < h->n_levels; ++l) {
            if (!h->L[l].sharded) continue;
            bytes += 2LL * h->ghost_depth * h->L[l].m * 8 * sides;
            if (l + 1 < h->n_levels && h->L[l + 1].sharded) bytes += (int64_t)h->ghost_depth * h->L[l + 1].m * 8 * sides;
        }
        return bytes;
    }
    if (!strcmp(key, "sharded_levels")) {
        int c = 0;
        for (const auto& lv : h->L) c += lv.sharded ? 1 : 0;
        return c;
    }
    if (!strncmp(key, "dinv_pivots:", 12)) {        // 1: some element of the level swaps rows in its inverse
        const int l = atoi(key + 12);
        return valid_level(h, l) && h->L[l].set ? (h->L[l].dv_rec == 1) : -1;
    }
    if (!strncmp(key, "dinv_recompute:", 15)) {     // 1: the fused legs of this level invert A_di in registers
        const int l = atoi(key + 15);               //    instead of streaming the stored inverse
        if (!valid_level(h, l) || !h->L[l].set || l + 1 >= h->n_levels || !(leg_rec(h, h->L[l], h->T[l].mc) & 3)) return 0;
        if (h->opt_pattern && h->L[l].pat) return 0;
        return (h->L[l].m <= 5 && h->T[l].fusable) ? 1 : 0;
    }
    if (!strncmp(key, "structure:", 10)) {          // "structure:<level>" -> structure class (layout.cuh)
        const int l = atoi(key + 10);
        return valid_level(h, l) && h->L[l].set ? h->L[l].md.st : -1;
    }
    if (!strncmp(key, "tile_rows:", 10)) {          // "tile_rows:<level>" -> doubles stored per element
        const int l = atoi(key + 10);
        return valid_level(h, l) && h->L[l].set ? h->L[l].md.K : -1;
    }
    if (!strcmp(key, "rank")) return h->rank;
    if (!strcmp(key, "nranks")) return h->nranks;
    if (!strcmp(key, "dof_updates_per_sweep")) {
        int64_t s = 0;
        for (int l = 0; l < h->n_levels - 1; ++l) s += h->L[l].n_glob * h->L[l].m;
        return s;
    }
    if (!strcmp(key, "multi_columns")) return h->multi.k;
    if (!strcmp(key, "multi_launches_per_cycle")) return h->multi.launches_per_cycle;
    if (!strcmp(key, "multi_pcg_launches_per_iteration")) return h->multi.pcg_launches;
    if (!strncmp(key, "multi_legs:", 11)) {         // 1: the multi-column cycle reads this level's operator once for all
        const int l = atoi(key + 11);               //    columns (fused multi-column legs), 0: once per column
        if (!valid_level(h, l) || !h->finalized || h->nranks > 1 || l + 1 >= h->n_levels) return 0;
        if (h->tail_start > 0 && l >= h->tail_start) return 0;
        return multi_leg_level(h, l) ? 1 : 0;
    }
    return -1;
}

int amg1d_get_profile(amg1d_t* h, int level, int leg, double* total_ms, int* launches) {
    if (!h || !total_ms || !launches) return AMG1D_ERR_ARG;
    if (!valid_level(h, level) || leg < 0 || leg > 1) return fail(h, AMG1D_ERR_ARG, "bad level / leg");
    *total_ms = 0.0;
    *launches = 0;
    if (h->prof.size() <= (size_t)(level * 2 + leg)) return AMG1D_OK;
    CK(cudaStreamSynchronize(h->stream));
    auto& ev = h->prof[level * 2 + leg].ev;
    for (size_t i = 0; i + 1 < ev.size(); i += 2) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
        *total_ms += ms;
        *launches += 1;
    }
    return AMG1D_OK;
}

int amg1d_host_alloc(void** p, int64_t bytes) {
    amg1d* h = nullptr;
    if (!p || bytes < 0) return fail(h, AMG1D_ERR_ARG, "bad arguments");
    CK(cudaMallocHost(p, (size_t)std::max<int64_t>(bytes, 8)));
    return AMG1D_OK;
}

int amg1d_host_free(void* p) {
    amg1d* h = nullptr;
    if (p) CK(cudaFreeHost(p));
    return AMG1D_OK;
}

}  // extern "C"
