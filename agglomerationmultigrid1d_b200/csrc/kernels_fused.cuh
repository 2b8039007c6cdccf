// Fast kernel tier: templated on the block size M and the level's structure class ST (layout.cuh),
// one thread per element, operator read straight from the element-tile layout with fully coalesced
// 256-byte warp requests.
//
//  f_sweep / f_resnorm / f_residual_restrict  - streaming kernels (one pass over the operator each)
//  f_down   nPre sweeps + residual + restriction  in ONE pass over the level's operator
//  f_up     prolongation + correction + nPost sweeps (+ optional ||b - A x||^2)  in ONE pass
//  f_tail   the whole sub-V-cycle of the coarse levels (<= 512 elements) in ONE CTA, out of shared memory
//
// f_down / f_up keep the element's operator blocks in registers for the whole leg (Dinv in shared
// memory, staged with cp.async) and exchange only the M iterate values with the two neighbour
// threads through shared memory between sweeps (Jacobi needs the *old* neighbour values, so the
// exchange is double buffered).  A CTA owns a window of B consecutive elements; after s sweeps only
// the inner [s, B - s) elements are still exact, so the CTA emits the inner B - 2 halo elements and
// adjacent CTAs overlap by the halo (the overlap is re-read through L2, not HBM).  Per element the
// arithmetic and its order are identical to the generic tier, so both tiers agree bit for bit on x.
//
// Both smoother kinds (block Jacobi: Dinv = m x m; point Jacobi: Dinv = m) and both transfer kinds
// (single parent: dg_dg / aggdg_dg / aggdg_aggdg; two parents: cg_cg / dg_cg / aggdg_cg) are covered,
// the latter with the closed-form parent map  parent(e) = (e + shift) / ratio + base.
//
// Algorithmic bytes per element (FP64; Kop = doubles of the level's structure class, layout.cuh;
// coarse block size MC, ratio R children):
//   f_sweep               8 (Kop + 3 M)                           [zero guess: 8 (|Dinv| + 2 M)]
//   f_down (S sweeps)     8 (Kop + 3 M + MC / R)  (+ P block if it is per-element)
//   f_up   (S sweeps)     8 (Kop + 3 M + MC / R)  (+ P block if it is per-element)
// against S * 8 (4 M^2 + 3 M) + 8 (3 M^2 + 2 M + ...) for the unfused dense sequence (SURVEY 8d B_ref).
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <type_traits>
#include <cstdint>
#include "kernels_generic.cuh"
#include "layout.cuh"
#include "halo_p2p.cuh"

// Position of a rank's slab inside its level (single GPU: gl = gr = e_off = c_off = 0).  Local element
// index e runs over [-gl, n + gr): gl / gr ghost elements (with operator blocks, rhs and iterate) on the
// left / right slab edge; e_off = global index of local element 0; c_off = global index of local coarse
// element 0; nc = coarse elements this rank owns.
struct Slab {
    int gl, gr;
    int64_t e_off, c_off, nc;
};

// Translation-invariant level (uniform mesh, amg1d_set_level_pattern) in "pattern-resident" form: the
// n_head + 1 + n_tail distinct block sets of the level as a small table tab[set][k] (k = tile row of
// layout.cuh), instead of one stored block set per element.  The fused legs then fetch an element's
// operator from the table (a few KB, served by L1 as a warp-wide broadcast) and HBM carries only the
// vectors.  tab == nullptr: the element tiles are streamed (the general per-element layout).
struct PatOp {
    const double* tab;
    int64_t n_glob;        // elements of the whole level (the table is indexed by GLOBAL element)
    int n_head, n_tail;
    const double* host_interior;   // HOST copy of the interior row tab[n_head][*] (pattern_resident = 2: the
                                   // launcher passes it by value as ParamOp), else nullptr; unused on the device
};

// Per-launch constants of a fused leg, computed on the host so that the per-thread index arithmetic
// (parent element, owner test, transfer-block index) is 32-bit: with out % ratio == 0 the CTA's first
// thread has (e_global + shift) = ratio * (blockIdx * opr + qdiv0) + qmod0.
struct WinIdx {
    int halo, out;     // recomputed window elements per side; elements emitted per CTA
    int opr;           // out / ratio
    int qmod0;         // floormod(e_off + shift - halo, ratio)
    int64_t qdiv0;     // floordiv(e_off + shift - halo, ratio)
    int pmod0;         // floormod(e_off - halo - n_head, period) + pbias, or -1: use TransferMap::blk (64-bit)
};

__device__ __forceinline__ void small_divmod(int x, int d, int* q, int* r) {   // x >= 0, d >= 1
    if (d == 1) { *q = x; *r = 0; }
    else if (d == 2) { *q = x >> 1; *r = x & 1; }
    else { *q = x / d; *r = x - *q * d; }
}

// transfer-block index of global fine element c = (window thread tc of this CTA), see TransferMap::blk
__device__ __forceinline__ int64_t win_blk(const TransferMap& tm, const WinIdx& w, int64_t c, int tc) {
    if (tm.period == 0 || w.pmod0 < 0) return tm.blk(c);
    if (c < tm.n_head) return c;
    if (c >= tm.n_fine - tm.n_tail) return tm.n_head + tm.period + (c - (tm.n_fine - tm.n_tail));
    int q, r;
    small_divmod(w.pmod0 + tc, tm.period, &q, &r);
    return tm.n_head + r;
}

// Programmatic dependent launch (PDL): every fused kernel first lets its successor in the stream start
// launching, issues the loads that do not depend on earlier kernels (the level's operator - most of its
// bytes), and only then waits for the preceding kernels to complete.  The successor's CTAs fill the SMs
// that the last wave of this grid leaves idle, and the launch latency of the small levels disappears.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// true while the most recent fused launch was one of the persistent pipelined legs (f_down_pp / f_up_pp): the kernel
// after such a leg is launched as an ordinary stream successor (see the comment above those kernels)
inline bool& fused_prev_persistent() {
    static thread_local bool v = false;      // per host thread: launches of one handle come from one thread at a time
    return v;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_fused(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem,
                                cudaStream_t st, bool pdl, Args... args) {
    if (fused_prev_persistent()) pdl = false;
    fused_prev_persistent() = false;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(block, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

#ifndef FUSED_B
#define FUSED_B 128  // window (threads) per CTA of f_down / f_up
#endif
#ifndef FUSED_MINB
#define FUSED_MINB 3   // __launch_bounds__ min CTAs per SM for f_down / f_up
#endif
#define TAIL_B 512     // threads (= max elements of the first tail level) of f_tail

// ---- small helpers ---------------------------------------------------------------------------------
template <int M>
__device__ __forceinline__ void load_vec(const double* __restrict__ p, double (&v)[M]) {
    if constexpr (M % 2 == 0) {
#pragma unroll
        for (int i = 0; i < M; i += 2) {
            const double2 t = *reinterpret_cast<const double2*>(p + i);
            v[i] = t.x;
            v[i + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) v[i] = p[i];
    }
}

template <int M>
__device__ __forceinline__ void store_vec(double* __restrict__ p, const double (&v)[M]) {
    if constexpr (M % 2 == 0) {
#pragma unroll
        for (int i = 0; i < M; i += 2) *reinterpret_cast<double2*>(p + i) = make_double2(v[i], v[i + 1]);
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) p[i] = v[i];
    }
}

// The fast tier handles ST_COLROW levels whose A_up row is the reference's DG trace row (local node 1,
// src/dg_mesh.jl:41-46: left end, right end, interior nodes), so that the row is a compile-time
// register; any other row index stays with the generic tier (fast_tier_ok below).
#define FUSED_COLROW_IUP 1

// Tile rows of the level's operator part per structure class.  The classes that keep the dense FMA chains
// (ST_DENSE, ST_REPEAT) read A_lo(i, j) / A_up(i, j) from the stored entry lo(i, j) / up(i, j).
template <int M, int ST>
struct OpShape {
    static constexpr int NO = ST ? M : M * M;           // stored entries of A_lo (and of A_up)
    static constexpr int O_DI = NO, O_UP = NO + M * M, O_DV = 2 * NO + M * M;
    static constexpr bool DENSE_CHAINS = ST == AMG1D_ST_DENSE || ST == AMG1D_ST_REPEAT;
    __host__ __device__ static constexpr int lo(int i, int j) { return ST == AMG1D_ST_REPEAT ? i : j * M + i; }
    __host__ __device__ static constexpr int up(int i, int j) { return ST == AMG1D_ST_REPEAT ? j : j * M + i; }
};

// y = A_lo xl + A_di xc + A_up xr with the operator streamed from the tile (T points at
// [tile][0][lane]).  Neighbour values: ST_COLROW needs only xl[ilo], passed as xl[0]; ST_ROWCOL needs
// only xr[iup], passed as xr[0]; ST_DENSE and ST_REPEAT need both blocks whole.  Same accumulation
// order as g_row_Ax.
template <int M, int ST>
__device__ __forceinline__ void stream_Ax(const double* __restrict__ T, int ilo, int iup,
                                          const double (&xl)[M], const double (&xc)[M],
                                          const double (&xr)[M], double (&y)[M]) {
    using S = OpShape<M, ST>;
    if constexpr (S::DENSE_CHAINS) {
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = 0.0;
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
            for (int i = 0; i < M; ++i) y[i] = fma(T[S::lo(i, j) * AMG1D_TILE], xl[j], y[i]);
    } else if constexpr (ST == AMG1D_ST_COLROW) {
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = fma(T[i * AMG1D_TILE], xl[0], 0.0);
    } else {
        double yr = 0.0;
#pragma unroll
        for (int j = 0; j < M; ++j) yr = fma(T[j * AMG1D_TILE], xl[j], yr);
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = (i == ilo) ? yr : 0.0;
    }
#pragma unroll
    for (int j = 0; j < M; ++j)
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = fma(T[(S::O_DI + j * M + i) * AMG1D_TILE], xc[j], y[i]);
    if constexpr (S::DENSE_CHAINS) {
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
            for (int i = 0; i < M; ++i) y[i] = fma(T[(S::O_UP + S::up(i, j)) * AMG1D_TILE], xr[j], y[i]);
    } else if constexpr (ST == AMG1D_ST_COLROW) {
        double yr = y[FUSED_COLROW_IUP];
#pragma unroll
        for (int j = 0; j < M; ++j) yr = fma(T[(S::O_UP + j) * AMG1D_TILE], xr[j], yr);
        y[FUSED_COLROW_IUP] = yr;
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = fma(T[(S::O_UP + i) * AMG1D_TILE], xr[0], y[i]);
    }
}

// Neighbour blocks of element e from a global vector, in the form stream_Ax / reg_Ax expect.
template <int M, int ST>
__device__ __forceinline__ void load_neighbours(const double* __restrict__ x, int64_t e, int ilo, int iup,
                                                double (&xl)[M], double (&xr)[M]) {
    if constexpr (ST == AMG1D_ST_COLROW) xl[0] = x[(e - 1) * M + ilo];
    else load_vec<M>(x + (e - 1) * M, xl);
    if constexpr (ST == AMG1D_ST_ROWCOL) xr[0] = x[(e + 1) * M + iup];
    else load_vec<M>(x + (e + 1) * M, xr);
}

// ---- streaming kernels --------------------------------------------------------------------------------
template <int M, bool DIAG, int ST>
__global__ void __launch_bounds__(256) f_sweep(const double* __restrict__ mat, int ilo, int iup,
                                               const double* __restrict__ b,
                                               const double* __restrict__ xin,
                                               double* __restrict__ xout, int64_t n, double alpha,
                                               int zero_guess) {
    using S = OpShape<M, ST>;
    constexpr int K = S::O_DV + (DIAG ? M : M * M);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const double* T = mat + (e >> 5) * (int64_t)(K * AMG1D_TILE) + (e & 31);
    double r[M], xc[M], bb[M];
    load_vec<M>(b + e * M, bb);
    if (zero_guess) {
#pragma unroll
        for (int i = 0; i < M; ++i) { xc[i] = 0.0; r[i] = bb[i] - 0.0; }
    } else {
        double xl[M], xr[M], y[M];
        load_vec<M>(xin + e * M, xc);
        load_neighbours<M, ST>(xin, e, ilo, iup, xl, xr);
        stream_Ax<M, ST>(T, ilo, iup, xl, xc, xr, y);
#pragma unroll
        for (int i = 0; i < M; ++i) r[i] = bb[i] - y[i];
    }
    double xn[M];
    if constexpr (DIAG) {
#pragma unroll
        for (int i = 0; i < M; ++i)
            xn[i] = __dadd_rn(xc[i], __dmul_rn(alpha, T[(S::O_DV + i) * AMG1D_TILE] * r[i]));
    } else {
        double z[M];
#pragma unroll
        for (int i = 0; i < M; ++i) z[i] = 0.0;
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
            for (int i = 0; i < M; ++i) z[i] = fma(T[(S::O_DV + j * M + i) * AMG1D_TILE], r[j], z[i]);
#pragma unroll
        for (int i = 0; i < M; ++i) xn[i] = __dadd_rn(xc[i], __dmul_rn(alpha, z[i]));
    }
    store_vec<M>(xout + e * M, xn);
}

// partial[blockIdx] = sum over the block's elements of || b - A x ||^2
template <int M, int ST>
__global__ void __launch_bounds__(256) f_resnorm(const double* __restrict__ mat, int K, int ilo, int iup,
                                                 const double* __restrict__ b,
                                                 const double* __restrict__ x, int64_t n,
                                                 double* __restrict__ partial) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double s = 0.0;
    if (e < n) {
        const double* T = mat + (e >> 5) * (int64_t)K * AMG1D_TILE + (e & 31);
        double xl[M], xc[M], xr[M], y[M], bb[M];
        load_vec<M>(b + e * M, bb);
        load_vec<M>(x + e * M, xc);
        load_neighbours<M, ST>(x, e, ilo, iup, xl, xr);
        stream_Ax<M, ST>(T, ilo, iup, xl, xc, xr, y);
#pragma unroll
        for (int i = 0; i < M; ++i) { const double r = bb[i] - y[i]; s = fma(r, r, s); }
    }
    s = block_sum(s);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

// y = A x and partial[blockIdx] = sum over the block's elements of x . y   (the p' A p of conjugate
// gradients fused into the product; partial may be null)
template <int M, int ST>
__global__ void __launch_bounds__(256) f_matvec_dot(const double* __restrict__ mat, int K, int ilo, int iup,
                                                    const double* __restrict__ x, double* __restrict__ y,
                                                    int64_t n, double* __restrict__ partial) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double s = 0.0;
    if (e < n) {
        const double* T = mat + (e >> 5) * (int64_t)K * AMG1D_TILE + (e & 31);
        double xl[M], xc[M], xr[M], yy[M];
        load_vec<M>(x + e * M, xc);
        load_neighbours<M, ST>(x, e, ilo, iup, xl, xr);
        stream_Ax<M, ST>(T, ilo, iup, xl, xc, xr, yy);
        store_vec<M>(y + e * M, yy);
#pragma unroll
        for (int i = 0; i < M; ++i) s = fma(xc[i], yy[i], s);
    }
    if (partial) {
        s = block_sum(s);
        if (threadIdx.x == 0) partial[blockIdx.x] = s;
    }
}

// ---- register-resident multi-sweep kernels -----------------------------------------------------------
// Shared-memory exchange buffers, structure-of-arrays so that neighbouring threads hit neighbouring
// banks: xs[buf][i][slot], slot = thread + 1, slots 0 and B+1 stay zero.
template <int M, int B>
struct Exchange {
    double xs[2][M][B + 2];
};

template <int M, int B>
__device__ __forceinline__ void exch_init(Exchange<M, B>& ex) {
    if (threadIdx.x < 2 * M * 2) {
        const int buf = threadIdx.x / (2 * M);
        const int i = (threadIdx.x / 2) % M;
        const int side = threadIdx.x & 1;
        ex.xs[buf][i][side ? B + 1 : 0] = 0.0;
    }
}

// The element's A_lo / A_di / A_up in registers (only the stored entries of the structure class).
template <int M, int ST>
struct RegOp {
    static constexpr bool has_dv = false;
    double lo[OpShape<M, ST>::NO], di[M * M], up[OpShape<M, ST>::NO];
};

// One block set (A_lo, A_di, A_up, Dinv in tile-row order = one row of a pattern table) passed BY VALUE as a
// __grid_constant__ kernel parameter: the entries are constant-bank operands of the FMAs - no loads, no
// registers, no shared memory for the operator.  Used by f_down_c / f_up_c for the CTAs whose whole window
// lies in the translation-invariant interior of a level (option pattern_resident = 2).
template <int M, int ST, bool DIAG>
struct ParamOp {
    static constexpr bool has_dv = true;
    double lo[OpShape<M, ST>::NO], di[M * M], up[OpShape<M, ST>::NO], dv[DIAG ? M : M * M];
};

// The element's blocks AND its block-Jacobi inverse in registers (f_down_dv / f_up_dv: the inverse is computed
// in registers and never goes through shared memory).
template <int M, int ST>
struct RegOpDv {
    static constexpr bool has_dv = true;
    double lo[OpShape<M, ST>::NO], di[M * M], up[OpShape<M, ST>::NO], dv[M * M];
};

template <int M, int ST, class OP>
__device__ __forceinline__ void reg_Ax(const OP& A, int ilo, int iup, const double (&xl)[M],
                                       const double (&xc)[M], const double (&xr)[M], double (&y)[M]) {
    using S = OpShape<M, ST>;
    if constexpr (S::DENSE_CHAINS) {
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = 0.0;
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
            for (int i = 0; i < M; ++i) y[i] = fma(A.lo[S::lo(i, j)], xl[j], y[i]);
    } else if constexpr (ST == AMG1D_ST_COLROW) {
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = fma(A.lo[i], xl[0], 0.0);
    } else {
        double yr = 0.0;
#pragma unroll
        for (int j = 0; j < M; ++j) yr = fma(A.lo[j], xl[j], yr);
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = (i == ilo) ? yr : 0.0;
    }
#pragma unroll
    for (int j = 0; j < M; ++j)
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = fma(A.di[j * M + i], xc[j], y[i]);
    if constexpr (S::DENSE_CHAINS) {
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
            for (int i = 0; i < M; ++i) y[i] = fma(A.up[S::up(i, j)], xr[j], y[i]);
    } else if constexpr (ST == AMG1D_ST_COLROW) {
        double yr = y[FUSED_COLROW_IUP];
#pragma unroll
        for (int j = 0; j < M; ++j) yr = fma(A.up[j], xr[j], yr);
        y[FUSED_COLROW_IUP] = yr;
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = fma(A.up[i], xr[0], y[i]);
    }
}

// one damped (block-)Jacobi sweep on register-resident blocks; same operation order as g_sweep.
// Dinv is read from shared memory: dcol points at this thread's column of ds[k][thread], stride DS.
template <int M, int ST, bool DIAG, int DS, class OP>
__device__ __forceinline__ void reg_sweep(const OP& A, int ilo, int iup,
                                          const double* __restrict__ dcol, const double (&bb)[M],
                                          const double (&xl)[M], double (&xc)[M], const double (&xr)[M],
                                          double alpha, bool zero_guess) {
    double r[M];
    if (zero_guess) {
#pragma unroll
        for (int i = 0; i < M; ++i) r[i] = bb[i] - 0.0;
    } else {
        double y[M];
        reg_Ax<M, ST, OP>(A, ilo, iup, xl, xc, xr, y);
#pragma unroll
        for (int i = 0; i < M; ++i) r[i] = bb[i] - y[i];
    }
    if constexpr (DIAG) {
#pragma unroll
        for (int i = 0; i < M; ++i) {
            double dvi;
            if constexpr (OP::has_dv) dvi = A.dv[i]; else dvi = dcol[i * DS];
            xc[i] = __dadd_rn(xc[i], __dmul_rn(alpha, dvi * r[i]));
        }
    } else {
        double z[M];
#pragma unroll
        for (int i = 0; i < M; ++i) z[i] = 0.0;
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
            for (int i = 0; i < M; ++i) {
                double dvk;
                if constexpr (OP::has_dv) dvk = A.dv[j * M + i]; else dvk = dcol[(j * M + i) * DS];
                z[i] = fma(dvk, r[j], z[i]);
            }
#pragma unroll
        for (int i = 0; i < M; ++i) xc[i] = __dadd_rn(xc[i], __dmul_rn(alpha, z[i]));
    }
}

__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gmem_src) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// In-register inverse of a dense M x M block (column-major: entry (r, c) at a[c * M + r]): Gauss-Jordan with
// partial pivoting, statement for statement the arithmetic of k_dinv_recompute (device_setup.cuh) so that the
// result equals the stored inverse bit for bit.  The pivot search is a chain of compare-and-swap steps (row r
// is swapped up whenever |a(r, c)| exceeds the current pivot candidate, which leaves the largest entry on the
// diagonal) recorded as booleans: every array index is a compile-time constant and the swaps are selects, so
// the block never leaves the register file (an integer pivot index made the compiler index local memory).
// PIV = false: the level's set-up pass found that no element ever swaps (every pivot already sits on the diagonal,
// as for the symmetric positive definite, diagonally heavy blocks of the DG operators) - the compare-and-swap
// chain is skipped, which leaves exactly the same arithmetic at a third of the instructions.
template <int M, bool PIV>
__device__ __forceinline__ void reg_invert(double (&a)[M * M]) {
    bool sw[M][M];
#pragma unroll
    for (int c = 0; c < M; ++c) {
        if constexpr (PIV) {
#pragma unroll
        for (int r = c + 1; r < M; ++r) {
            const bool s = fabs(a[c * M + r]) > fabs(a[c * M + c]);
            sw[c][r] = s;
#pragma unroll
            for (int q = 0; q < M; ++q) {
                const double x = a[q * M + c], y = a[q * M + r];
                a[q * M + c] = s ? y : x;
                a[q * M + r] = s ? x : y;
            }
        }
        }
        const double dd = 1.0 / a[c * M + c];
        a[c * M + c] = 1.0;
#pragma unroll
        for (int q = 0; q < M; ++q) a[q * M + c] *= dd;
#pragma unroll
        for (int r = 0; r < M; ++r) {
            if (r == c) continue;
            const double f = a[c * M + r];
            a[c * M + r] = 0.0;
#pragma unroll
            for (int q = 0; q < M; ++q) a[q * M + r] = fma(-f, a[q * M + c], a[q * M + r]);
        }
    }
    if constexpr (PIV) {
#pragma unroll
    for (int c = M - 1; c >= 0; --c) {            // undo the row swaps as column swaps, in reverse order
#pragma unroll
        for (int r2 = M - 1; r2 > c; --r2) {
            const bool s = sw[c][r2];
#pragma unroll
            for (int r = 0; r < M; ++r) {
                const double x = a[c * M + r], y = a[r2 * M + r];
                a[c * M + r] = s ? y : x;
                a[r2 * M + r] = s ? x : y;
            }
        }
    }
    }
}

// Option recompute_dinv: this thread's Dinv = inv(A_di) from the registers into its shared-memory column
// (rec = 1: with the pivot chain, 2: the level never pivots).  Called right after the operator loads, BEFORE the
// programmatic-dependency wait and the vector loads: placing it after them (to overlap their latency) was
// measured 40 % slower on T level 0 - the vectors' registers are then live across the inversion and it spills.
template <int M, int B, int ST, bool DIAG>
__device__ __forceinline__ void recompute_dinv(const RegOp<M, ST>& A, double (*ds)[B], bool active, int rec) {
    if constexpr (!DIAG) {
        if (rec && active) {
            double w[M * M];
#pragma unroll
            for (int k = 0; k < M * M; ++k) w[k] = A.di[k];
            if (rec == 2) reg_invert<M, false>(w); else reg_invert<M, true>(w);
#pragma unroll
            for (int k = 0; k < M * M; ++k) ds[k][threadIdx.x] = w[k];
        }
    }
}
template <int M, int B, int ST, bool DIAG>
__device__ __forceinline__ void recompute_dinv(const ParamOp<M, ST, DIAG>&, double (*)[B], bool, int) {}

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }

template <int M, int ST, class OP>
__device__ __forceinline__ void reg_residual(const OP& A, int ilo, int iup,
                                             const double (&bb)[M], const double (&xl)[M],
                                             const double (&xc)[M], const double (&xr)[M],
                                             double (&r)[M]) {
    double y[M];
    reg_Ax<M, ST, OP>(A, ilo, iup, xl, xc, xr, y);
#pragma unroll
    for (int i = 0; i < M; ++i) r[i] = bb[i] - y[i];
}

// publish x into exchange buffer `buf`, barrier, fetch what the structure class needs of both neighbours
template <int M, int B, int ST>
__device__ __forceinline__ void exchange(Exchange<M, B>& ex, int buf, int ilo, int iup,
                                         const double (&xc)[M], double (&xl)[M], double (&xr)[M]) {
    const int t = threadIdx.x;
#pragma unroll
    for (int i = 0; i < M; ++i) ex.xs[buf][i][t + 1] = xc[i];
    __syncthreads();
    if constexpr (ST == AMG1D_ST_COLROW) {
        xl[0] = ex.xs[buf][ilo][t];
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) xl[i] = ex.xs[buf][i][t];
    }
    if constexpr (ST == AMG1D_ST_ROWCOL) {
        xr[0] = ex.xs[buf][iup][t + 2];
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) xr[i] = ex.xs[buf][i][t + 2];
    }
}

// A_lo / A_di / A_up go to registers; Dinv (used once per sweep) is copied global -> shared with
// cp.async, i.e. without register staging, into this thread's own column ds[k][thread].
// rec (block smoothers, streamed tiles only): Dinv is NOT loaded - the leg inverts A.di in registers
// (recompute_dinv) and puts the result into the same shared-memory column.
template <int M, int B, int ST, bool DIAG, int STRIDE>
__device__ __forceinline__ void load_blocks_from(const double* __restrict__ T, RegOp<M, ST>& A, double (*ds)[B],
                                                 bool rec = false) {
    using S = OpShape<M, ST>;
    constexpr int ND = DIAG ? M : M * M;
    const int t = threadIdx.x;
    if constexpr (STRIDE == 1) {   // pattern table: every lane reads the same address - plain loads broadcast
#pragma unroll                     // (cp.async with one source address per warp was measured far slower)
        for (int k = 0; k < ND; ++k) ds[k][t] = T[S::O_DV + k];
    } else {
        if (!rec) {
#pragma unroll
            for (int k = 0; k < ND; ++k) cp_async8(&ds[k][t], T + (S::O_DV + k) * STRIDE);
        }
    }
#pragma unroll
    for (int k = 0; k < S::NO; ++k) A.lo[k] = T[k * STRIDE];
#pragma unroll
    for (int k = 0; k < M * M; ++k) A.di[k] = T[(S::O_DI + k) * STRIDE];
#pragma unroll
    for (int k = 0; k < S::NO; ++k) A.up[k] = T[(S::O_UP + k) * STRIDE];
}

// e = local element index (addresses the element tiles), eg = global element index (addresses the
// pattern table of a translation-invariant level, PatOp)
template <int M, int B, int ST, bool DIAG>
__device__ __forceinline__ void load_blocks(const double* __restrict__ mat, const PatOp& po, int64_t e,
                                            int64_t eg, bool active, RegOp<M, ST>& A, double (*ds)[B],
                                            bool rec = false) {
    using S = OpShape<M, ST>;
    constexpr int ND = DIAG ? M : M * M;
    constexpr int K = S::O_DV + ND;
    const int t = threadIdx.x;
    if (po.tab != nullptr) active = active && eg >= 0 && eg < po.n_glob;
    if (active) {
        if (po.tab != nullptr) {
            const int64_t s = eg < po.n_head ? eg
                            : (eg >= po.n_glob - po.n_tail ? po.n_head + 1 + (eg - (po.n_glob - po.n_tail))
                                                           : po.n_head);
            load_blocks_from<M, B, ST, DIAG, 1>(po.tab + s * K, A, ds);
        } else {
            load_blocks_from<M, B, ST, DIAG, AMG1D_TILE>(mat + (e >> 5) * (int64_t)(K * AMG1D_TILE) + (e & 31), A, ds,
                                                         rec);
        }
    } else {
#pragma unroll
        for (int k = 0; k < ND; ++k) ds[k][t] = 0.0;
#pragma unroll
        for (int k = 0; k < S::NO; ++k) { A.lo[k] = 0.0; A.up[k] = 0.0; }
#pragma unroll
        for (int k = 0; k < M * M; ++k) A.di[k] = 0.0;
    }
}

// Resident CTAs per SM the register allocation aims for.  Dense 4x4 blocks keep 48 operator doubles in
// registers (164 registers, 3 CTAs of 128 threads); the compressed structure classes keep 24 and fit 5
// CTAs (<= 102 registers, no spills), which is what hides the compute phase of one CTA behind the load
// phase of the others (measured on B200, T level 0: 5.0 -> 4.5 ms per leg; 6 CTAs spill and lose).  The
// 2x2 and 1x1 kernels are capped at 64 registers for 8 CTAs/SM.
#ifndef FUSED_MINB_SMALL
#define FUSED_MINB_SMALL 8   // m <= 2: <= 64 registers, no spills; measured best of 3 / 8 / 10 / 12 (T: -4 %)
#endif                       // ST_REPEAT 2x2 legs: 56 registers; 10 CTAs (48, spills) measured slower (DESIGN 6)
constexpr int fused_min_blocks(int m, int st) {
    return m >= 5 ? (st != AMG1D_ST_DENSE ? 3 : 2)
         : m == 4 ? (st != AMG1D_ST_DENSE ? 5 : 3)
         : m <= 2 ? FUSED_MINB_SMALL : FUSED_MINB;
}
#define FUSED_BOUNDS(M) __launch_bounds__(B, fused_min_blocks(M, ST))
// The constant-operand legs (f_down_c / f_up_c) keep no operator in registers on their interior path, so
// they can be given more resident CTAs than f_down / f_up; their table path (the few CTAs at the ends of a
// level) then spills, which costs nothing measurable.  0 = the bounds of f_down / f_up.
#ifndef FUSED_C_MINB3
#define FUSED_C_MINB3 8   // C3 level 1 (3 x 3 dense): 0.535 / 0.546 ms per leg at 3 CTAs/SM, 0.369 / 0.364 at 8
#endif
#ifndef FUSED_C_MINB4
#define FUSED_C_MINB4 8   // measured on B200 (T level 0, profiles/r01e_sweep_const.jsonl): 5 CTAs/SM (the bounds
#endif                    // of f_down / f_up) 2.31 / 2.03 ms per leg, 6: 2.12 / 1.94, 8 (64 registers): 1.99 / 1.92
#ifndef FUSED_C_MINB5
#define FUSED_C_MINB5 0   // 5 x 5: the interior path needs the registers (6 CTAs/SM: 1.86 / 1.81 ms against 1.01 / 0.98;
#endif                    // profiles/r01f_sweep_const.jsonl)
constexpr int fused_c_min_blocks(int m, int st) {
    return (m == 3 && FUSED_C_MINB3) ? FUSED_C_MINB3 : (m == 4 && FUSED_C_MINB4) ? FUSED_C_MINB4
         : (m >= 5 && FUSED_C_MINB5) ? FUSED_C_MINB5 : fused_min_blocks(m, st);
}
#define FUSED_C_BOUNDS(M) __launch_bounds__(B, fused_c_min_blocks(M, ST))

// nsweep pre-smoothing sweeps, residual, restriction to the coarse right-hand side.
//   halo window elements on each side are recomputed (nsweep + 1, plus `ratio` for two-parent
//   transfers whose coarse elements also gather from the children of their left neighbour);
//   out = elements emitted per CTA (a multiple of the agglomeration ratio).
//   Coarse element Kc is gathered by the thread of its first P0-child, in the order of g_restrict:
//   the P1 blocks of the children of Kc - 1, then the P0 blocks of its own children.
// down_body: the leg of window `win` (elements [win * out - halo, win * out - halo + B) of the slab) once the
// operator (A: RegOp in registers + Dinv column dcol in shared memory, RegOpDv, or ParamOp in the constant bank) and
// the thread's right-hand side bb / incoming iterate xc are in registers.  One CTA per window (f_down, f_down_dv,
// f_down_c: win = blockIdx.x) or a persistent CTA walking over windows (f_down_pp).
// SINGLE: the launcher knows that every coarse element has exactly one child and one parent transfer (ratio == 1, no
// P1 - the p-coarsening transfers dg_dg): the thread restricts its own residual straight from registers, the trip
// through shared memory and its barrier are not needed (same products in the same order).
template <int M, int MC, int B, int ST, bool DIAG, class OP, int NSW = 0, bool SINGLE = false>   // NSW > 0: nsweep known at compile time
__device__ __forceinline__ void
down_body(const OP& A, const double* __restrict__ dcol, Exchange<M, B>& ex, double (*rs)[B + 8], int64_t e, int64_t win,
          const double (&bb)[M], double (&xc)[M], int ilo, int iup, double* __restrict__ xout,
          const double* __restrict__ P0, const double* __restrict__ P1, const TransferMap& tm,
          double* __restrict__ rc, int64_t n, double alpha, int nsweep, int zero_guess, const WinIdx& wi,
          const Slab& sl, const HaloLeg& hl) {
    const int t = threadIdx.x;
    const int halo = wi.halo, out = wi.out;
    double xl[M], xr[M];
    int buf = 0;
    if constexpr (NSW > 0) {
#pragma unroll
        for (int s = 0; s < NSW; ++s) {
            const bool zg = zero_guess && s == 0;
            if (!zg) {
                exchange<M, B, ST>(ex, buf, ilo, iup, xc, xl, xr);
                buf ^= 1;
            }
            reg_sweep<M, ST, DIAG, B>(A, ilo, iup, dcol, bb, xl, xc, xr, alpha, zg);
        }
    } else {
        for (int s = 0; s < nsweep; ++s) {
            const bool zg = zero_guess && s == 0;
            if (!zg) {
                exchange<M, B, ST>(ex, buf, ilo, iup, xc, xl, xr);
                buf ^= 1;
            }
            reg_sweep<M, ST, DIAG, B>(A, ilo, iup, dcol, bb, xl, xc, xr, alpha, zg);
        }
    }
    const bool mine = t >= halo && t < halo + out;              // this window's share of the level (e >= 0)
    if (mine && e < n) {
        store_vec<M>(xout + e * M, xc);
        if (hl.on) halo_leg_push<M>(xc, e, n, hl.gd, hl.x_left, hl.x_right, hl.f_left, hl.f_right);
    }
    // residual with the final iterate, then restriction
    exchange<M, B, ST>(ex, buf, ilo, iup, xc, xl, xr);
    double r[M];
    reg_residual<M, ST>(A, ilo, iup, bb, xl, xc, xr, r);
    const int64_t eg = e + sl.e_off;                            // global element index
    if constexpr (SINGLE) {
        if (mine && eg < tm.n_fine) {
            const int64_t Kc = win * wi.opr + wi.qdiv0 + (wi.qmod0 + t) + tm.base;     // ratio == 1: kdiv = qmod0 + t, kmod = 0
            const int64_t Kl = Kc - sl.c_off;                   // local coarse element index
            if (Kc >= 0 && Kc < tm.n_coarse && Kl >= 0 && Kl < sl.nc) {
                const double* P = P0 + win_blk(tm, wi, eg, t) * (M * MC);
                double acc[MC];
#pragma unroll
                for (int j = 0; j < MC; ++j) acc[j] = 0.0;
#pragma unroll
                for (int j = 0; j < MC; ++j)
#pragma unroll
                    for (int i = 0; i < M; ++i) acc[j] = fma(P[j * M + i], r[i], acc[j]);
#pragma unroll
                for (int j = 0; j < MC; ++j) rc[Kl * MC + j] = acc[j];
                if (hl.on) halo_leg_push<MC>(acc, Kl, hl.nc, hl.gd, hl.c_left, hl.c_right, hl.f_left, hl.f_right);
            }
        }
        return;
    }
#pragma unroll
    for (int i = 0; i < M; ++i) rs[i][t] = r[i];
    __syncthreads();
    if (mine && eg < tm.n_fine) {
        int kdiv, kmod;                                         // (eg + shift) = ratio * (.. + kdiv) + kmod
        small_divmod(wi.qmod0 + t, tm.ratio, &kdiv, &kmod);
        if (kmod == 0) {
            const int64_t Kc = win * wi.opr + wi.qdiv0 + kdiv + tm.base;   // eg == tm.first(Kc)
            const int64_t Kl = Kc - sl.c_off;                   // local coarse element index
            if (Kc >= 0 && Kc < tm.n_coarse && Kl >= 0 && Kl < sl.nc) {
                double acc[MC];
#pragma unroll
                for (int j = 0; j < MC; ++j) acc[j] = 0.0;
                if (P1) {                                       // children of Kc - 1: [eg - ratio, eg), clamped
                    const int k0 = eg >= tm.ratio ? -tm.ratio : -(int)eg;
                    for (int k = k0; k < 0; ++k) {
                        const double* P = P1 + win_blk(tm, wi, eg + k, t + k) * (M * MC);
                        const int w = t + k;
#pragma unroll
                        for (int j = 0; j < MC; ++j)
#pragma unroll
                            for (int i = 0; i < M; ++i) acc[j] = fma(P[j * M + i], rs[i][w], acc[j]);
                    }
                }
                const int k1 = eg + tm.ratio <= tm.n_fine ? tm.ratio : (int)(tm.n_fine - eg);   // own children
                for (int k = 0; k < k1; ++k) {
                    const double* P = P0 + win_blk(tm, wi, eg + k, t + k) * (M * MC);
                    const int w = t + k;
#pragma unroll
                    for (int j = 0; j < MC; ++j)
#pragma unroll
                        for (int i = 0; i < M; ++i) acc[j] = fma(P[j * M + i], rs[i][w], acc[j]);
                }
#pragma unroll
                for (int j = 0; j < MC; ++j) rc[Kl * MC + j] = acc[j];
                if (hl.on) halo_leg_push<MC>(acc, Kl, hl.nc, hl.gd, hl.c_left, hl.c_right, hl.f_left, hl.f_right);
            }
        }
    }
}

// The one-window-per-CTA leg after the operator has been placed: everything from the dependency wait on.
template <int M, int MC, int B, int ST, bool DIAG, class OP>
__device__ __forceinline__ void
down_leg(const OP& A, const double* __restrict__ dcol, Exchange<M, B>& ex, double (*rs)[B + 8], int64_t e,
         bool active, int ilo, int iup, const double* __restrict__ b, const double* __restrict__ xin,
         double* __restrict__ xout, const double* __restrict__ P0, const double* __restrict__ P1,
         const TransferMap& tm, double* __restrict__ rc, int64_t n, double alpha, int nsweep, int zero_guess,
         const WinIdx& wi, const Slab& sl, const HaloLeg& hl) {
    double bb[M], xc[M];
    pdl_wait();                                                  // b, x and everything written below are not
    {   // peer-memory exchange: CTAs whose window reaches a slab edge wait for the neighbour's edge (halo_p2p.cuh)
        const int64_t e0 = (int64_t)blockIdx.x * wi.out - wi.halo;
        halo_leg_wait(hl, sl.gl > 0 && e0 < 0, sl.gr > 0 && e0 + B > n);
    }
    if (active) {
        load_vec<M>(b + e * M, bb);
        if (zero_guess) {
#pragma unroll
            for (int i = 0; i < M; ++i) xc[i] = 0.0;
        } else {
            load_vec<M>(xin + e * M, xc);
        }
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) { bb[i] = 0.0; xc[i] = 0.0; }
    }
    cp_async_commit_wait_all();  // this thread's Dinv column has landed (only this thread reads it)
    __syncthreads();             // exch_init visible
    down_body<M, MC, B, ST, DIAG>(A, dcol, ex, rs, e, (int64_t)blockIdx.x, bb, xc, ilo, iup, xout, P0, P1, tm, rc, n,
                                  alpha, nsweep, zero_guess, wi, sl, hl);
}

template <int M, int MC, int B, int ST, bool DIAG>
__global__ void FUSED_BOUNDS(M)
f_down(const double* __restrict__ mat, PatOp po, int ilo, int iup, const double* __restrict__ b,
       const double* __restrict__ xin, double* __restrict__ xout, const double* __restrict__ P0,
       const double* __restrict__ P1, TransferMap tm, double* __restrict__ rc, int64_t n, double alpha,
       int nsweep, int zero_guess, WinIdx wi, Slab sl, int rec, const __grid_constant__ HaloLeg hl) {
    __shared__ Exchange<M, B> ex;
    __shared__ double rs[M][B + 8];
    __shared__ double ds[DIAG ? M : M * M][B];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + t;     // local element index (ghosts < 0, >= n)
    const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
    exch_init<M, B>(ex);
    RegOp<M, ST> A;
    load_blocks<M, B, ST, DIAG>(mat, po, e, e + sl.e_off, active, A, ds, rec != 0);   // operator: independent of earlier kernels
    recompute_dinv<M, B, ST, DIAG>(A, ds, active, rec);          // before the dependency wait: few registers are live yet
    down_leg<M, MC, B, ST, DIAG>(A, &ds[0][t], ex, rs, e, active, ilo, iup, b, xin, xout, P0, P1, tm, rc, n, alpha,
                                 nsweep, zero_guess, wi, sl, hl);
}

// CTA-uniform test of the constant-operand legs: the whole window of this CTA is active (inside the slab
// and its ghosts) and lies in the translation-invariant interior of the level, i.e. every thread would
// fetch row n_head of the pattern table.
__device__ __forceinline__ bool window_is_interior(const PatOp& po, const WinIdx& wi, const Slab& sl, int64_t n,
                                                   int B) {
    const int64_t e0 = (int64_t)blockIdx.x * wi.out - wi.halo;        // local element of thread 0
    const int64_t g0 = e0 + sl.e_off;                                 // its global number
    return e0 >= -(int64_t)sl.gl && e0 + B <= n + sl.gr && g0 >= po.n_head && g0 + B <= po.n_glob - po.n_tail;
}

// f_down with the interior block set of a pattern level as a by-value kernel parameter (ParamOp): interior
// CTAs run the leg with constant-bank operands, the few CTAs that touch the head / tail block sets, a slab
// end or the end of the level take the register path of f_down (pattern table, po.tab != nullptr).
template <int M, int MC, int B, int ST, bool DIAG>
__global__ void FUSED_C_BOUNDS(M)
f_down_c(const __grid_constant__ ParamOp<M, ST, DIAG> pk, PatOp po, int ilo, int iup,
         const double* __restrict__ b, const double* __restrict__ xin, double* __restrict__ xout,
         const double* __restrict__ P0, const double* __restrict__ P1, TransferMap tm, double* __restrict__ rc,
         int64_t n, double alpha, int nsweep, int zero_guess, WinIdx wi, Slab sl,
         const __grid_constant__ HaloLeg hl) {
    __shared__ Exchange<M, B> ex;
    __shared__ double rs[M][B + 8];
    __shared__ double ds[DIAG ? M : M * M][B];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + t;
    exch_init<M, B>(ex);
    if (window_is_interior(po, wi, sl, n, B)) {
        down_leg<M, MC, B, ST, DIAG>(pk, nullptr, ex, rs, e, true, ilo, iup, b, xin, xout, P0, P1, tm, rc, n, alpha,
                                     nsweep, zero_guess, wi, sl, hl);
    } else {
        const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
        RegOp<M, ST> A;
        load_blocks<M, B, ST, DIAG>(nullptr, po, e, e + sl.e_off, active, A, ds);
        down_leg<M, MC, B, ST, DIAG>(A, &ds[0][t], ex, rs, e, active, ilo, iup, b, xin, xout, P0, P1, tm, rc, n,
                                     alpha, nsweep, zero_guess, wi, sl, hl);
    }
}

// x += P0 x_c[parent] (+ P1 x_c[parent + 1]) for window thread t of window `win`; c0 / c1 = the MC values of the
// parent(s) (same operation order as g_prolong)
template <int M, int MC>
__device__ __forceinline__ void up_correct(double (&xc)[M], const double* __restrict__ P0, const double* __restrict__ P1,
                                           int64_t pb, const double (&c0)[MC], const double (&c1)[MC]) {
    double y[M];
#pragma unroll
    for (int i = 0; i < M; ++i) y[i] = 0.0;
#pragma unroll
    for (int j = 0; j < MC; ++j)
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = fma(P0[pb + j * M + i], c0[j], y[i]);
    if (P1) {
#pragma unroll
        for (int j = 0; j < MC; ++j)
#pragma unroll
            for (int i = 0; i < M; ++i) y[i] = fma(P1[pb + j * M + i], c1[j], y[i]);
    }
#pragma unroll
    for (int i = 0; i < M; ++i) xc[i] = xc[i] + y[i];
}

// up_body: nsweep post-smoothing sweeps of window `win` on the corrected iterate xc, emission, optional
// || b - A x ||^2 partial sum of the window (partial[win]).
template <int M, int MC, int B, int ST, bool DIAG, class OP, int NSW = 0>
__device__ __forceinline__ void
up_body(const OP& A, const double* __restrict__ dcol, Exchange<M, B>& ex, int64_t e, int64_t win,
        const double (&bb)[M], double (&xc)[M], int ilo, int iup, double* __restrict__ xout, int64_t n, double alpha,
        int nsweep, const WinIdx& wi, double* __restrict__ partial, const HaloLeg& hl) {
    const int t = threadIdx.x;
    const int halo = wi.halo, out = wi.out;
    double xl[M], xr[M];
    int buf = 0;
    if constexpr (NSW > 0) {
#pragma unroll
        for (int s = 0; s < NSW; ++s) {
            exchange<M, B, ST>(ex, buf, ilo, iup, xc, xl, xr);
            buf ^= 1;
            reg_sweep<M, ST, DIAG, B>(A, ilo, iup, dcol, bb, xl, xc, xr, alpha, false);
        }
    } else {
        for (int s = 0; s < nsweep; ++s) {
            exchange<M, B, ST>(ex, buf, ilo, iup, xc, xl, xr);
            buf ^= 1;
            reg_sweep<M, ST, DIAG, B>(A, ilo, iup, dcol, bb, xl, xc, xr, alpha, false);
        }
    }
    const bool emit = e < n && t >= halo && t < halo + out;     // e >= 0 for these threads
    if (emit) {
        store_vec<M>(xout + e * M, xc);
        if (hl.on) halo_leg_push<M>(xc, e, n, hl.gd, hl.x_left, hl.x_right, hl.f_left, hl.f_right);
    }
    if (partial) {
        exchange<M, B, ST>(ex, buf, ilo, iup, xc, xl, xr);
            double r[M];
        reg_residual<M, ST>(A, ilo, iup, bb, xl, xc, xr, r);
        double s2 = 0.0;
        if (emit) {
#pragma unroll
            for (int i = 0; i < M; ++i) s2 = fma(r[i], r[i], s2);
        }
        s2 = block_sum(s2);
        if (t == 0) partial[win] = s2;
    }
}

// prolongation + correction, nsweep post-smoothing sweeps, optional || b - A x ||^2 partial sums.
template <int M, int MC, int B, int ST, bool DIAG, class OP>
__device__ __forceinline__ void
up_leg(const OP& A, const double* __restrict__ dcol, Exchange<M, B>& ex, int64_t e, bool active, int ilo, int iup,
       const double* __restrict__ b, const double* __restrict__ xin, double* __restrict__ xout,
       const double* __restrict__ P0, const double* __restrict__ P1, const TransferMap& tm,
       const double* __restrict__ xcoarse, int64_t n, double alpha, int nsweep, const WinIdx& wi,
       double* __restrict__ partial, const Slab& sl, const HaloLeg& hl) {
    const int t = threadIdx.x;
    double bb[M], xc[M];
    pdl_wait();
    {   // peer-memory exchange: the CTAs near a slab edge read fine ghosts and / or ghosts of the coarse correction
        const int64_t e0 = (int64_t)blockIdx.x * wi.out - wi.halo;
        halo_leg_wait(hl, sl.gl > 0 && e0 < tm.ratio + 1, sl.gr > 0 && e0 + B + tm.ratio + 1 > n);
    }
    if (active) {
        load_vec<M>(b + e * M, bb);
        load_vec<M>(xin + e * M, xc);
        // x += P0 x_c[parent] (+ P1 x_c[parent + 1])   (same operation order as g_prolong)
        const int64_t eg = e + sl.e_off;
        const int64_t pb = win_blk(tm, wi, eg, t) * (M * MC);
        int kdiv, kmod;
        small_divmod(wi.qmod0 + t, tm.ratio, &kdiv, &kmod);
        const int64_t par = (int64_t)blockIdx.x * wi.opr + wi.qdiv0 + kdiv + tm.base;   // == tm.par(eg)
        const double* c0 = xcoarse + (par - sl.c_off) * MC;
        double y[M];
#pragma unroll
        for (int i = 0; i < M; ++i) y[i] = 0.0;
#pragma unroll
        for (int j = 0; j < MC; ++j) {
            const double cj = c0[j];
#pragma unroll
            for (int i = 0; i < M; ++i) y[i] = fma(P0[pb + j * M + i], cj, y[i]);
        }
        if (P1) {
#pragma unroll
            for (int j = 0; j < MC; ++j) {
                const double cj = c0[MC + j];
#pragma unroll
                for (int i = 0; i < M; ++i) y[i] = fma(P1[pb + j * M + i], cj, y[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < M; ++i) xc[i] = xc[i] + y[i];
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) { bb[i] = 0.0; xc[i] = 0.0; }
    }
    cp_async_commit_wait_all();
    __syncthreads();
    up_body<M, MC, B, ST, DIAG>(A, dcol, ex, e, (int64_t)blockIdx.x, bb, xc, ilo, iup, xout, n, alpha, nsweep, wi,
                                partial, hl);
}

template <int M, int MC, int B, int ST, bool DIAG>
__global__ void FUSED_BOUNDS(M)
f_up(const double* __restrict__ mat, PatOp po, int ilo, int iup, const double* __restrict__ b,
     const double* __restrict__ xin, double* __restrict__ xout, const double* __restrict__ P0,
     const double* __restrict__ P1, TransferMap tm, const double* __restrict__ xcoarse, int64_t n,
     double alpha, int nsweep, WinIdx wi, double* __restrict__ partial, Slab sl, int rec,
     const __grid_constant__ HaloLeg hl) {
    __shared__ Exchange<M, B> ex;
    __shared__ double ds[DIAG ? M : M * M][B];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + t;
    const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
    exch_init<M, B>(ex);
    RegOp<M, ST> A;
    load_blocks<M, B, ST, DIAG>(mat, po, e, e + sl.e_off, active, A, ds, rec != 0);   // operator: independent of earlier kernels
    recompute_dinv<M, B, ST, DIAG>(A, ds, active, rec);          // before the dependency wait: few registers are live yet
    up_leg<M, MC, B, ST, DIAG>(A, &ds[0][t], ex, e, active, ilo, iup, b, xin, xout, P0, P1, tm, xcoarse, n, alpha,
                               nsweep, wi, partial, sl, hl);
}

// ---- the legs with the inverse in REGISTERS (option dinv_registers) ---------------------------------------------
// ncu of f_down / f_up with the recomputed inverse (profiles/r02_summary.md): DRAM traffic = algorithmic bytes, but
// the L1 / shared-memory pipe is the busiest unit at 82-85 % - operator loads, iterate exchange, and the inverse
// written to and read back from shared memory once per sweep (64 of ~165 LSU instructions per element).  These
// variants keep the inverse where reg_invert leaves it: 16 more live doubles (4 x 4), hence 4 instead of 5 resident
// CTAs per SM, no shared memory for it at all.  Block smoothers, streamed tiles only; same arithmetic, same bits.
template <int M, int ST>
__device__ __forceinline__ void load_blocks_dv(const double* __restrict__ mat, int64_t e, bool active, int rec,
                                               RegOpDv<M, ST>& A) {
    using S = OpShape<M, ST>;
    constexpr int K = S::O_DV + M * M;
    if (active) {
        const double* T = mat + (e >> 5) * (int64_t)(K * AMG1D_TILE) + (e & 31);
#pragma unroll
        for (int k = 0; k < S::NO; ++k) A.lo[k] = T[k * AMG1D_TILE];
#pragma unroll
        for (int k = 0; k < M * M; ++k) A.di[k] = T[(S::O_DI + k) * AMG1D_TILE];
#pragma unroll
        for (int k = 0; k < S::NO; ++k) A.up[k] = T[(S::O_UP + k) * AMG1D_TILE];
#pragma unroll
        for (int k = 0; k < M * M; ++k) A.dv[k] = A.di[k];
        if ((rec & 3) == 2) reg_invert<M, false>(A.dv); else reg_invert<M, true>(A.dv);
    } else {
#pragma unroll
        for (int k = 0; k < S::NO; ++k) { A.lo[k] = 0.0; A.up[k] = 0.0; }
#pragma unroll
        for (int k = 0; k < M * M; ++k) { A.di[k] = 0.0; A.dv[k] = 0.0; }
    }
}

constexpr int fused_dv_min_blocks(int m) { return m >= 4 ? 4 : 8; }
inline bool fused_has_dv(int m, int mc, int st, int diag) {
    return !diag && ((m == 4 && st == AMG1D_ST_COLROW && (mc == 2 || mc == 3)) || (m == 2 && mc == 2 && st != AMG1D_ST_ROWCOL));
}

template <int M, int MC, int B, int ST>
__global__ void __launch_bounds__(B, fused_dv_min_blocks(M))
f_down_dv(const double* __restrict__ mat, int ilo, int iup, const double* __restrict__ b,
          const double* __restrict__ xin, double* __restrict__ xout, const double* __restrict__ P0,
          const double* __restrict__ P1, TransferMap tm, double* __restrict__ rc, int64_t n, double alpha,
          int nsweep, int zero_guess, WinIdx wi, Slab sl, int rec, const __grid_constant__ HaloLeg hl) {
    __shared__ Exchange<M, B> ex;
    __shared__ double rs[M][B + 8];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + t;
    const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
    exch_init<M, B>(ex);
    RegOpDv<M, ST> A;
    load_blocks_dv<M, ST>(mat, e, active, rec, A);               // operator + inversion: independent of earlier kernels
    down_leg<M, MC, B, ST, false>(A, nullptr, ex, rs, e, active, ilo, iup, b, xin, xout, P0, P1, tm, rc, n, alpha,
                                  nsweep, zero_guess, wi, sl, hl);
}

template <int M, int MC, int B, int ST>
__global__ void __launch_bounds__(B, fused_dv_min_blocks(M))
f_up_dv(const double* __restrict__ mat, int ilo, int iup, const double* __restrict__ b,
        const double* __restrict__ xin, double* __restrict__ xout, const double* __restrict__ P0,
        const double* __restrict__ P1, TransferMap tm, const double* __restrict__ xcoarse, int64_t n,
        double alpha, int nsweep, WinIdx wi, double* __restrict__ partial, Slab sl, int rec,
        const __grid_constant__ HaloLeg hl) {
    __shared__ Exchange<M, B> ex;
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + t;
    const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
    exch_init<M, B>(ex);
    RegOpDv<M, ST> A;
    load_blocks_dv<M, ST>(mat, e, active, rec, A);
    up_leg<M, MC, B, ST, false>(A, nullptr, ex, e, active, ilo, iup, b, xin, xout, P0, P1, tm, xcoarse, n, alpha,
                                nsweep, wi, partial, sl, hl);
}

// ---- pipelined persistent legs (option leg_pipeline): TMA bulk copies + mbarrier, one window ahead -----------------
// What still separates f_down_dv / f_up_dv from the HBM roofline is not a saturated unit but the life of a CTA: load
// the operator (one memory latency), invert, wait for the predecessor, load the vectors (a second latency), sweep,
// store - with 4 resident CTAs per SM the bytes in flight per SM average ~45 KB, about what 6.5 TB/s needs at the
// loaded latency, and nothing hides the gaps.  f_down_pp / f_up_pp are the same legs as PERSISTENT CTAs (4 per SM):
// CTA c walks over the windows c, c + grid, c + 2 grid ...; while it computes window w out of registers, the
// operator tiles and the b / x slices of its NEXT window are already in flight into shared memory - 1-D bulk copies
// (cp.async.bulk.shared::cluster.global, the TMA engine: no registers, no LSU instructions) issued by the lanes of
// warp 0 and signalled through one mbarrier per CTA (expect_tx = bytes issued; parity flips per window).  A window of
// B = 128 elements starts at w * out - halo, which is never tile aligned, so the stage holds the B / 32 + 1 element
// tiles it touches - only their A_lo / A_di / A_up rows, which are contiguous at the start of a tile; the inverse
// is recomputed in registers (reg_invert) as in f_*_dv - the neighbouring windows' copies of the shared tiles are
// served by L2.  The coarse values of the up leg (a few doubles per thread at a thread-dependent address) follow
// through per-thread cp.async into the thread's own shared-memory slots.  ~52 KB of shared memory per CTA: one
// operator stage suffices because the operator moves to registers at the start of a window and the stage is
// refilled right after (one block-wide barrier; folding the refill into the leg's first exchange barrier was
// measured slower - the longer live ranges spill).  Arithmetic, order and emitted values are those of f_down / f_up
// (down_body / up_body): bit-identical.  Used on levels of at least leg_pipeline_min elements per rank: below ~2^19
// the two ordinary stream dependencies around a persistent leg (next paragraph) cost more than the pipeline gains.  Slab edges: thread 0 waits for the neighbour's flags before the first copy of a window that
// touches an edge (the spin of halo_leg_wait), the edge owners push as in f_down / f_up.
// The persistent legs are launched as ordinary stream successors, not as programmatic dependents: an early
// launch places their CTAs on SMs that still run the predecessor's last wave under ITS shared-memory carve-out,
// fewer than pipe_min_blocks fit, the SM can never be reconfigured while a persistent CTA lives on it, and the
// CTAs that found no place run as a second wave; and a programmatic successor of a persistent leg starts on SMs
// that still hold persistent CTAs, inherits their maximal shared-memory carve-out (no L1 to speak of) and hands it
// down the whole PDL chain, because no SM ever drains (measured on T: 17.0 instead of 15.6 ms per cycle).  So the
// legs before and after a persistent leg are separated by ordinary stream dependencies (fused_prev_persistent).
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// A bulk copy that never completes (a bad address would fault instead) must not hang the GPU: give up after ~2 s.
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity))
        if (clock64() - t0 > 4000000000LL) __trap();
}

template <int M, int B, int ST>
struct PipeStage {
    static constexpr int NT = B / AMG1D_TILE + 1;      // element tiles a window of B elements can touch
    static constexpr int NR = OpShape<M, ST>::O_DV;    // tile rows of A_lo, A_di, A_up (contiguous at the tile's start)
    alignas(128) double op[NT][NR][AMG1D_TILE];
    alignas(16) double bv[B * M];
    alignas(16) double xv[B * M];
    alignas(8) unsigned long long bar;
};

// Warp 0 (all 32 lanes call this): the bulk copies of the window that starts at local element e0 - parts & 1: its
// operator tiles, parts & 2: its b / x slices followed by the ONE arrival that arms the barrier with the bytes of
// both parts (the prologue issues the operator before the dependency wait and the vectors after it).  A window that
// lies inside the slab needs every tile and both slices whole: lanes 0 .. NT + 1 issue one copy each, side by side,
// and lane 0 arrives with the constant byte count - the common case costs the warp one copy's worth of
// instructions.  Windows at the ends of the slab are clipped by lane 0 alone.
template <int M, int B, int ST>
__device__ __forceinline__ void pipe_issue_window(PipeStage<M, B, ST>& st, const double* __restrict__ mat,
                                                  const double* __restrict__ b, const double* __restrict__ xin,
                                                  int64_t e0, int64_t lo, int64_t hi, int parts) {
    using PS = PipeStage<M, B, ST>;
    constexpr int K = OpShape<M, ST>::O_DV + M * M;
    constexpr unsigned TB = PS::NR * AMG1D_TILE * 8, VB = B * M * 8;
    const int lane = threadIdx.x;
    const int64_t t0 = e0 >> 5, t1 = (e0 + B - 1) >> 5;
    if (e0 >= lo && e0 + B <= hi && t1 - t0 == PS::NT - 1) {        // warp-uniform
        if (lane < PS::NT) {
            if (parts & 1) bulk_g2s(&st.op[lane][0][0], mat + (t0 + lane) * (int64_t)(K * AMG1D_TILE), TB, &st.bar);
        } else if (lane == PS::NT) {
            if (parts & 2) bulk_g2s(st.bv, b + e0 * M, VB, &st.bar);
        } else if (lane == PS::NT + 1) {
            if ((parts & 2) && xin) bulk_g2s(st.xv, xin + e0 * M, VB, &st.bar);
        }
        if (lane == 0 && (parts & 2)) mbar_arrive_expect_tx(&st.bar, PS::NT * TB + (xin ? 2 * VB : VB));
        return;
    }
    if (lane != 0) return;
    const int64_t tlo = lo >> 5, thi = (hi - 1) >> 5;
    unsigned bytes = 0;
#pragma unroll
    for (int j = 0; j < PS::NT; ++j) {
        const int64_t tj = t0 + j;
        if (tj <= t1 && tj >= tlo && tj <= thi) {
            if (parts & 1) bulk_g2s(&st.op[j][0][0], mat + tj * (int64_t)(K * AMG1D_TILE), TB, &st.bar);
            bytes += TB;
        }
    }
    if (!(parts & 2)) return;
    const int64_t a = e0 > lo ? e0 : lo, z = e0 + B < hi ? e0 + B : hi;
    if (z > a) {
        const unsigned vb = (unsigned)(z - a) * (M * 8);
        bulk_g2s(st.bv + (a - e0) * M, b + a * M, vb, &st.bar);
        bytes += vb;
        if (xin) {
            bulk_g2s(st.xv + (a - e0) * M, xin + a * M, vb, &st.bar);
            bytes += vb;
        }
    }
    mbar_arrive_expect_tx(&st.bar, bytes);
}

// The window's operator from the stage into registers; the diagonal block is read twice - once as A.di and once as
// the start of the in-place inversion A.dv (16 shared-memory loads instead of 32 register moves).  GUARD = false: the
// whole window lies inside the slab (CTA-uniform test by the caller), no thread needs the zero fill.
template <int M, int B, int ST, bool GUARD>
__device__ __forceinline__ void pipe_take_op(const PipeStage<M, B, ST>& st, int64_t e0, int64_t e, bool active,
                                             RegOpDv<M, ST>& A) {
    using S = OpShape<M, ST>;
    if (!GUARD || active) {
        const double* T = &st.op[(int)((e >> 5) - (e0 >> 5))][0][(int)(e & 31)];
#pragma unroll
        for (int k = 0; k < S::NO; ++k) A.lo[k] = T[k * AMG1D_TILE];
#pragma unroll
        for (int k = 0; k < M * M; ++k) A.di[k] = T[(S::O_DI + k) * AMG1D_TILE];
#pragma unroll
        for (int k = 0; k < S::NO; ++k) A.up[k] = T[(S::O_UP + k) * AMG1D_TILE];
#pragma unroll
        for (int k = 0; k < M * M; ++k) A.dv[k] = T[(S::O_DI + k) * AMG1D_TILE];
    } else {
#pragma unroll
        for (int k = 0; k < S::NO; ++k) { A.lo[k] = 0.0; A.up[k] = 0.0; }
#pragma unroll
        for (int k = 0; k < M * M; ++k) { A.di[k] = 0.0; A.dv[k] = 0.0; }
    }
}

template <int M, int ST>
__device__ __forceinline__ void pipe_invert(RegOpDv<M, ST>& A, bool active, int rec) {
    if (active) {
        if ((rec & 3) == 2) reg_invert<M, false>(A.dv); else reg_invert<M, true>(A.dv);
    }
}

// persistent CTAs per SM: 4 x 4 blocks keep 40 operator doubles per thread (128 registers, 4 CTAs of ~52 KB), 2 x 2
// blocks 12 - 16 (64 registers, 8 CTAs of ~26 KB)
constexpr int pipe_min_blocks(int m) { return m >= 4 ? 4 : 8; }
#define PIPE_MINB(M) pipe_min_blocks(M)

template <int M, int MC, int B, int ST>
struct PipeDownSmem {
    PipeStage<M, B, ST> st;
    Exchange<M, B> ex;
    double rs[M][B + 8];
};

template <int M, int MC, int B, int ST, int NSW, bool SINGLE>
__global__ void __launch_bounds__(B, PIPE_MINB(M))
f_down_pp(const double* __restrict__ mat, int ilo, int iup, const double* __restrict__ b,
          const double* __restrict__ xin, double* __restrict__ xout, const double* __restrict__ P0,
          const double* __restrict__ P1, TransferMap tm, double* __restrict__ rc, int64_t n, double alpha,
          int nsweep, int zero_guess, WinIdx wi, Slab sl, int rec, const __grid_constant__ HaloLeg hl, int64_t n_win) {
    extern __shared__ __align__(128) unsigned char pipe_smem[];
    PipeDownSmem<M, MC, B, ST>& S = *reinterpret_cast<PipeDownSmem<M, MC, B, ST>*>(pipe_smem);
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t lo = -(int64_t)sl.gl, hi = n + sl.gr;
    const double* xsrc = zero_guess ? nullptr : xin;
    if (t == 0) mbar_init(&S.st.bar, 1);
    exch_init<M, B>(S.ex);
    __syncthreads();
    int64_t win = blockIdx.x;
    {
        const int64_t e0 = win * wi.out - wi.halo;
        if (t < 32) pipe_issue_window<M, B, ST>(S.st, mat, b, xsrc, e0, lo, hi, 1);    // operator: independent of earlier kernels
        pdl_wait();
        halo_leg_wait(hl, sl.gl > 0 && e0 < 0, sl.gr > 0 && e0 + B > n);
        if (t < 32) {
            fence_proxy_async();
            pipe_issue_window<M, B, ST>(S.st, mat, b, xsrc, e0, lo, hi, 2);
        }
    }
    unsigned parity = 0;
    for (; win < n_win; win += gridDim.x) {
        const int64_t e0 = win * wi.out - wi.halo, e = e0 + t;
        const bool active = e >= lo && e < hi;
        RegOpDv<M, ST> A;
        double bb[M], xc[M];
        mbar_wait(&S.st.bar, parity);
        parity ^= 1;
        if (e0 >= lo && e0 + B <= hi) {                          // CTA-uniform: the whole window is inside the slab
            pipe_take_op<M, B, ST, false>(S.st, e0, e, true, A);
            load_vec<M>(&S.st.bv[t * M], bb);
            if (zero_guess) {
#pragma unroll
                for (int i = 0; i < M; ++i) xc[i] = 0.0;
            } else {
                load_vec<M>(&S.st.xv[t * M], xc);
            }
        } else {
            pipe_take_op<M, B, ST, true>(S.st, e0, e, active, A);
            if (active) {
                load_vec<M>(&S.st.bv[t * M], bb);
                if (zero_guess) {
#pragma unroll
                    for (int i = 0; i < M; ++i) xc[i] = 0.0;
                } else {
                    load_vec<M>(&S.st.xv[t * M], xc);
                }
            } else {
#pragma unroll
                for (int i = 0; i < M; ++i) { bb[i] = 0.0; xc[i] = 0.0; }
            }
        }
        // once every thread has taken its share of the stage: refill it for the next window
        const int64_t wn = win + gridDim.x;
        auto refill = [&]() {
            if (wn < n_win) {                                    // CTA-uniform
                const int64_t en = wn * wi.out - wi.halo;
                halo_leg_wait(hl, sl.gl > 0 && en < 0, sl.gr > 0 && en + B > n);
                if (t < 32) {
                    fence_proxy_async();
                    pipe_issue_window<M, B, ST>(S.st, mat, b, xsrc, en, lo, hi, 3);
                }
            }
        };
        __syncthreads();
        refill();
        pipe_invert<M, ST>(A, active, rec);
        down_body<M, MC, B, ST, false, RegOpDv<M, ST>, NSW, SINGLE>(A, nullptr, S.ex, S.rs, e, win, bb, xc, ilo, iup, xout, P0,
                                                                     P1, tm, rc, n, alpha, nsweep, zero_guess, wi, sl, hl);
    }
}

template <int M, int MC, int B, int ST>
struct PipeUpSmem {
    PipeStage<M, B, ST> st;
    Exchange<M, B> ex;
    double cs[2 * MC][B];        // coarse values of the thread's parent(s), filled by the thread's own cp.async
};

// all threads: the coarse values window thread t of window `win` needs, into its own slots cs[.][t]
template <int M, int MC, int B>
__device__ __forceinline__ void pipe_issue_coarse(double (*cs)[B], const double* __restrict__ xcoarse, bool two,
                                                  const TransferMap& tm, const WinIdx& wi, const Slab& sl, int64_t win,
                                                  bool active) {
    const int t = threadIdx.x;
    if (active) {
        int kdiv, kmod;
        small_divmod(wi.qmod0 + t, tm.ratio, &kdiv, &kmod);
        const int64_t par = win * wi.opr + wi.qdiv0 + kdiv + tm.base;     // == tm.par(global element)
        const double* c0 = xcoarse + (par - sl.c_off) * MC;
#pragma unroll
        for (int j = 0; j < MC; ++j) cp_async8(&cs[j][t], c0 + j);
        if (two) {
#pragma unroll
            for (int j = 0; j < MC; ++j) cp_async8(&cs[MC + j][t], c0 + MC + j);
        }
    }
    cp_async_commit();
}

template <int M, int MC, int B, int ST, int NSW>
__global__ void __launch_bounds__(B, PIPE_MINB(M))
f_up_pp(const double* __restrict__ mat, int ilo, int iup, const double* __restrict__ b,
        const double* __restrict__ xin, double* __restrict__ xout, const double* __restrict__ P0,
        const double* __restrict__ P1, TransferMap tm, const double* __restrict__ xcoarse, int64_t n,
        double alpha, int nsweep, WinIdx wi, double* __restrict__ partial, Slab sl, int rec,
        const __grid_constant__ HaloLeg hl, int64_t n_win) {
    extern __shared__ __align__(128) unsigned char pipe_smem[];
    PipeUpSmem<M, MC, B, ST>& S = *reinterpret_cast<PipeUpSmem<M, MC, B, ST>*>(pipe_smem);
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t lo = -(int64_t)sl.gl, hi = n + sl.gr;
    if (t == 0) mbar_init(&S.st.bar, 1);
    exch_init<M, B>(S.ex);
    __syncthreads();
    int64_t win = blockIdx.x;
    {
        const int64_t e0 = win * wi.out - wi.halo;
        if (t < 32) pipe_issue_window<M, B, ST>(S.st, mat, b, xin, e0, lo, hi, 1);     // operator: independent of earlier kernels
        pdl_wait();
        halo_leg_wait(hl, sl.gl > 0 && e0 < tm.ratio + 1, sl.gr > 0 && e0 + B + tm.ratio + 1 > n);
        if (t < 32) {
            fence_proxy_async();
            pipe_issue_window<M, B, ST>(S.st, mat, b, xin, e0, lo, hi, 2);
        }
        pipe_issue_coarse<M, MC, B>(S.cs, xcoarse, P1 != nullptr, tm, wi, sl, win, e0 + t >= lo && e0 + t < hi);
    }
    unsigned parity = 0;
    for (; win < n_win; win += gridDim.x) {
        const int64_t e0 = win * wi.out - wi.halo, e = e0 + t;
        const bool active = e >= lo && e < hi;
        RegOpDv<M, ST> A;
        double bb[M], xc[M];
        mbar_wait(&S.st.bar, parity);
        parity ^= 1;
        if (e0 >= lo && e0 + B <= hi) pipe_take_op<M, B, ST, false>(S.st, e0, e, true, A);     // CTA-uniform
        else pipe_take_op<M, B, ST, true>(S.st, e0, e, active, A);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        if (active) {
            load_vec<M>(&S.st.bv[t * M], bb);
            load_vec<M>(&S.st.xv[t * M], xc);
            double c0[MC], c1[MC];
#pragma unroll
            for (int j = 0; j < MC; ++j) { c0[j] = S.cs[j][t]; c1[j] = P1 ? S.cs[MC + j][t] : 0.0; }
            const int64_t pb = win_blk(tm, wi, e + sl.e_off, t) * (M * MC);
            up_correct<M, MC>(xc, P0, P1, pb, c0, c1);
        } else {
#pragma unroll
            for (int i = 0; i < M; ++i) { bb[i] = 0.0; xc[i] = 0.0; }
        }
        // once every thread has taken its share of the stage: refill it for the next window
        const int64_t wn = win + gridDim.x;
        auto refill = [&]() {
            if (wn < n_win) {                                    // CTA-uniform
                const int64_t en = wn * wi.out - wi.halo;
                halo_leg_wait(hl, sl.gl > 0 && en < tm.ratio + 1, sl.gr > 0 && en + B + tm.ratio + 1 > n);
                if (t < 32) {
                    fence_proxy_async();
                    pipe_issue_window<M, B, ST>(S.st, mat, b, xin, en, lo, hi, 3);
                }
                pipe_issue_coarse<M, MC, B>(S.cs, xcoarse, P1 != nullptr, tm, wi, sl, wn, en + t >= lo && en + t < hi);
            }
        };
        __syncthreads();
        refill();
        pipe_invert<M, ST>(A, active, rec);
        up_body<M, MC, B, ST, false, RegOpDv<M, ST>, NSW>(A, nullptr, S.ex, e, win, bb, xc, ilo, iup, xout, n, alpha, nsweep,
                                                           wi, partial, hl);
    }
}

inline bool fused_has_pp(int m, int mc, int st, int diag) {
    return !diag && ((m == 4 && st == AMG1D_ST_COLROW && (mc == 2 || mc == 3)) || (m == 2 && mc == 2 && st != AMG1D_ST_ROWCOL));
}

// persistent grid of the pipelined legs: pipe_min_blocks(m) CTAs per SM of the current device; the dynamic
// shared-memory limit of the kernels is raised once per device context (pipe_configure_all, at amg1d_finalize)
inline int pipe_sm_count() {
    static int sms[64] = {0};                // per device ordinal
    int dev = 0;
    cudaGetDevice(&dev);
    const int slot = (dev >= 0 && dev < 64) ? dev : 0;
    if (!sms[slot]) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        sms[slot] = v;
    }
    return sms[slot];
}
template <class KERN>
inline cudaError_t pipe_configure(KERN kern, size_t smem) {
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}
// once per device context, outside stream capture (amg1d_finalize): the pipelined legs need > 48 KB per CTA
inline cudaError_t pipe_configure_all() {
    cudaError_t e = cudaSuccess;
#define PP(MM, MCC, SS)                                                                                            \
    if (e == cudaSuccess) e = pipe_configure(f_down_pp<MM, MCC, FUSED_B, SS, 0, false>, sizeof(PipeDownSmem<MM, MCC, FUSED_B, SS>)); \
    if (e == cudaSuccess) e = pipe_configure(f_down_pp<MM, MCC, FUSED_B, SS, 3, false>, sizeof(PipeDownSmem<MM, MCC, FUSED_B, SS>)); \
    if (e == cudaSuccess) e = pipe_configure(f_down_pp<MM, MCC, FUSED_B, SS, 0, true>, sizeof(PipeDownSmem<MM, MCC, FUSED_B, SS>)); \
    if (e == cudaSuccess) e = pipe_configure(f_down_pp<MM, MCC, FUSED_B, SS, 3, true>, sizeof(PipeDownSmem<MM, MCC, FUSED_B, SS>)); \
    if (e == cudaSuccess) e = pipe_configure(f_up_pp<MM, MCC, FUSED_B, SS, 0>, sizeof(PipeUpSmem<MM, MCC, FUSED_B, SS>)); \
    if (e == cudaSuccess) e = pipe_configure(f_up_pp<MM, MCC, FUSED_B, SS, 3>, sizeof(PipeUpSmem<MM, MCC, FUSED_B, SS>));
    PP(4, 2, 1) PP(4, 3, 1) PP(2, 2, 0) PP(2, 2, 1) PP(2, 2, 3)
#undef PP
    return e;
}

// f_up with constant-bank operands for the interior CTAs of a pattern level (see f_down_c)
template <int M, int MC, int B, int ST, bool DIAG>
__global__ void FUSED_C_BOUNDS(M)
f_up_c(const __grid_constant__ ParamOp<M, ST, DIAG> pk, PatOp po, int ilo, int iup, const double* __restrict__ b,
       const double* __restrict__ xin, double* __restrict__ xout, const double* __restrict__ P0,
       const double* __restrict__ P1, TransferMap tm, const double* __restrict__ xcoarse, int64_t n,
       double alpha, int nsweep, WinIdx wi, double* __restrict__ partial, Slab sl,
       const __grid_constant__ HaloLeg hl) {
    __shared__ Exchange<M, B> ex;
    __shared__ double ds[DIAG ? M : M * M][B];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + t;
    exch_init<M, B>(ex);
    if (window_is_interior(po, wi, sl, n, B)) {
        up_leg<M, MC, B, ST, DIAG>(pk, nullptr, ex, e, true, ilo, iup, b, xin, xout, P0, P1, tm, xcoarse, n, alpha,
                                   nsweep, wi, partial, sl, hl);
    } else {
        const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
        RegOp<M, ST> A;
        load_blocks<M, B, ST, DIAG>(nullptr, po, e, e + sl.e_off, active, A, ds);
        up_leg<M, MC, B, ST, DIAG>(A, &ds[0][t], ex, e, active, ilo, iup, b, xin, xout, P0, P1, tm, xcoarse, n, alpha,
                                   nsweep, wi, partial, sl, hl);
    }
}

// residual + restriction, streaming (single-parent transfers; used when the multi-sweep kernel does
// not apply)
template <int M, int MC, int B, int ST>
__global__ void __launch_bounds__(B)
f_residual_restrict(const double* __restrict__ mat, int K, int ilo, int iup, const double* __restrict__ b,
                    const double* __restrict__ x, const double* __restrict__ P0, TransferMap tm,
                    double* __restrict__ rc, int64_t n, int out) {
    __shared__ double rs[M][B + 8];
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * out + t;
    const bool active = e < n && t < out;
    double r[M];
    if (e < n) {
        const double* T = mat + (e >> 5) * (int64_t)K * AMG1D_TILE + (e & 31);
        double xl[M], xc[M], xr[M], y[M], bb[M];
        load_vec<M>(b + e * M, bb);
        load_vec<M>(x + e * M, xc);
        load_neighbours<M, ST>(x, e, ilo, iup, xl, xr);
        stream_Ax<M, ST>(T, ilo, iup, xl, xc, xr, y);
#pragma unroll
        for (int i = 0; i < M; ++i) r[i] = bb[i] - y[i];
    } else {
#pragma unroll
        for (int i = 0; i < M; ++i) r[i] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < M; ++i) rs[i][t] = r[i];
    __syncthreads();
    const int ratio = tm.ratio;
    if (active && (e % ratio) == 0) {
        double acc[MC];
#pragma unroll
        for (int j = 0; j < MC; ++j) acc[j] = 0.0;
        for (int c = 0; c < ratio && e + c < n; ++c) {
            const double* P = P0 + tm.blk(e + c) * (M * MC);
#pragma unroll
            for (int j = 0; j < MC; ++j)
#pragma unroll
                for (int i = 0; i < M; ++i) acc[j] = fma(P[j * M + i], rs[i][t + c], acc[j]);
        }
        const int64_t Kc = e / ratio;
#pragma unroll
        for (int j = 0; j < MC; ++j) rc[Kc * MC + j] = acc[j];
    }
}

// ---- single-CTA coarse tail ----------------------------------------------------------------------------
// The sub-V-cycle of the coarse levels (at most TAIL_B elements each, one block size M, block
// smoothers, single-parent closed-form transfers) in ONE CTA that works entirely out of shared memory:
//   * at entry every tail level's operator tiles (and transfer blocks) are copied global -> shared with
//     cp.async - BEFORE the programmatic-dependency wait, so under PDL this prefetch overlaps the last
//     f_down of the levels above;
//   * one thread per element; per leg the element's blocks go shared -> registers, iterates are
//     exchanged through shared memory, the right-hand sides and pre-smoothed iterates of all tail
//     levels stay in shared memory between the down and the up leg;
//   * the only dependent global traffic is the first level's right-hand side in and its iterate out.
// It replaces two launches per level (each a few microseconds of latency for a few hundred bytes of
// work) by one launch.  Arithmetic per element is that of f_down / f_up / g_coarse_solve, so the
// results are bit-identical to the per-level kernels.
#define TAIL_MAXL 16
struct TailLevel {
    MatDesc md;
    const double* mat;
    int64_t n;
    double* x;          // iterate buffer 0 of the level (element 0); written for the first tail level only
    double* b;          // right-hand side; read for the first tail level only
    TransferMap tm;     // transfer to the next tail level (unused on the last one)
    const double* P0;
    int op_off, op_len; // this level's tiles inside the shared operator area (doubles)
    int vec_off;        // this level's vectors inside the shared b / x areas (doubles)
    int p_off, p_len;   // this level's transfer blocks inside the shared P area (doubles)
};

// shared-memory carve-up of f_tail (in doubles, after the descriptors)
struct TailPlan {
    int n_desc, ex, rs, cw, ops, bvec, xvec, pblk, total;   // offsets; total = size in doubles
};
inline TailPlan tail_plan(int m, int op_total, int vec_total, int p_total) {
    TailPlan p;
    int o = 0;
    p.n_desc = o; o += (int)((TAIL_MAXL * sizeof(TailLevel) + 7) / 8);
    p.ex = o; o += 2 * m * (TAIL_B + 2);
    p.rs = o; o += m * (TAIL_B + 8);
    p.cw = o; o += 64;
    o = (o + 1) & ~1;                                   // 16-byte alignment for cp.async
    p.ops = o; o += op_total;
    p.pblk = o; o += (p_total + 1) & ~1;
    p.bvec = o; o += vec_total;
    p.xvec = o; o += vec_total;
    p.total = o;
    return p;
}

__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gmem_src) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem_src) : "memory");
}

// Dense register copy of the element's operator whatever the level's structure class (entries that
// the class does not store are exact zeros or, ST_REPEAT, copies of the stored column / row, so the
// dense chains give identical results).  T points at
// the element's lane of its (shared-memory) tile.
template <int M>
__device__ __forceinline__ void tail_load(const MatDesc& d, const double* T, bool active, RegOp<M, 0>& A) {
    if (active) {
#pragma unroll
        for (int k = 0; k < M * M; ++k) A.di[k] = T[(d.o_di + k) * AMG1D_TILE];
        if (d.st == AMG1D_ST_DENSE) {
#pragma unroll
            for (int k = 0; k < M * M; ++k) { A.lo[k] = T[k * AMG1D_TILE]; A.up[k] = T[(d.o_up + k) * AMG1D_TILE]; }
        } else if (d.st == AMG1D_ST_REPEAT) {
#pragma unroll
            for (int j = 0; j < M; ++j)
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    A.lo[j * M + i] = T[i * AMG1D_TILE];
                    A.up[j * M + i] = T[(d.o_up + j) * AMG1D_TILE];
                }
        } else {
#pragma unroll
            for (int j = 0; j < M; ++j)
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    if (d.st == AMG1D_ST_COLROW) {
                        A.lo[j * M + i] = (j == d.ilo) ? T[i * AMG1D_TILE] : 0.0;
                        A.up[j * M + i] = (i == d.iup) ? T[(d.o_up + j) * AMG1D_TILE] : 0.0;
                    } else {
                        A.lo[j * M + i] = (i == d.ilo) ? T[j * AMG1D_TILE] : 0.0;
                        A.up[j * M + i] = (j == d.iup) ? T[(d.o_up + i) * AMG1D_TILE] : 0.0;
                    }
                }
        }
    } else {
#pragma unroll
        for (int k = 0; k < M * M; ++k) { A.lo[k] = 0.0; A.di[k] = 0.0; A.up[k] = 0.0; }
    }
}

// one damped block-Jacobi sweep with Dinv read from the element's shared tile (inactive threads: x stays 0)
template <int M>
__device__ __forceinline__ void tail_sweep(const RegOp<M, 0>& A, const double* dcol, bool active,
                                           const double (&bb)[M], const double (&xl)[M], double (&xc)[M],
                                           const double (&xr)[M], double alpha, bool zero_guess) {
    if (active) reg_sweep<M, 0, false, AMG1D_TILE>(A, 0, 0, dcol, bb, xl, xc, xr, alpha, zero_guess);
}

template <int M>
__global__ void __launch_bounds__(TAIL_B, 1)
f_tail(const TailLevel* __restrict__ lv, int nl, const double* __restrict__ fac, int nPre, int nPost,
       double alpha, TailPlan pl) {
    extern __shared__ __align__(16) double tsm[];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    TailLevel* sd = reinterpret_cast<TailLevel*>(tsm + pl.n_desc);
    Exchange<M, TAIL_B>& ex = *reinterpret_cast<Exchange<M, TAIL_B>*>(tsm + pl.ex);
    double (*rs)[TAIL_B + 8] = reinterpret_cast<double (*)[TAIL_B + 8]>(tsm + pl.rs);
    double* cw = tsm + pl.cw;
    double* ops = tsm + pl.ops;
    double* pblk = tsm + pl.pblk;
    double* bvec = tsm + pl.bvec;
    double* xvec = tsm + pl.xvec;
    // descriptors, then every level's operator tiles and transfer blocks: read-only data, fetched before
    // the dependency wait
    for (int i = t; i < (int)(nl * sizeof(TailLevel) / 8); i += TAIL_B)
        (tsm + pl.n_desc)[i] = reinterpret_cast<const double*>(lv)[i];
    exch_init<M, TAIL_B>(ex);
    __syncthreads();
    for (int l = 0; l < nl; ++l) {
        const TailLevel& L = sd[l];
        for (int i = 2 * t; i < L.op_len; i += 2 * TAIL_B) cp_async16(ops + L.op_off + i, L.mat + i);
        for (int i = t; i < L.p_len; i += TAIL_B) cp_async8(pblk + L.p_off + i, L.P0 + i);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    pdl_wait();
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    RegOp<M, 0> A;
    double bb[M], xc[M], xl[M], xr[M];
    int buf = 0;
    // ---- down: zero guess, nPre sweeps, residual, restriction ----
    for (int l = 0; l < nl - 1; ++l) {
        const TailLevel& L = sd[l];
        const bool active = t < L.n;
        const double* T = ops + L.op_off + (t >> 5) * (L.md.K * AMG1D_TILE) + (t & 31);
        const double* dcol = T + L.md.o_dv * AMG1D_TILE;
        double* bl = bvec + L.vec_off;
        tail_load<M>(L.md, T, active, A);
#pragma unroll
        for (int i = 0; i < M; ++i) {
            bb[i] = active ? (l == 0 ? L.b[t * M + i] : bl[t * M + i]) : 0.0;
            xc[i] = 0.0;
        }
        if (l == 0 && active) {
#pragma unroll
            for (int i = 0; i < M; ++i) bl[t * M + i] = bb[i];       // kept for the up leg
        }
        for (int s = 0; s < nPre; ++s) {
            if (s > 0) {
                exchange<M, TAIL_B, 0>(ex, buf, 0, 0, xc, xl, xr);
                buf ^= 1;
            }
            tail_sweep<M>(A, dcol, active, bb, xl, xc, xr, alpha, s == 0);
        }
        if (active) {
#pragma unroll
            for (int i = 0; i < M; ++i) xvec[L.vec_off + t * M + i] = xc[i];
        }
        exchange<M, TAIL_B, 0>(ex, buf, 0, 0, xc, xl, xr);
        buf ^= 1;
        double r[M];
        reg_residual<M, 0>(A, 0, 0, bb, xl, xc, xr, r);
#pragma unroll
        for (int i = 0; i < M; ++i) rs[i][t] = r[i];
        __syncthreads();
        const int ratio = L.tm.ratio;
        if (active && (t % ratio) == 0) {
            double acc[M];
#pragma unroll
            for (int j = 0; j < M; ++j) acc[j] = 0.0;
            for (int c = 0; c < ratio && t + c < L.n; ++c) {
                const double* P = pblk + L.p_off + L.tm.blk(t + c) * (M * M);
#pragma unroll
                for (int j = 0; j < M; ++j)
#pragma unroll
                    for (int i = 0; i < M; ++i) acc[j] = fma(P[j * M + i], rs[i][t + c], acc[j]);
            }
            double* bc = bvec + sd[l + 1].vec_off + (t / ratio) * M;
#pragma unroll
            for (int j = 0; j < M; ++j) bc[j] = acc[j];
        }
        __syncthreads();
    }
    // ---- coarsest level: block-Thomas substitution by one warp ----
    {
        const TailLevel& L = sd[nl - 1];
        if (t < 32) coarse_solve_warp(fac, M, L.n, bvec + L.vec_off, xvec + L.vec_off, cw, cw + 32);
        __syncthreads();
    }
    // ---- up: prolongation + correction, nPost sweeps ----
    for (int l = nl - 2; l >= 0; --l) {
        const TailLevel& L = sd[l];
        const bool active = t < L.n;
        const double* T = ops + L.op_off + (t >> 5) * (L.md.K * AMG1D_TILE) + (t & 31);
        const double* dcol = T + L.md.o_dv * AMG1D_TILE;
        tail_load<M>(L.md, T, active, A);
        if (active) {
            const double* P = pblk + L.p_off + L.tm.blk(t) * (M * M);
            const double* c0 = xvec + sd[l + 1].vec_off + (t / L.tm.ratio) * M;
            double y[M];
#pragma unroll
            for (int i = 0; i < M; ++i) {
                bb[i] = bvec[L.vec_off + t * M + i];
                xc[i] = xvec[L.vec_off + t * M + i];
                y[i] = 0.0;
            }
#pragma unroll
            for (int j = 0; j < M; ++j) {
                const double cj = c0[j];
#pragma unroll
                for (int i = 0; i < M; ++i) y[i] = fma(P[j * M + i], cj, y[i]);
            }
#pragma unroll
            for (int i = 0; i < M; ++i) xc[i] = xc[i] + y[i];
        } else {
#pragma unroll
            for (int i = 0; i < M; ++i) { bb[i] = 0.0; xc[i] = 0.0; }
        }
        for (int s = 0; s < nPost; ++s) {
            exchange<M, TAIL_B, 0>(ex, buf, 0, 0, xc, xl, xr);
            buf ^= 1;
            tail_sweep<M>(A, dcol, active, bb, xl, xc, xr, alpha, false);
        }
        if (active) {
#pragma unroll
            for (int i = 0; i < M; ++i) xvec[L.vec_off + t * M + i] = xc[i];
            if (l == 0) store_vec<M>(L.x + t * M, xc);
        }
        __syncthreads();
    }
}

// ---- host-side dispatch ---------------------------------------------------------------------------------
#define FUSED_FOR_M(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9)

// structure classes need m >= 2, and ST_COLROW the DG trace row (see FUSED_COLROW_IUP); ST_REPEAT is
// instantiated for block-Jacobi 2 x 2 levels only, the only ones amg1d.cu gives that class
inline bool fast_tier_ok(const MatDesc& d) {
    if (d.st == AMG1D_ST_DENSE) return true;
    if (d.m < 2) return false;
    return d.st != AMG1D_ST_COLROW || d.iup == FUSED_COLROW_IUP;
}

inline bool fused_sweep(const MatDesc& d, const double* mat, const double* b, const double* xin,
                        double* xout, int64_t n, double alpha, int zero_guess, cudaStream_t st) {
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (!fast_tier_ok(d)) return false;
    switch ((d.m * 2 + d.diag) * 4 + d.st) {
#define Y(MM, DG, SS)                                                                                     \
    case (MM * 2 + DG) * 4 + SS:                                                                          \
        f_sweep<MM, DG != 0, SS><<<grid, 256, 0, st>>>(mat, d.ilo, d.iup, b, xin, xout, n, alpha, zero_guess); \
        return true;
#define X(MM) Y(MM, 0, 0) Y(MM, 1, 0) Y(MM, 0, 1) Y(MM, 1, 1) Y(MM, 0, 2) Y(MM, 1, 2)
        FUSED_FOR_M(X) Y(2, 0, 3)
#undef X
#undef Y
        default: return false;
    }
}

inline bool fused_resnorm(const MatDesc& d, const double* mat, const double* b, const double* x,
                          int64_t n, double* partial, int64_t partial_cap, int* nblocks,
                          cudaStream_t st) {
    const int64_t grid = (n + 255) / 256;
    if (grid > partial_cap || !fast_tier_ok(d)) return false;
    *nblocks = (int)grid;
    switch (d.m * 4 + d.st) {
#define Y(MM, SS)                                                                                       \
    case MM * 4 + SS:                                                                                   \
        f_resnorm<MM, SS><<<(unsigned)grid, 256, 0, st>>>(mat, d.K, d.ilo, d.iup, b, x, n, partial);    \
        return true;
#define X(MM) Y(MM, 0) Y(MM, 1) Y(MM, 2)
        FUSED_FOR_M(X) Y(2, 3)
#undef X
#undef Y
        default: return false;
    }
}

inline bool fused_matvec_dot(const MatDesc& d, const double* mat, const double* x, double* y, int64_t n,
                             double* partial, int64_t partial_cap, int* nblocks, cudaStream_t st) {
    const int64_t grid = (n + 255) / 256;
    if (grid > partial_cap || !fast_tier_ok(d)) return false;
    *nblocks = (int)grid;
    switch (d.m * 4 + d.st) {
#define Y(MM, SS)                                                                                       \
    case MM * 4 + SS:                                                                                   \
        f_matvec_dot<MM, SS><<<(unsigned)grid, 256, 0, st>>>(mat, d.K, d.ilo, d.iup, x, y, n, partial); \
        return true;
#define X(MM) Y(MM, 0) Y(MM, 1) Y(MM, 2)
        FUSED_FOR_M(X) Y(2, 3)
#undef X
#undef Y
        default: return false;
    }
}

// (M, MC, ST, DIAG) combinations with a register-resident multi-sweep kernel:
//   block Jacobi, dense, DG-assembled and repeated column / row structure (DG / agglomerated levels);
//   point Jacobi on CG levels in group form (m = 1: CG p=1; m >= 2: ST_ROWCOL).
#define FUSED_COMBOS(X)                                                                              \
    X(1, 1, 0, false) X(2, 1, 0, false) X(2, 2, 0, false) X(3, 1, 0, false) X(3, 2, 0, false)         \
    X(4, 2, 0, false) X(4, 3, 0, false) X(5, 3, 0, false)                                             \
    X(2, 1, 1, false) X(2, 2, 1, false) X(3, 1, 1, false) X(3, 2, 1, false)                           \
    X(4, 2, 1, false) X(4, 3, 1, false) X(5, 3, 1, false)                                             \
    X(2, 1, 3, false) X(2, 2, 3, false)                                                               \
    X(1, 1, 0, true) X(1, 2, 0, true) X(2, 1, 2, true) X(3, 1, 2, true) X(4, 2, 2, true)

inline int fused_key(int m, int mc, int st, int diag) { return ((m * 16 + mc) * 4 + st) * 2 + (diag ? 1 : 0); }

// halo, elements emitted per CTA and the 32-bit index constants for a leg of nsweep sweeps
inline int64_t floordiv64(int64_t a, int64_t b) { int64_t q = a / b; return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q; }
inline WinIdx fused_window(int nsweep, const TransferMap& tm, bool wide, const Slab& sl, int window = FUSED_B) {
    WinIdx w;
    w.halo = nsweep + 1 + (wide ? tm.ratio : 0);
    w.out = ((window - 2 * w.halo) / tm.ratio) * tm.ratio;
    if (w.out < 1) w.out = 0;
    w.opr = w.out / tm.ratio;
    const int64_t q0 = sl.e_off + tm.shift - w.halo;
    w.qdiv0 = floordiv64(q0, tm.ratio);
    w.qmod0 = (int)(q0 - w.qdiv0 * tm.ratio);
    w.pmod0 = -1;
    if (tm.period > 0 && w.out % tm.period == 0) {
        const int64_t p0 = sl.e_off - w.halo - tm.n_head;
        const int64_t pm = p0 - floordiv64(p0, tm.period) * tm.period;            // floormod
        w.pmod0 = (int)pm + ((tm.ratio + tm.period - 1) / tm.period) * tm.period; // bias: thread offsets >= -ratio
    }
    return w;
}

// tm must be a closed-form map (parent == cp == nullptr); P1 != nullptr selects the two-parent form.
// n_cover: local elements whose coarse parents this rank may have to gather (n, or n + ratio when the
// right slab neighbour's first children contribute to this rank's last coarse element).
// Return value of fused_down / fused_up: FUSED_NA = no such kernel (the caller takes the streaming /
// generic path), FUSED_OK = launched, FUSED_ERR = the launch itself failed (*err holds the CUDA error;
// never silently papered over by a fall-back).
enum { FUSED_NA = 0, FUSED_OK = 1, FUSED_ERR = -1 };

inline int fused_down(const MatDesc& d, int mc, const TransferMap& tm, int nsweep, bool zero,
                       const double* mat, const PatOp& po, const double* b, const double* xin, double* xout,
                       const double* P0, const double* P1, double* rc, int64_t n, int64_t n_cover,
                       double alpha, const Slab& sl, cudaStream_t st, bool pdl, cudaError_t* err, int rec = 0,
                       const HaloLeg& hl = HaloLeg()) {
    const WinIdx w = fused_window(nsweep, tm, P1 != nullptr || tm.shift != 0 || tm.base != 0, sl);
    if (w.out < tm.ratio || w.out < FUSED_B / 2 || !fast_tier_ok(d)) return FUSED_NA;
    const unsigned grid = (unsigned)((n_cover + w.out - 1) / w.out);
    if ((rec & 16) && (rec & 3) && !po.tab && fused_has_pp(d.m, mc, d.st, d.diag) &&
        (((uintptr_t)b | (uintptr_t)xin | (uintptr_t)mat) & 15) == 0) {               // pipelined persistent leg
#define PP(MM, MCC, SS)                                                                                   \
        if (d.m == MM && mc == MCC && d.st == SS) {                                                       \
            const size_t smem = sizeof(PipeDownSmem<MM, MCC, FUSED_B, SS>);                               \
            const int64_t pg = std::min<int64_t>((int64_t)grid, (int64_t)pipe_sm_count() * PIPE_MINB(MM));    \
            const bool single = tm.ratio == 1 && P1 == nullptr;      /* one child per coarse element */ \
            *err = launch_fused(single ? (nsweep == 3 ? f_down_pp<MM, MCC, FUSED_B, SS, 3, true>                   \
                                                      : f_down_pp<MM, MCC, FUSED_B, SS, 0, true>)                  \
                                       : (nsweep == 3 ? f_down_pp<MM, MCC, FUSED_B, SS, 3, false>                  \
                                                      : f_down_pp<MM, MCC, FUSED_B, SS, 0, false>),                \
                                (unsigned)pg, FUSED_B, smem, st, false, mat, d.ilo,                       \
                                d.iup, b, xin, xout, P0, P1, tm, rc, n, alpha, nsweep, zero ? 1 : 0, w, sl, rec, hl, \
                                (int64_t)grid);                                                           \
            fused_prev_persistent() = true;                                                               \
            return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;                                            \
        }
        PP(4, 2, 1) PP(4, 3, 1) PP(2, 2, 0) PP(2, 2, 1) PP(2, 2, 3)
#undef PP
    }
    if ((rec & 8) && (rec & 3) && !po.tab && fused_has_dv(d.m, mc, d.st, d.diag)) {   // inverse in registers
#define DV(MM, MCC, SS)                                                                                   \
        if (d.m == MM && mc == MCC && d.st == SS) {                                                       \
            *err = launch_fused(f_down_dv<MM, MCC, FUSED_B, SS>, grid, FUSED_B, 0, st, pdl, mat, d.ilo, d.iup, b, xin, \
                                xout, P0, P1, tm, rc, n, alpha, nsweep, zero ? 1 : 0, w, sl, rec, hl);     \
            return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;                                            \
        }
        DV(4, 2, 1) DV(4, 3, 1) DV(2, 2, 0) DV(2, 2, 1) DV(2, 2, 3)
#undef DV
    }
    switch (fused_key(d.m, mc, d.st, d.diag)) {
#define X(MM, MCC, SS, DG)                                                                               \
    case ((MM * 16 + MCC) * 4 + SS) * 2 + (DG ? 1 : 0):                                                  \
        if (po.tab && po.host_interior && sizeof(ParamOp<MM, SS, DG>) == (size_t)d.K * 8) {                                                                \
            ParamOp<MM, SS, DG> pk;                                                                      \
            memcpy(&pk, po.host_interior, sizeof(pk));                                                   \
            *err = launch_fused(f_down_c<MM, MCC, FUSED_B, SS, DG>, grid, FUSED_B, 0, st, pdl, pk, po, d.ilo, \
                                d.iup, b, xin, xout, P0, P1, tm, rc, n, alpha, nsweep, zero ? 1 : 0, w, sl, hl); \
        } else                                                                                           \
        *err = launch_fused(f_down<MM, MCC, FUSED_B, SS, DG>, grid, FUSED_B, 0, st, pdl, mat, po, d.ilo, d.iup, \
                            b, xin, xout, P0, P1, tm, rc, n, alpha, nsweep, zero ? 1 : 0, w, sl,         \
                            ((!po.tab && !DG) ? (rec & 3) : 0), hl);                                  \
        return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;
        FUSED_COMBOS(X)
#undef X
        default: return FUSED_NA;
    }
}

inline int fused_up(const MatDesc& d, int mc, const TransferMap& tm, int nsweep, const double* mat,
                     const PatOp& po, const double* b, const double* xin, double* xout, const double* P0,
                     const double* P1, const double* xcoarse, int64_t n, double alpha, double* partial,
                     int64_t partial_cap, int* nblocks, const Slab& sl, cudaStream_t st, bool pdl,
                     cudaError_t* err, int rec = 0, const HaloLeg& hl = HaloLeg()) {
    const WinIdx w = fused_window(nsweep, tm, false, sl);
    if (w.out < tm.ratio || w.out < FUSED_B / 2 || !fast_tier_ok(d)) return FUSED_NA;
    const int64_t grid = (n + w.out - 1) / w.out;
    if (partial && grid > partial_cap) return FUSED_NA;
    if (nblocks) *nblocks = (int)grid;
    if ((rec & 16) && (rec & 3) && !po.tab && fused_has_pp(d.m, mc, d.st, d.diag) &&
        (((uintptr_t)b | (uintptr_t)xin | (uintptr_t)mat) & 15) == 0) {               // pipelined persistent leg
#define PP(MM, MCC, SS)                                                                                   \
        if (d.m == MM && mc == MCC && d.st == SS) {                                                       \
            const size_t smem = sizeof(PipeUpSmem<MM, MCC, FUSED_B, SS>);                                 \
            const int64_t pg = std::min<int64_t>(grid, (int64_t)pipe_sm_count() * PIPE_MINB(MM));             \
            *err = launch_fused(nsweep == 3 ? f_up_pp<MM, MCC, FUSED_B, SS, 3> : f_up_pp<MM, MCC, FUSED_B, SS, 0>, \
                                (unsigned)pg, FUSED_B, smem, st, false, mat, d.ilo,                       \
                                d.iup, b, xin, xout, P0, P1, tm, xcoarse, n, alpha, nsweep, w, partial, sl, rec, hl, \
                                grid);                                                                    \
            fused_prev_persistent() = true;                                                               \
            return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;                                            \
        }
        PP(4, 2, 1) PP(4, 3, 1) PP(2, 2, 0) PP(2, 2, 1) PP(2, 2, 3)
#undef PP
    }
    if ((rec & 8) && (rec & 3) && !po.tab && fused_has_dv(d.m, mc, d.st, d.diag)) {
#define DV(MM, MCC, SS)                                                                                   \
        if (d.m == MM && mc == MCC && d.st == SS) {                                                       \
            *err = launch_fused(f_up_dv<MM, MCC, FUSED_B, SS>, (unsigned)grid, FUSED_B, 0, st, pdl, mat, d.ilo, d.iup, b, \
                                xin, xout, P0, P1, tm, xcoarse, n, alpha, nsweep, w, partial, sl, rec, hl); \
            return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;                                            \
        }
        DV(4, 2, 1) DV(4, 3, 1) DV(2, 2, 0) DV(2, 2, 1) DV(2, 2, 3)
#undef DV
    }
    switch (fused_key(d.m, mc, d.st, d.diag)) {
#define X(MM, MCC, SS, DG)                                                                               \
    case ((MM * 16 + MCC) * 4 + SS) * 2 + (DG ? 1 : 0):                                                  \
        if (po.tab && po.host_interior && sizeof(ParamOp<MM, SS, DG>) == (size_t)d.K * 8) {                                                                \
            ParamOp<MM, SS, DG> pk;                                                                      \
            memcpy(&pk, po.host_interior, sizeof(pk));                                                   \
            *err = launch_fused(f_up_c<MM, MCC, FUSED_B, SS, DG>, (unsigned)grid, FUSED_B, 0, st, pdl, pk, po, \
                                d.ilo, d.iup, b, xin, xout, P0, P1, tm, xcoarse, n, alpha, nsweep, w, partial, sl, hl); \
        } else                                                                                           \
        *err = launch_fused(f_up<MM, MCC, FUSED_B, SS, DG>, (unsigned)grid, FUSED_B, 0, st, pdl, mat, po,    \
                            d.ilo, d.iup, b, xin, xout, P0, P1, tm, xcoarse, n, alpha, nsweep, w, partial, sl, \
                            ((!po.tab && !DG) ? (rec & 3) : 0), hl);                                  \
        return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;
        FUSED_COMBOS(X)
#undef X
        default: return FUSED_NA;
    }
}

// (M, MC) pairs of the streaming residual + restriction kernel (single-parent transfers)
#define FRR_PAIRS(X) X(1, 1) X(2, 1) X(2, 2) X(3, 1) X(3, 2) X(4, 2) X(4, 3) X(5, 3) X(9, 5) X(5, 2) X(9, 2)

inline bool fused_residual_restrict(const MatDesc& d, int mc, const TransferMap& tm, const double* mat,
                                    const double* b, const double* x, const double* P0, double* rc,
                                    int64_t n, cudaStream_t st) {
    const int out = (FUSED_B / tm.ratio) * tm.ratio;
    if (out < tm.ratio || !fast_tier_ok(d)) return false;
    const unsigned grid = (unsigned)((n + out - 1) / out);
    switch ((d.m * 16 + mc) * 4 + d.st) {
#define Y(MM, MCC, SS)                                                                                  \
    case (MM * 16 + MCC) * 4 + SS:                                                                      \
        f_residual_restrict<MM, MCC, FUSED_B, SS><<<grid, FUSED_B, 0, st>>>(mat, d.K, d.ilo, d.iup, b, x, P0, \
                                                                             tm, rc, n, out);           \
        return true;
#define X(MM, MCC) Y(MM, MCC, 0) Y(MM, MCC, 1) Y(MM, MCC, 2)
        FRR_PAIRS(X) Y(2, 1, 3) Y(2, 2, 3)
#undef X
#undef Y
        default: return false;
    }
}

// Block sizes with a single-CTA tail kernel.
inline bool tail_supported(int m) { return m == 1 || m == 2; }
#define TAIL_SMEM_MAX (227 * 1024)

template <int M>
inline cudaError_t tail_configure_t(size_t smem) {
    return cudaFuncSetAttribute(f_tail<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

// once per device context and tail shape, before the first launch (amg1d_finalize)
inline cudaError_t tail_configure(int m, size_t smem) {
    switch (m) {
        case 1: return tail_configure_t<1>(smem);
        case 2: return tail_configure_t<2>(smem);
        default: return cudaErrorInvalidValue;
    }
}

inline cudaError_t tail_launch(int m, const TailLevel* lv, int nl, const double* fac, int nPre, int nPost,
                               double alpha, const TailPlan& pl, cudaStream_t st, bool pdl) {
    const size_t smem = (size_t)pl.total * 8;
    switch (m) {
        case 1: return launch_fused(f_tail<1>, 1, TAIL_B, smem, st, pdl, lv, nl, fac, nPre, nPost, alpha, pl);
        case 2: return launch_fused(f_tail<2>, 1, TAIL_B, smem, st, pdl, lv, nl, fac, nPre, nPost, alpha, pl);
        default: return cudaErrorInvalidValue;
    }
}
