// Multi-column fused legs: one V-cycle leg for up to MULTI_MAX_COLS right-hand sides that reads the level's operator
// once.  The reference applies ldiv!(y, H, b) (src/solvers.jl:63-92) one vector at a time; a caller that preconditions
// a block of vectors (block Krylov methods, time steps, many loads on one operator) otherwise streams every level's
// operator from HBM once per vector.
//
//  f_down_multi / f_up_multi        operator from the element tiles or the pattern table into registers (Dinv into
//                                   shared memory, or inverted there in registers: rec), then the leg body of f_down /
//                                   f_up (down_leg / up_leg, kernels_fused.cuh) once per column
//  f_down_multi_dv / f_up_multi_dv  the same with the inverse kept in registers (load_blocks_dv): the form of the levels
//                                   whose single-column legs are f_*_dv or the pipelined f_*_pp
//  f_matvec_dot_multi               y_c = A x_c and the per-block partial sums of x_c . y_c of every column (the A p,
//                                   p . A p step of amg1d_dev_pcg_multi): f_matvec_dot with the operator read once
//
// Per column the arithmetic, its order and the window partition (fused_window) are those of the single-column leg, so
// every column's iterate, coarse right-hand side and per-window ||b - A x||^2 partial sums are bit-identical to a
// single-column cycle on that column.  Between columns the CTA synchronises: the exchange buffers restart at buf = 0
// and the restriction buffer rs is reused.  On a slab-sharded level the kernels read the ghost windows (Slab) as the
// single-column legs do; the slab edges travel between launches (NCCL, amg1d.cu), never from inside these kernels.
//
// Algorithmic bytes per element and column, k columns (FP64; Kop = doubles of the level's structure class, layout.cuh;
// coarse block size MC, ratio R; rec: the inverse is not read):
//   f_down_multi   8 (Kop / k + 3 M + MC / R)     against 8 (Kop + 3 M + MC / R) for f_down
//   f_up_multi     8 (Kop / k + 3 M + MC / R)     against 8 (Kop + 3 M + MC / R) for f_up
//   f_matvec_dot_multi  8 (Kop' / k + 2 M)          against 8 (Kop' + 2 M) for f_matvec_dot (Kop' = Kop without Dinv)
// (T level 0: Kop = 24, M = 4: 38 -> 24 / k + 14 doubles per element and column; matvec: Kop' = 24, 32 -> 24 / k + 8.)
#pragma once
#include "kernels_fused.cuh"

// Per-column vectors of one multi-column leg (device pointers at element 0 of the level).
struct MultiCols {
    const double* b[MULTI_MAX_COLS];    // right-hand side
    const double* xin[MULTI_MAX_COLS];  // incoming iterate
    double* xout[MULTI_MAX_COLS];       // outgoing iterate
    double* xc[MULTI_MAX_COLS];         // down: coarse right-hand side (written); up: coarse iterate (read)
    double* partial[MULTI_MAX_COLS];    // up: per-window ||b - A x||^2 of the column, or nullptr
};

// Resident CTAs per SM the register allocation aims for: those of f_down / f_up / f_*_dv, one step lower where the
// column loop (its counter, the per-column pointers) would push the capped kernels into spills - 4 x 4 compressed
// blocks 5 -> 4 CTAs (128 registers), 2 x 2 and 1 x 1 blocks 8 -> 6 (80 registers).
constexpr int multi_min_blocks(int m, int st) {
    return (m == 4 && st != AMG1D_ST_DENSE) ? 4 : m <= 2 ? 6 : fused_min_blocks(m, st);
}
constexpr int multi_dv_min_blocks(int m) { return m <= 2 ? 6 : fused_dv_min_blocks(m); }

// The element index as a value the compiler cannot see through: everything the up-leg body derives from it (vector and
// transfer-block addresses, parent indices) is recomputed per column instead of being hoisted out of the column loop
// and held in registers across it, which pushed the register-capped legs into spills.
__device__ __forceinline__ int64_t opaque(int64_t v) {
    asm volatile("" : "+l"(v));
    return v;
}

template <int M, int MC, int B, int ST, bool DIAG>
__global__ void __launch_bounds__(B, multi_min_blocks(M, ST))
f_down_multi(const double* __restrict__ mat, PatOp po, int ilo, int iup, const __grid_constant__ MultiCols cols,
             int k, const double* __restrict__ P0, const double* __restrict__ P1, TransferMap tm, int64_t n,
             double alpha, int nsweep, int zero_guess, WinIdx wi, Slab sl, int rec) {
    __shared__ Exchange<M, B> ex;
    __shared__ double rs[M][B + 8];
    __shared__ double ds[DIAG ? M : M * M][B];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + t;
    const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
    exch_init<M, B>(ex);
    RegOp<M, ST> A;
    load_blocks<M, B, ST, DIAG>(mat, po, e, e + sl.e_off, active, A, ds, rec != 0);
    recompute_dinv<M, B, ST, DIAG>(A, ds, active, rec);
    const HaloLeg hl{};
#pragma unroll 1
    for (int c = 0; c < k; ++c) {
        if (c) __syncthreads();
        down_leg<M, MC, B, ST, DIAG>(A, &ds[0][t], ex, rs, e, active, ilo, iup, cols.b[c], cols.xin[c], cols.xout[c],
                                     P0, P1, tm, cols.xc[c], n, alpha, nsweep, zero_guess, wi, sl, hl);
    }
}

template <int M, int MC, int B, int ST, bool DIAG>
__global__ void __launch_bounds__(B, multi_min_blocks(M, ST))
f_up_multi(const double* __restrict__ mat, PatOp po, int ilo, int iup, const __grid_constant__ MultiCols cols, int k,
           const double* __restrict__ P0, const double* __restrict__ P1, TransferMap tm, int64_t n, double alpha,
           int nsweep, WinIdx wi, Slab sl, int rec) {
    __shared__ Exchange<M, B> ex;
    __shared__ double ds[DIAG ? M : M * M][B];
    pdl_launch_dependents();
    const int t = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + t;
    const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
    exch_init<M, B>(ex);
    RegOp<M, ST> A;
    load_blocks<M, B, ST, DIAG>(mat, po, e, e + sl.e_off, active, A, ds, rec != 0);
    recompute_dinv<M, B, ST, DIAG>(A, ds, active, rec);
    const HaloLeg hl{};
#pragma unroll 1
    for (int c = 0; c < k; ++c) {
        if (c) __syncthreads();
        const int64_t ec = opaque(e);
        up_leg<M, MC, B, ST, DIAG>(A, &ds[0][t], ex, ec, active, ilo, iup, cols.b[c], cols.xin[c], cols.xout[c], P0, P1,
                                   tm, cols.xc[c], n, alpha, nsweep, wi, cols.partial[c], sl, hl);
    }
}

template <int M, int MC, int B, int ST>
__global__ void __launch_bounds__(B, multi_dv_min_blocks(M))
f_down_multi_dv(const double* __restrict__ mat, int ilo, int iup, const __grid_constant__ MultiCols cols, int k,
                const double* __restrict__ P0, const double* __restrict__ P1, TransferMap tm, int64_t n, double alpha,
                int nsweep, int zero_guess, WinIdx wi, Slab sl, int rec) {
    __shared__ Exchange<M, B> ex;
    __shared__ double rs[M][B + 8];
    pdl_launch_dependents();
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + threadIdx.x;
    const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
    exch_init<M, B>(ex);
    RegOpDv<M, ST> A;
    load_blocks_dv<M, ST>(mat, e, active, rec, A);
    const HaloLeg hl{};
#pragma unroll 1
    for (int c = 0; c < k; ++c) {
        if (c) __syncthreads();
        down_leg<M, MC, B, ST, false>(A, nullptr, ex, rs, e, active, ilo, iup, cols.b[c], cols.xin[c], cols.xout[c],
                                      P0, P1, tm, cols.xc[c], n, alpha, nsweep, zero_guess, wi, sl, hl);
    }
}

template <int M, int MC, int B, int ST>
__global__ void __launch_bounds__(B, multi_dv_min_blocks(M))
f_up_multi_dv(const double* __restrict__ mat, int ilo, int iup, const __grid_constant__ MultiCols cols, int k,
              const double* __restrict__ P0, const double* __restrict__ P1, TransferMap tm, int64_t n, double alpha,
              int nsweep, WinIdx wi, Slab sl, int rec) {
    __shared__ Exchange<M, B> ex;
    pdl_launch_dependents();
    const int64_t e = (int64_t)blockIdx.x * wi.out - wi.halo + threadIdx.x;
    const bool active = e >= -(int64_t)sl.gl && e < n + sl.gr;
    exch_init<M, B>(ex);
    RegOpDv<M, ST> A;
    load_blocks_dv<M, ST>(mat, e, active, rec, A);
    const HaloLeg hl{};
#pragma unroll 1
    for (int c = 0; c < k; ++c) {
        if (c) __syncthreads();
        const int64_t ec = opaque(e);
        up_leg<M, MC, B, ST, false>(A, nullptr, ex, ec, active, ilo, iup, cols.b[c], cols.xin[c], cols.xout[c], P0, P1,
                                    tm, cols.xc[c], n, alpha, nsweep, wi, cols.partial[c], sl, hl);
    }
}

// ---- host-side dispatch -----------------------------------------------------------------------------------------
// Same conditions as fused_down / fused_up (FUSED_NA exactly where they return it, so that the caller can run the
// single-column fall-back per column), same window, same grid.  rec as for fused_down: the register-inverse form
// where the single-column leg would be f_*_dv or f_*_pp (bit 3 or 4 with bits 0-1), f_*_multi otherwise; pattern-
// resident levels read the pattern table (pattern_resident = 1 and 2 alike: the same arithmetic as f_*_c).
inline bool multi_dv_form(const MatDesc& d, int mc, const PatOp& po, int rec) {
    return (rec & 24) && (rec & 3) && !po.tab && fused_has_dv(d.m, mc, d.st, d.diag);
}

inline bool fused_multi_available(const MatDesc& d, int mc) {
    if (!fast_tier_ok(d)) return false;
    switch (fused_key(d.m, mc, d.st, d.diag)) {
#define X(MM, MCC, SS, DG) case ((MM * 16 + MCC) * 4 + SS) * 2 + (DG ? 1 : 0): return true;
        FUSED_COMBOS(X)
#undef X
        default: return false;
    }
}

// n_cover as for fused_down: the local elements whose coarse parents this rank gathers (past n on a slab whose right
// neighbour's first children own coarse elements of this rank - two-parent transfers).
inline int fused_down_multi(const MatDesc& d, int mc, const TransferMap& tm, int nsweep, bool zero, const double* mat,
                            const PatOp& po, const MultiCols& cols, int k, const double* P0, const double* P1, int64_t n,
                            int64_t n_cover, double alpha, const Slab& sl, cudaStream_t st, bool pdl, cudaError_t* err,
                            int rec) {
    const WinIdx w = fused_window(nsweep, tm, P1 != nullptr || tm.shift != 0 || tm.base != 0, sl);
    if (w.out < tm.ratio || w.out < FUSED_B / 2 || !fast_tier_ok(d)) return FUSED_NA;
    const unsigned grid = (unsigned)((n_cover + w.out - 1) / w.out);
    if (multi_dv_form(d, mc, po, rec)) {
#define DV(MM, MCC, SS)                                                                                               \
        if (d.m == MM && mc == MCC && d.st == SS) {                                                                   \
            *err = launch_fused(f_down_multi_dv<MM, MCC, FUSED_B, SS>, grid, FUSED_B, 0, st, pdl, mat, d.ilo, d.iup, \
                                cols, k, P0, P1, tm, n, alpha, nsweep, zero ? 1 : 0, w, sl, rec);                    \
            return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;                                                        \
        }
        DV(4, 2, 1) DV(4, 3, 1) DV(2, 2, 0) DV(2, 2, 1) DV(2, 2, 3)
#undef DV
    }
    switch (fused_key(d.m, mc, d.st, d.diag)) {
#define X(MM, MCC, SS, DG)                                                                                            \
    case ((MM * 16 + MCC) * 4 + SS) * 2 + (DG ? 1 : 0):                                                               \
        *err = launch_fused(f_down_multi<MM, MCC, FUSED_B, SS, DG>, grid, FUSED_B, 0, st, pdl, mat, po, d.ilo, d.iup,  \
                            cols, k, P0, P1, tm, n, alpha, nsweep, zero ? 1 : 0, w, sl,                               \
                            ((!po.tab && !DG) ? (rec & 3) : 0));                                                      \
        return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;
        FUSED_COMBOS(X)
#undef X
        default: return FUSED_NA;
    }
}

// with_norm: every column's partial[] receives the per-window sums (nblocks of them, at most partial_cap)
inline int fused_up_multi(const MatDesc& d, int mc, const TransferMap& tm, int nsweep, const double* mat,
                          const PatOp& po, const MultiCols& cols, int k, const double* P0, const double* P1, int64_t n,
                          double alpha, bool with_norm, int64_t partial_cap, int* nblocks, const Slab& sl,
                          cudaStream_t st, bool pdl, cudaError_t* err, int rec) {
    const WinIdx w = fused_window(nsweep, tm, false, sl);
    if (w.out < tm.ratio || w.out < FUSED_B / 2 || !fast_tier_ok(d)) return FUSED_NA;
    const int64_t grid = (n + w.out - 1) / w.out;
    if (with_norm && grid > partial_cap) return FUSED_NA;
    if (nblocks) *nblocks = (int)grid;
    if (multi_dv_form(d, mc, po, rec)) {
#define DV(MM, MCC, SS)                                                                                               \
        if (d.m == MM && mc == MCC && d.st == SS) {                                                                   \
            *err = launch_fused(f_up_multi_dv<MM, MCC, FUSED_B, SS>, (unsigned)grid, FUSED_B, 0, st, pdl, mat, d.ilo, \
                                d.iup, cols, k, P0, P1, tm, n, alpha, nsweep, w, sl, rec);                           \
            return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;                                                        \
        }
        DV(4, 2, 1) DV(4, 3, 1) DV(2, 2, 0) DV(2, 2, 1) DV(2, 2, 3)
#undef DV
    }
    switch (fused_key(d.m, mc, d.st, d.diag)) {
#define X(MM, MCC, SS, DG)                                                                                            \
    case ((MM * 16 + MCC) * 4 + SS) * 2 + (DG ? 1 : 0):                                                               \
        *err = launch_fused(f_up_multi<MM, MCC, FUSED_B, SS, DG>, (unsigned)grid, FUSED_B, 0, st, pdl, mat, po,      \
                            d.ilo, d.iup, cols, k, P0, P1, tm, n, alpha, nsweep, w, sl,                               \
                            ((!po.tab && !DG) ? (rec & 3) : 0));                                                      \
        return *err == cudaSuccess ? FUSED_OK : FUSED_ERR;
        FUSED_COMBOS(X)
#undef X
        default: return FUSED_NA;
    }
}

// ---- y = A x with x . y for every column (the matvec of amg1d_dev_pcg_multi) ---------------------------------------
struct MatvecCols {
    const double* x[MULTI_MAX_COLS];
    double* y[MULTI_MAX_COLS];
    double* partial[MULTI_MAX_COLS];   // per-block x . y partial sums of the column, or nullptr
};

// Operators of at most this many doubles per element (A_lo, A_di, A_up: every 1 x 1 .. 4 x 4 class, 5 x 5 .. 7 x 7
// compressed) stay in registers across the column loop; larger ones are re-read from the element tile per column,
// columns after the first finding it in L1 / L2 (a register copy of a 9 x 9 dense operator would be 243 doubles).
template <int M, int ST>
struct MatvecOpInRegs { static constexpr bool value = 2 * OpShape<M, ST>::NO + M * M <= 64; };

// Grid and one element per thread as f_matvec_dot; per column the operator application is stream_Ax's FMA order
// (reg_Ax is the same sequence on the register copy), so each column's y and partial sums are f_matvec_dot's bits.
template <int M, int ST>
__global__ void __launch_bounds__(256) f_matvec_dot_multi(const double* __restrict__ mat, int K, int ilo, int iup,
                                                          const __grid_constant__ MatvecCols cols, int k, int64_t n) {
    using S = OpShape<M, ST>;
    constexpr bool REG = MatvecOpInRegs<M, ST>::value;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = e < n;
    const double* T = mat + (e >> 5) * (int64_t)K * AMG1D_TILE + (e & 31);
    RegOp<M, ST> A;
    if constexpr (REG) {
        if (active) {
#pragma unroll
            for (int q = 0; q < S::NO; ++q) A.lo[q] = T[q * AMG1D_TILE];
#pragma unroll
            for (int q = 0; q < M * M; ++q) A.di[q] = T[(S::O_DI + q) * AMG1D_TILE];
#pragma unroll
            for (int q = 0; q < S::NO; ++q) A.up[q] = T[(S::O_UP + q) * AMG1D_TILE];
        }
    }
#pragma unroll 1
    for (int c = 0; c < k; ++c) {
        if (c) __syncthreads();                  // block_sum's shared scratch is reused by the next column
        double s = 0.0;
        if (active) {
            const double* x = cols.x[c];
            double xl[M], xc[M], xr[M], yy[M];
            load_vec<M>(x + e * M, xc);
            load_neighbours<M, ST>(x, e, ilo, iup, xl, xr);
            if constexpr (REG) reg_Ax<M, ST>(A, ilo, iup, xl, xc, xr, yy);
            else stream_Ax<M, ST>(T, ilo, iup, xl, xc, xr, yy);
            store_vec<M>(cols.y[c] + e * M, yy);
#pragma unroll
            for (int i = 0; i < M; ++i) s = fma(xc[i], yy[i], s);
        }
        if (cols.partial[c]) {
            s = block_sum(s);
            if (threadIdx.x == 0) cols.partial[c][blockIdx.x] = s;
        }
    }
}

// Exactly fused_matvec_dot's predicate and grid: where it returns false the caller runs op_matvec_dot per column.
inline bool fused_matvec_dot_multi(const MatDesc& d, const double* mat, const MatvecCols& cols, int k, int64_t n,
                                   int64_t partial_cap, int* nblocks, cudaStream_t st) {
    const int64_t grid = (n + 255) / 256;
    if (grid > partial_cap || !fast_tier_ok(d)) return false;
    *nblocks = (int)grid;
    switch (d.m * 4 + d.st) {
#define Y(MM, SS)                                                                                                   \
    case MM * 4 + SS:                                                                                               \
        f_matvec_dot_multi<MM, SS><<<(unsigned)grid, 256, 0, st>>>(mat, d.K, d.ilo, d.iup, cols, k, n);             \
        return true;
#define X(MM) Y(MM, 0) Y(MM, 1) Y(MM, 2)
        FUSED_FOR_M(X) Y(2, 3)
#undef X
#undef Y
        default: return false;
    }
}
