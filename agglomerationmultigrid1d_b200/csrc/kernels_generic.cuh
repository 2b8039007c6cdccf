// Generic kernel tier: any block size m <= 32, any structure class (layout.cuh), diagonal or block
// smoother, one- or two-parent transfers with arbitrary (non-decreasing) parent maps.  One thread per (element, row); launch with
// blockDim = (32 lanes, m rows, Z tiles).  These are the always-available, always-correct kernels;
// the templated thread-per-element kernels in kernels_fused.cuh replace them on the hot levels.
//
// Reference operations (file:line relative to the reference tree):
//   g_sweep        u += alpha * S^-1 (rhs - A u)          src/solvers.jl:32-35, :43-46 with
//                                                         src/smoother.jl:52-58 / :69-81
//   g_apply        A u   or   rhs - A u                   src/solvers.jl:33, :129
//   g_restrict     L' r                                   src/solvers.jl:36
//   g_prolong      u += L u_c   or   u = L u_c            src/solvers.jl:42
#pragma once
#include "layout.cuh"

// Parent of fine element e and index of its transfer block.
struct TransferMap {
    const int64_t* parent;   // explicit map (may be null -> formula below)
    const int64_t* cp;       // child pointers, n_coarse + 2 entries: children with parent q-1 start at cp[q]
    int64_t n_fine, n_coarse;
    int ratio, shift, base;  // parent[e] = (e + shift) / ratio + base
    int period, n_head, n_tail; // block index pattern; period == 0 -> one block per element
    __device__ __forceinline__ int64_t par(int64_t e) const {
        return parent ? parent[e] : (e + shift) / ratio + base;
    }
    __device__ __forceinline__ int64_t blk(int64_t e) const {
        if (period == 0) return e;
        if (e < n_head) return e;
        if (e >= n_fine - n_tail) return n_head + period + (e - (n_fine - n_tail));
        return n_head + (e - n_head) % period;
    }
    // children whose parent is q: [first(q), first(q+1))
    __device__ __forceinline__ int64_t first(int64_t q) const {
        if (cp) return cp[q + 1];
        // smallest e with (e + shift) / ratio + base >= q
        int64_t v = (q - base) * (int64_t)ratio - shift;
        if (v < 0) v = 0;
        if (v > n_fine) v = n_fine;
        return v;
    }
};

// Row i of  A_lo x_l + A_di x_c + A_up x_r  for one element; T points at [tile][0][lane].  Terms are
// accumulated in ascending column order, A_lo first, then A_di, then A_up (the order of a CSC SpMV over
// the reference's DOF numbering); the compressed structure classes skip exact zeros only (ST_REPEAT
// skips nothing: it reads every A_lo(i, j) from c[i] and every A_up(i, j) from r[j]).
__device__ __forceinline__ double g_row_Ax(const double* __restrict__ T, const MatDesc& d, int i,
                                           const double* xl, const double* xc, const double* xr) {
    const int m = d.m;
    double y = 0.0;
    if (d.st == AMG1D_ST_DENSE) {
        for (int j = 0; j < m; ++j) y = fma(T[(j * m + i) * AMG1D_TILE], xl[j], y);
    } else if (d.st == AMG1D_ST_REPEAT) {
        for (int j = 0; j < m; ++j) y = fma(T[i * AMG1D_TILE], xl[j], y);
    } else if (d.st == AMG1D_ST_COLROW) {
        y = fma(T[i * AMG1D_TILE], xl[d.ilo], y);
    } else if (i == d.ilo) {
        for (int j = 0; j < m; ++j) y = fma(T[j * AMG1D_TILE], xl[j], y);
    }
    const double* D = T + (int64_t)d.o_di * AMG1D_TILE;
    for (int j = 0; j < m; ++j) y = fma(D[(j * m + i) * AMG1D_TILE], xc[j], y);
    const double* U = T + (int64_t)d.o_up * AMG1D_TILE;
    if (d.st == AMG1D_ST_DENSE) {
        for (int j = 0; j < m; ++j) y = fma(U[(j * m + i) * AMG1D_TILE], xr[j], y);
    } else if (d.st == AMG1D_ST_REPEAT) {
        for (int j = 0; j < m; ++j) y = fma(U[j * AMG1D_TILE], xr[j], y);
    } else if (d.st == AMG1D_ST_ROWCOL) {
        y = fma(U[i * AMG1D_TILE], xr[d.iup], y);
    } else if (i == d.iup) {
        for (int j = 0; j < m; ++j) y = fma(U[j * AMG1D_TILE], xr[j], y);
    }
    return y;
}

// Row i of Dinv r (block smoother) or Dinv_i r_i (diagonal smoother); r is the element's residual.
__device__ __forceinline__ double g_row_Dinv(const double* __restrict__ T, const MatDesc& d, int i,
                                             const double* r, int rstride) {
    const double* V = T + (int64_t)d.o_dv * AMG1D_TILE;
    if (d.diag) return V[i * AMG1D_TILE] * r[i * rstride];
    double z = 0.0;
    for (int j = 0; j < d.m; ++j) z = fma(V[(j * d.m + i) * AMG1D_TILE], r[j * rstride], z);
    return z;
}

// x_new = x + alpha * Dinv (b - A x).  zero_guess: x is taken as 0 and A is not read.
__global__ void g_sweep(const double* __restrict__ mat, MatDesc d, const double* __restrict__ b,
                        const double* __restrict__ xin, double* __restrict__ xout, int64_t n,
                        double alpha, int zero_guess) {
    extern __shared__ double r_s[];  // [Z][m][32]
    const int m = d.m;
    const int lane = threadIdx.x, i = threadIdx.y, tz = threadIdx.z;
    const int64_t tile = (int64_t)blockIdx.x * blockDim.z + tz;
    const int64_t e = tile * AMG1D_TILE + lane;
    const bool valid = e < n;
    const double* T = mat + tile * (int64_t)d.K * AMG1D_TILE + lane;
    double r = 0.0;
    if (valid) {
        double y = 0.0;
        if (!zero_guess) y = g_row_Ax(T, d, i, xin + (e - 1) * m, xin + e * m, xin + (e + 1) * m);
        r = b[e * m + i] - y;
    }
    double* rs = r_s + (size_t)tz * m * AMG1D_TILE;
    rs[i * AMG1D_TILE + lane] = r;
    __syncthreads();
    if (valid) {
        const double z = g_row_Dinv(T, d, i, rs + lane, AMG1D_TILE);
        const double x0 = zero_guess ? 0.0 : xin[e * m + i];
        xout[e * m + i] = __dadd_rn(x0, __dmul_rn(alpha, z));
    }
}

// out = A x (mode 0) or out = b - A x (mode 1).
__global__ void g_apply(const double* __restrict__ mat, MatDesc d, const double* __restrict__ b,
                        const double* __restrict__ x, double* __restrict__ out, int64_t n, int mode) {
    const int m = d.m;
    const int lane = threadIdx.x, i = threadIdx.y, tz = threadIdx.z;
    const int64_t tile = (int64_t)blockIdx.x * blockDim.z + tz;
    const int64_t e = tile * AMG1D_TILE + lane;
    if (e >= n) return;
    const double* T = mat + tile * (int64_t)d.K * AMG1D_TILE + lane;
    const double y = g_row_Ax(T, d, i, x + (e - 1) * m, x + e * m, x + (e + 1) * m);
    out[e * m + i] = mode ? b[e * m + i] - y : y;
}

// Y = alpha * Dinv * B  (apply_smoother, src/smoother.jl:52-58, :69-81)
__global__ void g_apply_smoother(const double* __restrict__ mat, MatDesc d,
                                 const double* __restrict__ B, double* __restrict__ Y, int64_t n,
                                 double alpha) {
    const int m = d.m;
    const int lane = threadIdx.x, i = threadIdx.y, tz = threadIdx.z;
    const int64_t tile = (int64_t)blockIdx.x * blockDim.z + tz;
    const int64_t e = tile * AMG1D_TILE + lane;
    if (e >= n) return;
    const double* T = mat + tile * (int64_t)d.K * AMG1D_TILE + lane;
    Y[e * m + i] = __dmul_rn(alpha, g_row_Dinv(T, d, i, B + e * m, 1));
}

// xout = x + alpha * (S r) for a block-tridiagonal smoother operator S stored like a level operator
// (overlapping Schwarz smoothers, src/smoother.jl:1-46); x == nullptr: xout = alpha * (S r), which is
// apply_smoother itself.  r must carry zero (or valid) ghost elements.
__global__ void g_apply_tri_smoother(const double* __restrict__ smat, MatDesc d, const double* __restrict__ r,
                                     const double* __restrict__ x, double* __restrict__ xout, int64_t n,
                                     double alpha) {
    const int m = d.m;
    const int lane = threadIdx.x, i = threadIdx.y, tz = threadIdx.z;
    const int64_t tile = (int64_t)blockIdx.x * blockDim.z + tz;
    const int64_t e = tile * AMG1D_TILE + lane;
    if (e >= n) return;
    const double* T = smat + tile * (int64_t)d.K * AMG1D_TILE + lane;
    const double z = g_row_Ax(T, d, i, r + (e - 1) * m, r + e * m, r + (e + 1) * m);
    const double az = __dmul_rn(alpha, z);
    xout[e * m + i] = x ? __dadd_rn(x[e * m + i], az) : az;
}

// rc[Kc] = sum_{parent(e) = Kc-1} P1[e]' rf[e] + sum_{parent(e) = Kc} P0[e]' rf[e]
// one thread per (coarse element, coarse row); P blocks are m_f x m_c column-major.
__global__ void g_restrict(TransferMap tm, int mf, int mc, const double* __restrict__ P0,
                           const double* __restrict__ P1, const double* __restrict__ rf,
                           double* __restrict__ rc) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= tm.n_coarse * mc) return;
    const int64_t Kc = idx / mc;
    const int jc = (int)(idx % mc);
    const int bs = mf * mc;
    double acc = 0.0;
    if (P1) {
        const int64_t e0 = tm.first(Kc - 1), e1 = tm.first(Kc);
        for (int64_t e = e0; e < e1; ++e) {
            const double* P = P1 + tm.blk(e) * bs + jc * mf;
            const double* r = rf + e * mf;
            for (int i = 0; i < mf; ++i) acc = fma(P[i], r[i], acc);
        }
    }
    {
        const int64_t e0 = tm.first(Kc), e1 = tm.first(Kc + 1);
        for (int64_t e = e0; e < e1; ++e) {
            const double* P = P0 + tm.blk(e) * bs + jc * mf;
            const double* r = rf + e * mf;
            for (int i = 0; i < mf; ++i) acc = fma(P[i], r[i], acc);
        }
    }
    rc[idx] = acc;
}

// xf[e] (+)= P0[e] xc[parent(e)] + P1[e] xc[parent(e) + 1]; one thread per (fine element, row).
__global__ void g_prolong(TransferMap tm, int mf, int mc, const double* __restrict__ P0,
                          const double* __restrict__ P1, const double* __restrict__ xc,
                          double* __restrict__ xf, int add) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= tm.n_fine * mf) return;
    const int64_t e = idx / mf;
    const int i = (int)(idx % mf);
    const int bs = mf * mc;
    const int64_t par = tm.par(e);
    const int64_t pb = tm.blk(e) * bs;
    double y = 0.0;
    const double* c0 = xc + par * mc;
    for (int j = 0; j < mc; ++j) y = fma(P0[pb + j * mf + i], c0[j], y);
    if (P1) {
        const double* c1 = xc + (par + 1) * mc;
        for (int j = 0; j < mc; ++j) y = fma(P1[pb + j * mf + i], c1[j], y);
    }
    xf[idx] = add ? xf[idx] + y : y;
}

// Coarsest level: block-Thomas substitution with the factors prepared at finalize.
//   forward  y_k = b_k - W_k y_{k-1}          W_k = A_lo[k] * Sinv_{k-1}
//   backward x_k = Sinv_k (y_k - A_up[k] x_{k+1})
// One warp, lane i owns row i (m <= 32).  fac[k] = { W (m*m), Sinv (m*m), U (m*m) } column-major.
// yp / wk: m doubles of shared memory each.
__device__ __forceinline__ void coarse_solve_warp(const double* __restrict__ fac, int m, int64_t n,
                                                  const double* b, double* x, double* yp, double* wk) {
    const int i = threadIdx.x & 31;
    const int mm = m * m;
    // forward sweep; y stored temporarily in x
    for (int64_t k = 0; k < n; ++k) {
        if (i < m) {
            double acc = 0.0;
            if (k > 0) {
                const double* W = fac + k * 3 * mm;
                for (int j = 0; j < m; ++j) acc = fma(W[j * m + i], yp[j], acc);
            }
            wk[i] = b[k * m + i] - acc;
        }
        __syncwarp();
        if (i < m) { yp[i] = wk[i]; x[k * m + i] = wk[i]; }
        __syncwarp();
    }
    // backward sweep; yp now holds x_{k+1}
    for (int64_t k = n - 1; k >= 0; --k) {
        const double* Sinv = fac + k * 3 * mm + mm;
        const double* U = fac + k * 3 * mm + 2 * mm;
        if (i < m) {
            double acc = x[k * m + i];
            if (k < n - 1)
                for (int j = 0; j < m; ++j) acc = fma(-U[j * m + i], yp[j], acc);
            wk[i] = acc;
        }
        __syncwarp();
        double xi = 0.0;
        if (i < m)
            for (int j = 0; j < m; ++j) xi = fma(Sinv[j * m + i], wk[j], xi);
        __syncwarp();
        if (i < m) { yp[i] = xi; x[k * m + i] = xi; }
        __syncwarp();
    }
}

__global__ void g_coarse_solve(const double* __restrict__ fac, int m, int64_t n,
                               const double* __restrict__ b, double* __restrict__ x) {
    extern __shared__ double sh[];  // y_prev[m], work[m]
    coarse_solve_warp(fac, m, n, b, x, sh, sh + m);
}

// ---- reductions (deterministic: fixed partial layout, fixed final order) -----------------------
#define AMG1D_RED_BLOCKS 1024
#define AMG1D_RED_THREADS 256

__device__ __forceinline__ double block_sum(double v) {
    __shared__ double ws[32];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) ws[w] = v;
    __syncthreads();
    double t = 0.0;
    if (w == 0) {
        t = (l < (blockDim.x >> 5)) ? ws[l] : 0.0;
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    }
    return t;  // valid in thread 0
}

// The per-element statements of the reductions and CG vector updates below, over this block's grid-stride slice
// (block blockIdx.x of gridDim.x).  The single-column kernels and their multi-column forms (column = blockIdx.y, the
// same gridDim.x per column) both call them, so each column's partial sums are those of the single-column kernel.
#define GRID_SLICE(i, n) \
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (int64_t)gridDim.x * blockDim.x)

__device__ __forceinline__ double sqdiff_slice(const double* __restrict__ a, const double* __restrict__ c, int64_t n) {
    double s = 0.0;
    GRID_SLICE(i, n) {
        const double d = c ? a[i] - c[i] : a[i];
        s = fma(d, d, s);
    }
    return s;
}

__device__ __forceinline__ double dot_slice(const double* __restrict__ a, const double* __restrict__ c, int64_t n) {
    double s = 0.0;
    GRID_SLICE(i, n) s = fma(a[i], c[i], s);
    return s;
}

__device__ __forceinline__ double sum_slice(const double* __restrict__ partial, int64_t np) {
    double s = 0.0;
    GRID_SLICE(i, np) s += partial[i];
    return s;
}

// one block: the final stage, in a fixed order (thread t sums entries t, t + blockDim.x, ...)
__device__ __forceinline__ double reduce_final_sum(const double* __restrict__ partial, int np) {
    double s = 0.0;
    for (int i = threadIdx.x; i < np; i += blockDim.x) s += partial[i];
    return block_sum(s);
}

// partial[b] = sum over a grid-stride slice of (a[i] - c[i])^2   (c may be null)
__global__ void k_sqdiff_partial(const double* __restrict__ a, const double* __restrict__ c,
                                 int64_t n, double* __restrict__ partial) {
    const double s = block_sum(sqdiff_slice(a, c, n));
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

// partial[b] = sum over a grid-stride slice of a[i] * c[i]
__global__ void k_dot_partial(const double* __restrict__ a, const double* __restrict__ c, int64_t n,
                              double* __restrict__ partial) {
    const double s = block_sum(dot_slice(a, c, n));
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

// ---- conjugate gradients (amg1d_pcg): scalars live in the device scalar array ------------------------
enum { CG_RES = 0, CG_NB = 2, CG_RZ = 3, CG_PAP = 4, CG_ALPHA = 5, CG_BETA = 6, CG_RZ_NEW = 7 };

__device__ __forceinline__ void axpy_slice(double* __restrict__ y, const double* __restrict__ x, int64_t n, double a) {
    GRID_SLICE(i, n) y[i] = fma(a, x[i], y[i]);
}

// alpha = rz / pAp
// (a zero denominator - b = 0, or an exact x0 - gives a zero step instead of 0/0 = NaN)
__device__ __forceinline__ void cg_alpha(double* s) { s[CG_ALPHA] = s[CG_PAP] != 0.0 ? s[CG_RZ] / s[CG_PAP] : 0.0; }
// beta = rz_new / rz; rz = rz_new
__device__ __forceinline__ void cg_beta(double* s) {
    s[CG_BETA] = s[CG_RZ] != 0.0 ? s[CG_RZ_NEW] / s[CG_RZ] : 0.0;
    s[CG_RZ] = s[CG_RZ_NEW];
}

// x += alpha p;  r -= alpha Ap;  returns the slice's sum of r[i]^2
__device__ __forceinline__ double cg_update_slice(double* __restrict__ x, double* __restrict__ r,
                                                  const double* __restrict__ p, const double* __restrict__ Ap,
                                                  int64_t n, double alpha) {
    double acc = 0.0;
    GRID_SLICE(i, n) {
        x[i] = fma(alpha, p[i], x[i]);
        const double ri = fma(-alpha, Ap[i], r[i]);
        r[i] = ri;
        acc = fma(ri, ri, acc);
    }
    return acc;
}

// p = z + beta p   (first: p = z)
__device__ __forceinline__ void cg_direction_slice(double* __restrict__ p, const double* __restrict__ z, int64_t n,
                                                   double beta, int first) {
    GRID_SLICE(i, n) p[i] = first ? z[i] : fma(beta, p[i], z[i]);
}

// y += a x
__global__ void k_axpy(double* __restrict__ y, const double* __restrict__ x, int64_t n, double a) {
    axpy_slice(y, x, n, a);
}

__global__ void k_cg_alpha(double* s) { cg_alpha(s); }
__global__ void k_cg_beta(double* s) { cg_beta(s); }

// x += alpha p;  r -= alpha Ap;  partial[b] = sum r[i]^2 over the block's slice
__global__ void k_cg_update(double* __restrict__ x, double* __restrict__ r, const double* __restrict__ p,
                            const double* __restrict__ Ap, int64_t n, const double* __restrict__ s,
                            double* __restrict__ partial) {
    const double acc = block_sum(cg_update_slice(x, r, p, Ap, n, s[CG_ALPHA]));
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

// p = z + beta p   (first = 1: p = z)
__global__ void k_cg_direction(double* __restrict__ p, const double* __restrict__ z, int64_t n,
                               const double* __restrict__ s, int first) {
    cg_direction_slice(p, z, n, first ? 0.0 : s[CG_BETA], first);
}

// second-stage partial sums for long partial arrays: out[b] = sum of a fixed grid-stride slice
__global__ void k_sum_partial(const double* __restrict__ partial, int64_t np, double* __restrict__ out) {
    const double s = block_sum(sum_slice(partial, np));
    if (threadIdx.x == 0) out[blockIdx.x] = s;
}

// out[slot] = sqrt(sum partial[0..np))
__global__ void k_reduce_final(const double* __restrict__ partial, int np, double* __restrict__ out,
                               int slot, int take_sqrt) {
    const double s = reduce_final_sum(partial, np);
    if (threadIdx.x == 0) out[slot] = take_sqrt ? sqrt(s) : s;
}

// ---- the same for up to MULTI_MAX_COLS columns in one launch (amg1d_dev_pcg_multi) --------------------
// Column i of a launch is blockIdx.y (the scalar kernels: threadIdx.x); every ColVecs entry i is that column's
// vector, partial array or scalar window.  Per column the grid, the slices and the partial layout are those of the
// single-column kernel, so the column's results are bit-identical to it.
#define MULTI_MAX_COLS 8

struct ColVecs {
    double* v[MULTI_MAX_COLS];
};

__global__ void k_sqdiff_partial_multi(const __grid_constant__ ColVecs a, int64_t n, const __grid_constant__ ColVecs partial) {
    const int c = blockIdx.y;
    const double s = block_sum(sqdiff_slice(a.v[c], nullptr, n));
    if (threadIdx.x == 0) partial.v[c][blockIdx.x] = s;
}

__global__ void k_dot_partial_multi(const __grid_constant__ ColVecs a, const __grid_constant__ ColVecs b, int64_t n,
                                    const __grid_constant__ ColVecs partial) {
    const int c = blockIdx.y;
    const double s = block_sum(dot_slice(a.v[c], b.v[c], n));
    if (threadIdx.x == 0) partial.v[c][blockIdx.x] = s;
}

__global__ void k_axpy_multi(const __grid_constant__ ColVecs y, const __grid_constant__ ColVecs x, int64_t n, double a) {
    axpy_slice(y.v[blockIdx.y], x.v[blockIdx.y], n, a);
}

__global__ void k_cg_alpha_multi(const __grid_constant__ ColVecs s) { cg_alpha(s.v[threadIdx.x]); }
__global__ void k_cg_beta_multi(const __grid_constant__ ColVecs s) { cg_beta(s.v[threadIdx.x]); }

__global__ void k_cg_update_multi(const __grid_constant__ ColVecs x, const __grid_constant__ ColVecs r,
                                  const __grid_constant__ ColVecs p, const __grid_constant__ ColVecs Ap, int64_t n,
                                  const __grid_constant__ ColVecs s, const __grid_constant__ ColVecs partial) {
    const int c = blockIdx.y;
    const double acc = block_sum(cg_update_slice(x.v[c], r.v[c], p.v[c], Ap.v[c], n, s.v[c][CG_ALPHA]));
    if (threadIdx.x == 0) partial.v[c][blockIdx.x] = acc;
}

__global__ void k_cg_direction_multi(const __grid_constant__ ColVecs p, const __grid_constant__ ColVecs z, int64_t n,
                                     const __grid_constant__ ColVecs s, int first) {
    const int c = blockIdx.y;
    cg_direction_slice(p.v[c], z.v[c], n, first ? 0.0 : s.v[c][CG_BETA], first);
}

__global__ void k_sum_partial_multi(const __grid_constant__ ColVecs partial, int64_t np,
                                    const __grid_constant__ ColVecs out) {
    const int c = blockIdx.y;
    const double s = block_sum(sum_slice(partial.v[c], np));
    if (threadIdx.x == 0) out.v[c][blockIdx.x] = s;
}

// out.v[i][slot] = sum (or its square root) of partial.v[i][0..np)
__global__ void k_reduce_final_multi(const __grid_constant__ ColVecs partial, int np, const __grid_constant__ ColVecs out,
                                     int slot, int take_sqrt) {
    const int c = blockIdx.y;
    const double s = reduce_final_sum(partial.v[c], np);
    if (threadIdx.x == 0) out.v[c][slot] = take_sqrt ? sqrt(s) : s;
}

// ---- set-up helpers -----------------------------------------------------------------------------
// Value of tile row k for an element whose uploaded blocks start at lo / di / up (m*m each, column
// major) and dinv (m*m or m).
__device__ __forceinline__ double tile_value(const MatDesc& d, int k, const double* lo, const double* di,
                                             const double* up, const double* dinv) {
    int which, idx;
    amg1d_row_source(d, k, &which, &idx);
    return which == 0 ? lo[idx] : which == 1 ? di[idx] : which == 2 ? up[idx] : dinv[idx];
}

// Repack element-block host layout (already copied to the device chunk buffers) into element tiles.
// src arrays hold `cnt` elements starting at element e0; dinv has m*m or m doubles per element.
__global__ void k_repack(const double* __restrict__ lo, const double* __restrict__ di,
                         const double* __restrict__ up, const double* __restrict__ dinv, MatDesc d,
                         int64_t e0, int64_t cnt, double* __restrict__ mat) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // t enumerates (tile_local, k, lane) over the tiles touched by [e0, e0+cnt); e0 % 32 == 0
    // (e0 = -32 addresses the spare front tile of a slab with left ghost elements)
    const int64_t per_tile = (int64_t)d.K * AMG1D_TILE;
    const int64_t tl = t / per_tile;
    const int k = (int)((t % per_tile) / AMG1D_TILE);
    const int lane = (int)(t % AMG1D_TILE);
    const int64_t el = tl * AMG1D_TILE + lane;
    if (el >= cnt) {
        if (tl < (cnt + AMG1D_TILE - 1) / AMG1D_TILE)
            mat[(e0 / AMG1D_TILE + tl) * per_tile + (int64_t)k * AMG1D_TILE + lane] = 0.0;
        return;
    }
    const int mm = d.m * d.m;
    const int dsz = d.diag ? d.m : mm;
    mat[(e0 / AMG1D_TILE + tl) * per_tile + (int64_t)k * AMG1D_TILE + lane] =
        tile_value(d, k, lo + el * mm, di + el * mm, up + el * mm, dinv + el * dsz);
}

// Fill the stored tiles of a (slab of a) level from a head / interior / tail pattern of
// n_head + 1 + n_tail element block sets.  `store` starts one tile before local element 0; local
// element e = stored index - 32 maps to global element start + e; only local elements in
// [e_lo, e_hi) that exist globally are filled, everything else is zero.
__global__ void k_fill_pattern(const double* __restrict__ lo, const double* __restrict__ di,
                               const double* __restrict__ up, const double* __restrict__ dinv,
                               MatDesc d, int64_t n_glob, int n_head, int n_tail, int64_t start,
                               int64_t e_lo, int64_t e_hi, int64_t ntiles, double* __restrict__ store) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t per_tile = (int64_t)d.K * AMG1D_TILE;
    const int64_t tile = t / per_tile;
    if (tile >= ntiles) return;
    const int k = (int)((t % per_tile) / AMG1D_TILE);
    const int lane = (int)(t % AMG1D_TILE);
    const int64_t e = tile * AMG1D_TILE + lane - AMG1D_TILE;   // local element index
    const int64_t eg = start + e;                              // global element index
    double v = 0.0;
    if (e >= e_lo && e < e_hi && eg >= 0 && eg < n_glob) {
        int64_t s;
        if (eg < n_head) s = eg;
        else if (eg >= n_glob - n_tail) s = n_head + 1 + (eg - (n_glob - n_tail));
        else s = n_head;
        const int mm = d.m * d.m;
        const int dsz = d.diag ? d.m : mm;
        v = tile_value(d, k, lo + s * mm, di + s * mm, up + s * mm, dinv + s * dsz);
    }
    store[t] = v;
}

// device slot s <- host-ordered vector (perm[s] = host DOF, -1 = padding)
__global__ void k_gather_perm(const int64_t* __restrict__ perm, const double* __restrict__ hostord,
                              double* __restrict__ dev, int64_t nslots) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nslots) return;
    const int64_t p = perm[s];
    dev[s] = p >= 0 ? hostord[p] : 0.0;
}

__global__ void k_scatter_perm(const int64_t* __restrict__ perm, const double* __restrict__ dev,
                               double* __restrict__ hostord, int64_t nslots) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nslots) return;
    const int64_t p = perm[s];
    if (p >= 0) hostord[p] = dev[s];
}

// b[i] = uniform(-1, 1) from a counter-based hash (splitmix64); x = 0
__global__ void k_fill_random(double* __restrict__ b, int64_t n, uint64_t seed, int64_t offset) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        uint64_t z = seed + 0x9E3779B97F4A7C15ull * (uint64_t)(i + offset + 1);   // global DOF index
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z = z ^ (z >> 31);
        b[i] = (double)(z >> 11) * (2.0 / 9007199254740992.0) - 1.0;
    }
}
