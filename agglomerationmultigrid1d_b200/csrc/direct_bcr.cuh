// GPU direct solver for block-tridiagonal systems: block cyclic reduction (BCR).
//
// Stands in for the sparse direct solves of the reference at any size:
//   mStiffness[end] \ rhs        src/solvers.jl:39    (coarsest level of a V-cycle)
//   A \ b  (u_exact)             src/solvers.jl:120, :194  (error histories of multigrid / smoother solve)
// (SuiteSparse behind Julia's `\`; SURVEY 8f-2).  The serial block-Thomas kernel (g_coarse_solve) remains
// for coarsest levels of a few elements; BCR takes over above AMG1D_BCR_MIN elements.
//
// One reduction step eliminates the odd-numbered blocks of the current system and leaves a block-
// tridiagonal system in the even-numbered ones (i = 2j, neighbours l = i-1, r = i+1):
//     al = -A_lo[i] inv(A_di[l])        ga = -A_up[i] inv(A_di[r])
//     A_di'[j] = A_di[i] + al A_up[l] + ga A_lo[r]     A_lo'[j] = al A_lo[l]     A_up'[j] = ga A_up[r]
//     b'[j]    = b[i]    + al b[l]    + ga b[r]
// and the back substitution recovers  x[l] = inv(A_di[l]) (b[l] - A_lo[l] x[l-1] - A_up[l] x[l+1]).
// ceil(log2 n) steps end in one block.  The factorisation (al, ga, the inverses of the eliminated
// diagonal blocks and the off-diagonal blocks of every step) is computed once on the device; a solve is
// one small kernel per step down and one per step up (2 ceil(log2 n) + 1 launches), every one of them
// parallel over the blocks of its step.  For the symmetric positive definite operators of this package
// cyclic reduction is Gaussian elimination in nested-dissection order without pivoting across blocks,
// which is stable; inside a block the inverse uses partial pivoting.
//
// Storage per step k (n_k blocks, element-block layout, column-major m x m blocks):
//     lo, di, up : n_k blocks each (di of the eliminated blocks is replaced by its inverse)
//     al, ga     : n_{k+1} blocks each
// i.e. about 2 n (3 + 2) m^2 doubles in total.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <vector>

#include "layout.cuh"

#define AMG1D_BCR_MIN 64        // coarsest levels with more elements than this use BCR
#define AMG1D_BCR_MAXM 32

// Element tiles (any structure class) -> plain element-block arrays lo / di / up (n blocks of m*m).
__global__ void k_bcr_extract(const double* __restrict__ mat, MatDesc d, int64_t n, double* __restrict__ lo,
                              double* __restrict__ di, double* __restrict__ up) {
    const int mm = d.m * d.m;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * mm) return;
    const int64_t e = t / mm;
    const int q = (int)(t % mm);
    const int j = q / d.m, i = q % d.m;
    const double* T = mat + (e >> 5) * (int64_t)d.K * AMG1D_TILE + (e & 31);
    double vlo, vup;
    if (d.st == AMG1D_ST_DENSE) {
        vlo = T[q * AMG1D_TILE];
        vup = T[(d.o_up + q) * AMG1D_TILE];
    } else if (d.st == AMG1D_ST_REPEAT) {
        vlo = T[i * AMG1D_TILE];
        vup = T[(d.o_up + j) * AMG1D_TILE];
    } else if (d.st == AMG1D_ST_COLROW) {
        vlo = (j == d.ilo) ? T[i * AMG1D_TILE] : 0.0;
        vup = (i == d.iup) ? T[(d.o_up + j) * AMG1D_TILE] : 0.0;
    } else {
        vlo = (i == d.ilo) ? T[j * AMG1D_TILE] : 0.0;
        vup = (j == d.iup) ? T[(d.o_up + i) * AMG1D_TILE] : 0.0;
    }
    lo[t] = vlo;
    di[t] = T[(d.o_di + q) * AMG1D_TILE];
    up[t] = vup;
}

// In-place inverse of the diagonal blocks first, first + stride, ... (Gauss-Jordan with partial
// pivoting, row swaps undone as column swaps at the end); one thread per block, working directly on
// the block in global memory (done once per factorisation).  flag[0] is set when a block is singular.
__global__ void k_bcr_invert_odd(double* __restrict__ di, int m, int64_t n, int first, int stride,
                                 int* __restrict__ flag) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t blk = first + j * stride;
    if (blk >= n) return;
    double* A = di + blk * m * m;                 // column-major: entry (r, c) at A[c * m + r]
    int piv[AMG1D_BCR_MAXM];
    for (int c = 0; c < m; ++c) {
        int p = c;
        double best = fabs(A[c * m + c]);
        for (int r = c + 1; r < m; ++r)
            if (fabs(A[c * m + r]) > best) { best = fabs(A[c * m + r]); p = r; }
        if (best == 0.0) { flag[0] = 1; return; }
        piv[c] = p;
        if (p != c)
            for (int q = 0; q < m; ++q) { const double s = A[q * m + c]; A[q * m + c] = A[q * m + p]; A[q * m + p] = s; }
        const double d = 1.0 / A[c * m + c];
        A[c * m + c] = 1.0;
        for (int q = 0; q < m; ++q) A[q * m + c] *= d;
        for (int r = 0; r < m; ++r) {
            if (r == c) continue;
            const double f = A[c * m + r];
            A[c * m + r] = 0.0;
            if (f == 0.0) continue;
            for (int q = 0; q < m; ++q) A[q * m + r] = fma(-f, A[q * m + c], A[q * m + r]);
        }
    }
    for (int c = m - 1; c >= 0; --c) {
        const int p = piv[c];
        if (p != c)
            for (int r = 0; r < m; ++r) { const double s = A[c * m + r]; A[c * m + r] = A[p * m + r]; A[p * m + r] = s; }
    }
}

// C(:, c) = -A B(:, c): helper for one column (A, B column-major m x m)
__device__ __forceinline__ void bcr_col_negprod(const double* A, const double* B, int m, int c, double* out) {
    for (int i = 0; i < m; ++i) {
        double s = 0.0;
        for (int k = 0; k < m; ++k) s = fma(A[k * m + i], B[c * m + k], s);
        out[i] = -s;
    }
}

// al[j] = -lo[2j] dinv[2j-1],  ga[j] = -up[2j] dinv[2j+1]; one thread per (kept block j, column c)
__global__ void k_bcr_alpha_gamma(const double* __restrict__ lo, const double* __restrict__ di,
                                  const double* __restrict__ up, int m, int64_t n, int64_t n_next,
                                  double* __restrict__ al, double* __restrict__ ga) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_next * m) return;
    const int64_t j = t / m;
    const int c = (int)(t % m);
    const int64_t i = 2 * j;
    const int mm = m * m;
    double col[AMG1D_BCR_MAXM];
    if (i - 1 >= 0) {
        bcr_col_negprod(lo + i * mm, di + (i - 1) * mm, m, c, col);
        for (int r = 0; r < m; ++r) al[j * mm + c * m + r] = col[r];
    } else {
        for (int r = 0; r < m; ++r) al[j * mm + c * m + r] = 0.0;
    }
    if (i + 1 < n) {
        bcr_col_negprod(up + i * mm, di + (i + 1) * mm, m, c, col);
        for (int r = 0; r < m; ++r) ga[j * mm + c * m + r] = col[r];
    } else {
        for (int r = 0; r < m; ++r) ga[j * mm + c * m + r] = 0.0;
    }
}

// next step's blocks from al, ga: one thread per (kept block j, column c)
__global__ void k_bcr_reduce(const double* __restrict__ lo, const double* __restrict__ di,
                             const double* __restrict__ up, const double* __restrict__ al,
                             const double* __restrict__ ga, int m, int64_t n, int64_t n_next,
                             double* __restrict__ lo2, double* __restrict__ di2, double* __restrict__ up2) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_next * m) return;
    const int64_t j = t / m;
    const int c = (int)(t % m);
    const int64_t i = 2 * j;
    const int mm = m * m;
    const double* A = al + j * mm;
    const double* G = ga + j * mm;
    const bool hasl = i - 1 >= 0, hasr = i + 1 < n;
    for (int r = 0; r < m; ++r) {
        double d = di[i * mm + c * m + r], l = 0.0, u = 0.0;
        if (hasl) {
            const double* UL = up + (i - 1) * mm;   // up[l]
            const double* LL = lo + (i - 1) * mm;   // lo[l]
            for (int k = 0; k < m; ++k) {
                d = fma(A[k * m + r], UL[c * m + k], d);
                l = fma(A[k * m + r], LL[c * m + k], l);
            }
        }
        if (hasr) {
            const double* LR = lo + (i + 1) * mm;   // lo[r]
            const double* UR = up + (i + 1) * mm;   // up[r]
            for (int k = 0; k < m; ++k) {
                d = fma(G[k * m + r], LR[c * m + k], d);
                u = fma(G[k * m + r], UR[c * m + k], u);
            }
        }
        di2[j * mm + c * m + r] = d;
        lo2[j * mm + c * m + r] = l;
        up2[j * mm + c * m + r] = u;
    }
}

// b'[j] = b[2j] + al[j] b[2j-1] + ga[j] b[2j+1]; one thread per (j, row)
__global__ void k_bcr_forward(const double* __restrict__ al, const double* __restrict__ ga, int m, int64_t n,
                              int64_t n_next, const double* __restrict__ b, double* __restrict__ b2) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_next * m) return;
    const int64_t j = t / m;
    const int r = (int)(t % m);
    const int64_t i = 2 * j;
    const int mm = m * m;
    double s = b[i * m + r];
    if (i - 1 >= 0)
        for (int k = 0; k < m; ++k) s = fma(al[j * mm + k * m + r], b[(i - 1) * m + k], s);
    if (i + 1 < n)
        for (int k = 0; k < m; ++k) s = fma(ga[j * mm + k * m + r], b[(i + 1) * m + k], s);
    b2[j * m + r] = s;
}

// x[2j] = x2[j];  x[2j+1] = dinv[2j+1] (b[2j+1] - lo[2j+1] x2[j] - up[2j+1] x2[j+1]); one thread per (block i, row)
__global__ void k_bcr_backward(const double* __restrict__ lo, const double* __restrict__ dinv,
                               const double* __restrict__ up, int m, int64_t n, int64_t n_next,
                               const double* __restrict__ b, const double* __restrict__ x2,
                               double* __restrict__ x) {
    extern __shared__ double w_s[];   // [blockDim.x]: the eliminated block's right-hand side after the neighbours' terms
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t i = t / m;
    const int r = (int)(t % m);
    const int mm = m * m;
    const bool valid = t < n * m;
    const bool odd = valid && (i & 1);
    double w = 0.0;
    if (odd) {
        const int64_t j = i >> 1;
        w = b[i * m + r];
        for (int k = 0; k < m; ++k) w = fma(-lo[i * mm + k * m + r], x2[j * m + k], w);
        if (j + 1 < n_next)
            for (int k = 0; k < m; ++k) w = fma(-up[i * mm + k * m + r], x2[(j + 1) * m + k], w);
    }
    w_s[threadIdx.x] = w;
    __syncthreads();
    if (!valid) return;
    if (!odd) { x[i * m + r] = x2[(i >> 1) * m + r]; return; }
    // blockDim.x is a multiple of m: the block's rows sit in consecutive threads
    const double* ws = w_s + (threadIdx.x - r);
    double s = 0.0;
    for (int k = 0; k < m; ++k) s = fma(dinv[i * mm + k * m + r], ws[k], s);
    x[i * m + r] = s;
}

// x = dinv b for the single block that remains
__global__ void k_bcr_last(const double* __restrict__ dinv, int m, const double* __restrict__ b,
                           double* __restrict__ x) {
    const int r = threadIdx.x;
    if (r >= m) return;
    double s = 0.0;
    for (int k = 0; k < m; ++k) s = fma(dinv[k * m + r], b[k], s);
    x[r] = s;
}

struct BcrSolver {
    int m = 0;
    int64_t n = 0;
    std::vector<int64_t> nk;                 // blocks of every step, nk.back() == 1
    std::vector<double*> lo, di, up, al, ga; // per step (al / ga: for the step's successor)
    std::vector<double*> bw, xw;             // work vectors per step (bw[0] / xw[0] are the caller's)
    int* flag = nullptr;
    int64_t bytes = 0;
    bool ready() const { return !nk.empty(); }
    int launches() const { return nk.empty() ? 0 : 2 * ((int)nk.size() - 1) + 1; }

    void release() {
        for (auto* v : {&lo, &di, &up, &al, &ga, &bw, &xw})
            for (double* p : *v) if (p) cudaFree(p);
        lo.clear(); di.clear(); up.clear(); al.clear(); ga.clear(); bw.clear(); xw.clear();
        if (flag) cudaFree(flag);
        flag = nullptr;
        nk.clear();
        bytes = 0;
    }

    // Factorise the level stored in element tiles `mat`.  Returns cudaSuccess, or an error with *singular set.
    cudaError_t factor(const double* mat, const MatDesc& d, int64_t n_elem, cudaStream_t st, bool* singular) {
        release();
        *singular = false;
        m = d.m;
        n = n_elem;
        const int mm = m * m;
        for (int64_t k = n; ; k = (k + 1) / 2) { nk.push_back(k); if (k == 1) break; }
        const size_t L = nk.size();
        lo.assign(L, nullptr); di.assign(L, nullptr); up.assign(L, nullptr);
        al.assign(L, nullptr); ga.assign(L, nullptr); bw.assign(L, nullptr); xw.assign(L, nullptr);
        cudaError_t e;
        auto alloc = [&](double** p, int64_t cnt) {
            cudaError_t r = cudaMalloc((void**)p, (size_t)std::max<int64_t>(cnt, 1) * 8);
            if (r == cudaSuccess) bytes += cnt * 8;
            return r;
        };
        if ((e = cudaMalloc((void**)&flag, sizeof(int))) != cudaSuccess) return e;
        cudaMemsetAsync(flag, 0, sizeof(int), st);
        for (size_t k = 0; k < L; ++k) {
            if ((e = alloc(&lo[k], nk[k] * mm)) != cudaSuccess) return e;
            if ((e = alloc(&di[k], nk[k] * mm)) != cudaSuccess) return e;
            if ((e = alloc(&up[k], nk[k] * mm)) != cudaSuccess) return e;
            if (k > 0) {
                if ((e = alloc(&bw[k], nk[k] * m)) != cudaSuccess) return e;
                if ((e = alloc(&xw[k], nk[k] * m)) != cudaSuccess) return e;
            }
            if (k + 1 < L) {
                if ((e = alloc(&al[k], nk[k + 1] * mm)) != cudaSuccess) return e;
                if ((e = alloc(&ga[k], nk[k + 1] * mm)) != cudaSuccess) return e;
            }
        }
        {
            const int64_t tot = n * mm;
            k_bcr_extract<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(mat, d, n, lo[0], di[0], up[0]);
        }
        for (size_t k = 0; k + 1 < L; ++k) {
            const int64_t nodd = nk[k] / 2;
            if (nodd > 0)
                k_bcr_invert_odd<<<(unsigned)((nodd + 31) / 32), 32, 0, st>>>(di[k], m, nk[k], 1, 2, flag);
            const int64_t tot = nk[k + 1] * m;
            k_bcr_alpha_gamma<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(lo[k], di[k], up[k], m, nk[k], nk[k + 1],
                                                                            al[k], ga[k]);
            k_bcr_reduce<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(lo[k], di[k], up[k], al[k], ga[k], m, nk[k],
                                                                       nk[k + 1], lo[k + 1], di[k + 1], up[k + 1]);
        }
        k_bcr_invert_odd<<<1, 32, 0, st>>>(di[L - 1], m, 1, 0, 1, flag);     // the last block
        int hflag = 0;
        if ((e = cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        *singular = hflag != 0;
        return cudaSuccess;
    }

    // x = A \ b (device pointers; b is not modified).  Returns the number of launches through *count.
    cudaError_t solve(const double* b, double* x, cudaStream_t st, int64_t* count) const {
        const size_t L = nk.size();
        const int tb = (128 / m) * m > 0 ? (128 / m) * m : m;       // threads per block: a multiple of m
        const double* bk = b;
        for (size_t k = 0; k + 1 < L; ++k) {
            const int64_t tot = nk[k + 1] * m;
            k_bcr_forward<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(al[k], ga[k], m, nk[k], nk[k + 1], bk, bw[k + 1]);
            bk = bw[k + 1];
        }
        k_bcr_last<<<1, 32, 0, st>>>(di[L - 1], m, bk, L == 1 ? x : xw[L - 1]);
        for (size_t k = L - 1; k-- > 0;) {
            const int64_t tot = nk[k] * m;
            const double* bsrc = k == 0 ? b : bw[k];
            double* xdst = k == 0 ? x : xw[k];
            k_bcr_backward<<<(unsigned)((tot + tb - 1) / tb), tb, tb * sizeof(double), st>>>(
                lo[k], di[k], up[k], m, nk[k], nk[k + 1], bsrc, xw[k + 1], xdst);
        }
        if (count) *count += launches();
        return cudaGetLastError();
    }
};
