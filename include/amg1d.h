/* amg1d.h - C ABI of libamg1d.so: the B200 (sm_100a) multigrid V-cycle of AgglomerationMultigrid1D.
 *
 * The reference (mheinz757/AgglomerationMultigrid1D, pure Julia) has no FFI; its boundary is Julia
 * dispatch on MeshHierarchy / BlockJacobi / JacobiSmoother.  Each entry point below names the
 * reference call it stands in for (file:line relative to the reference tree).  A host module (Julia
 * `ccall`, Python `ctypes`, C) assembles the operators at set-up - as the reference does - and uploads
 * them once per level; everything in src/solvers.jl then runs on the GPU.
 *
 * Conventions
 *   - every function returns an int status (AMG1D_OK = 0); text via amg1d_last_error().  Nothing
 *     throws or exits across this boundary.
 *   - all pointers are HOST pointers unless the name says `dev`; the caller owns them; the library
 *     copies what it needs before returning and never keeps a host pointer.
 *   - all floating point is FP64, all indices int64_t and 0-based (reference value - 1).
 *   - a "level" is a block-tridiagonal operator: n_elem element blocks of size m x m (m = p + 1).
 *     Blocks are column-major inside (entry (i,j) at [j*m + i]) and element-major outside, i.e. the
 *     block of element e starts at [e*m*m] (BSR-like).  Level 0 is the finest.
 *   - one handle = one CUDA stream; calls on one handle are not re-entrant.
 */
#ifndef AMG1D_H
#define AMG1D_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct amg1d amg1d_t;

enum {
    AMG1D_OK = 0,
    AMG1D_ERR_ARG = 1,      /* invalid argument / wrong call order (reference: ArgumentError) */
    AMG1D_ERR_CUDA = 2,     /* CUDA runtime error */
    AMG1D_ERR_NCCL = 3,     /* NCCL error */
    AMG1D_ERR_NOMEM = 4,    /* host or device allocation failed */
    AMG1D_ERR_STATE = 5,    /* hierarchy incomplete / not finalized */
    AMG1D_ERR_UNSUPPORTED = 6
};

/* Which device vector amg1d_dev_ptr() returns. */
enum { AMG1D_VEC_X = 0, AMG1D_VEC_B = 1, AMG1D_VEC_R = 2 };

/* ---- life cycle ------------------------------------------------------------------------------
 * Stands in for the end of MeshHierarchy(...) construction (src/mesh_heirarchy.jl:136-137,
 * :179-180): the host has built mStiffness / mSmoothers / mInterpolation and hands them over.
 * `stream` is a cudaStream_t to run on (e.g. the caller's current stream) or NULL to let the
 * library create its own. */
int amg1d_create(amg1d_t** h, int n_levels, int device, void* stream);
int amg1d_destroy(amg1d_t* h);
const char* amg1d_last_error(const amg1d_t* h); /* h may be NULL: error of the last failed create */
int amg1d_version(void);

/* Multi-GPU variant: contiguous element slabs, one rank per GPU (SURVEY 8e).  `nccl_id` is the
 * 128-byte ncclUniqueId made by amg1d_nccl_unique_id() on rank 0 and broadcast by the host. */
int amg1d_nccl_unique_id(void* id128);
int amg1d_create_dist(amg1d_t** h, int n_levels, int device, void* stream, int rank, int nranks,
                      const void* nccl_id);

/* ---- per-level upload ------------------------------------------------------------------------
 * mStiffness[l] as block-tridiagonal blocks plus mSmoothers[l] as explicit inverse blocks:
 *   A_lo[e] couples element e to e-1 (A_lo[0] must be 0), A_di[e] is the diagonal block,
 *   A_up[e] couples e to e+1 (A_up[n-1] must be 0); each array n_elem*m*m doubles.
 *   Dinv: inverse of the smoother block - n_elem*m*m doubles (BlockJacobi, src/smoother.jl:64-81,
 *   :154-164) or, with dinv_is_diagonal = 1, n_elem*m reciprocals of diag(A) (JacobiSmoother,
 *   src/smoother.jl:52-58, :92-98).
 *   perm: NULL when device slot s holds host DOF s (DG / agglomerated levels); otherwise n_elem*m
 *   entries mapping device slot -> host DOF, -1 for a padding slot (CG levels, whose vertex-first
 *   numbering, src/cg_mesh.jl:35-45, is regrouped into [vertex_k, interior_k] blocks).
 *   n_dof_host: length of the reference's vectors on this level (size(mStiffness[l], 1)). */
int amg1d_set_level(amg1d_t* h, int level, int64_t n_elem, int m, const double* A_lo,
                    const double* A_di, const double* A_up, const double* Dinv,
                    int dinv_is_diagonal, const int64_t* perm, int64_t n_dof_host);

/* ---- device-side set-up of the DG-type level chain (SURVEY 8f-1) -------------------------------------
 * Instead of mStiffness[l] and its smoother, the host hands over what the assembly produces - the flux
 * operators G, D, C of the level (block tridiagonal in the element grouping, blocks as in
 * amg1d_set_level) and the inverse element mass matrices Minv (n_elem*m*m, or ONE m*m block for all
 * elements with minv_is_constant = 1) - and the library forms, on the GPU,
 *     A = C - D M^-1 G                       (src/mesh_heirarchy.jl:85-86, :100-101, :172-173)
 * and the block-Jacobi inverses of its diagonal blocks (src/smoother.jl:154-164).  The level is then set
 * exactly as after amg1d_set_level with a block smoother.  The flux operators stay on the device until
 * amg1d_finalize so that amg1d_coarsen_level can project them. */
int amg1d_set_level_flux(amg1d_t* h, int level, int64_t n_elem, int m, const double* G_lo,
                         const double* G_di, const double* G_up, const double* D_lo, const double* D_di,
                         const double* D_up, const double* C_lo, const double* C_di, const double* C_up,
                         const double* Minv, int minv_is_constant);

/* Galerkin coarsening on the GPU: level + 1 <- level.  Needs the flux operators of `level` (from
 * amg1d_set_level_flux or an earlier amg1d_coarsen_level) and transfer `level` (single parent,
 * parent[e] = e / ratio: dg_dg / aggdg_dg / aggdg_aggdg).  Computes G, D, C <- L' (G, D, C) L
 * (src/mesh_heirarchy.jl:75-84, :89-99, :160-171), then A and the smoother of level + 1 as above with the
 * coarse elements' inverse mass matrices Minv_coarse. */
int amg1d_coarsen_level(amg1d_t* h, int level, const double* Minv_coarse, int minv_is_constant);

/* Galerkin coarsening of the stiffness matrix itself on the GPU: level + 1 <- level,
 *     mStiffness[level + 1] = L' mStiffness[level] L
 * - the CG loop of the reference's first constructor (src/mesh_heirarchy.jl:52-60, cg_cg_interpolation)
 * and any other level whose operator is the plain triple product.  `level` must be set (by any of the
 * set / coarsen calls), transfer `level` may have one parent or two (P1: cg_cg / dg_cg / aggdg_cg) and
 * an explicit or a closed-form parent map.  The library verifies that the product is block tridiagonal
 * in the coarse grouping (AMG1D_ERR_ARG otherwise) and builds the smoother of the coarse level from its
 * diagonal: reciprocals (dinv_is_diagonal = 1: JacobiSmoother, cg_smoother(:jac), src/smoother.jl:92-98)
 * or block inverses (0: BlockJacobi, :154-164).  n_coarse_elem: element blocks of the coarse level (for
 * a CG level in [vertex_k, interior_k] grouping: elements + 1); perm_coarse / n_dof_host_coarse as perm /
 * n_dof_host of amg1d_set_level (padding slots, perm = -1, get the identity). */
int amg1d_coarsen_level_galerkin(amg1d_t* h, int level, int64_t n_coarse_elem, int dinv_is_diagonal,
                                 const int64_t* perm_coarse, int64_t n_dof_host_coarse);

/* Download of a level as the element-block arrays of amg1d_set_level (A_lo, A_di, A_up: n_elem*m*m each;
 * Dinv: n_elem*m*m or n_elem*m) - for checking device-side set-up and for scripts that inspect
 * H.mStiffness[k] of a level the host never assembled. */
int amg1d_get_level(amg1d_t* h, int level, double* A_lo, double* A_di, double* A_up, double* Dinv);

/* Replaces the smoother of a level that has been set by a block-TRIDIAGONAL smoother operator S:
 * z = S r with S r[e] = S_lo[e] r[e-1] + S_di[e] r[e] + S_up[e] r[e+1] (blocks as in amg1d_set_level).
 * This is the form the overlapping Schwarz smoothers of CG levels take in the [vertex_k, interior_k]
 * grouping (AdditiveSchwarzSmoother / HybridSchwarzSmoother, src/smoother.jl:1-46, built by
 * cg_smoother(:addSchwarz / :hybridSchwarz), :104-135): an element's local solve touches its own group
 * and the first slot of the next one.  Such levels smooth with the generic (unfused) kernels. */
int amg1d_set_level_smoother(amg1d_t* h, int level, const double* S_lo, const double* S_di,
                             const double* S_up);

/* Same operator given as a translation-invariant pattern (uniform meshes at 2^20..2^26 elements,
 * where per-element host arrays would be tens of GB): the first n_head and last n_tail elements are
 * explicit, every element in between repeats the single `interior` block set.  Arrays hold
 * n_head + 1 + n_tail blocks in that order.  The device still stores every element's blocks (the
 * general layout, which every kernel can read) and keeps the n_head + 1 + n_tail block sets as a small
 * table next to them; with option "pattern_resident" = 1 or 2 the fused legs read the table (2: kernel
 * parameters in the interior of the level) instead of the per-element blocks (same numbers, same
 * arithmetic order: bit-identical iterates), so HBM carries only the vectors. */
int amg1d_set_level_pattern(amg1d_t* h, int level, int64_t n_elem, int m, int n_head, int n_tail,
                            const double* A_lo, const double* A_di, const double* A_up,
                            const double* Dinv, int dinv_is_diagonal);

/* mInterpolation[l] (prolongation from level l+1 to level l; restriction is its transpose,
 * src/solvers.jl:36,42) as element-local blocks: fine element e has parent element parent[e]
 * (non-decreasing) and
 *     x_f[e] += P0[e] * x_c[parent[e]]  (+ P1[e] * x_c[parent[e]+1] when P1 != NULL)
 * with m_f x m_c column-major blocks, n_fine_elem of them per array.  P1 carries the second parent of
 * the CG-type transfers (cg_cg / dg_cg / aggdg_cg, src/interpolation.jl:33-52, :158-216, :340-406),
 * NULL for dg_dg / aggdg_dg / aggdg_aggdg (:91-109, :226-292). */
int amg1d_set_transfer(amg1d_t* h, int level, int64_t n_fine_elem, int m_f, int m_c,
                       const int64_t* parent, const double* P0, const double* P1);

/* parent[e] may be -1 and parent[e] + 1 may equal the coarse element count: both address ghost
 * elements that hold zeros (the matching P block must be zero).
 *
 * Pattern form for uniform meshes: parent[e] = (e + shift) / ratio + base, and the block of element
 * e is   P_pat[e]                                       for e <  n_head,
 *        P_pat[n_head + (e - n_head) % period]          in between,
 *        P_pat[n_head + period + e - (n - n_tail)]      for e >= n - n_tail
 * (n_head + period + n_tail blocks per array; P1_pat NULL for single-parent transfers). */
int amg1d_set_transfer_pattern(amg1d_t* h, int level, int64_t n_fine_elem, int m_f, int m_c,
                               int ratio, int shift, int base, int period, int n_head, int n_tail,
                               const double* P0_pat, const double* P1_pat);

/* Allocates work vectors, factorises the coarsest level (block Thomas; replaces the sparse direct
 * solve of src/solvers.jl:39) and validates that the hierarchy is complete. */
int amg1d_finalize(amg1d_t* h);

/* ---- the hot path ----------------------------------------------------------------------------
 * multigrid_v_cycle(H, x0, b; nPre, nPost, alpha) - src/solvers.jl:19-50.  x: in x0, out x. */
int amg1d_vcycle(amg1d_t* h, double* x, const double* b, int nPre, int nPost, double alpha);

/* multigrid(H, x0, b, maxiter, tol) - src/solvers.jl:116-139.  res / err: maxiter doubles (err and
 * u_exact may be NULL: the reference computes u_exact = A \ b itself, here the host supplies it).
 * The reference always cycles with nPre = nPost = 3, alpha = 2/3; they are arguments here. */
int amg1d_solve(amg1d_t* h, double* x, const double* b, int maxiter, double tol, int nPre,
                int nPost, double alpha, int* iters, double* res, double* err,
                const double* u_exact);

/* ldiv!(y, H, b) / ldiv!(H, b) - src/solvers.jl:63-92: one V-cycle from a ZERO guess, y <- result (y may
 * alias b).  Unlike amg1d_vcycle no initial guess is uploaded, and the first pre-smoothing sweep of
 * the finest level skips the operator (x = alpha Dinv b), exactly as the levels below always do. */
int amg1d_ldiv(amg1d_t* h, double* y, const double* b, int nPre, int nPost, double alpha);

/* The same V-cycle on `count` independent problems, pipelined over PCIe: problem k + 1 is uploaded and the
 * iterate of problem k - 1 downloaded on two copy streams while problem k runs (one amg1d_vcycle call is bound
 * by its three serial vector transfers; PCIe is full duplex).  x[k]: in = initial guess, ignored with zero_guess
 * = 1 (the ldiv! form: x0 = 0 is neither uploaded nor read), out = the iterate; b[k]: right-hand side.  Host
 * vectors should be pinned (amg1d_host_alloc).  Bit-identical to `count` amg1d_vcycle / amg1d_ldiv calls. */
int amg1d_vcycle_batch(amg1d_t* h, int count, double* const* x, const double* const* b, int zero_guess,
                       int nPre, int nPost, double alpha);

/* Conjugate gradients on the finest level, preconditioned with ldiv!(z, H, r) - what the reference's
 * ldiv! methods exist for (src/solvers.jl:63-92 make MeshHierarchy usable as `Pl` of a Krylov solver
 * such as IterativeSolvers.cg; the reference ships no driver for it).  Textbook PCG: z = M^-1 r,
 * beta = r.z / (r.z)_old, p = z + beta p, alpha = r.z / p.Ap, x += alpha p, r -= alpha Ap; res[i] =
 * ||r_i||_2 of the recurrence residual; stops when res[i] < tol * ||b||_2 (the rule of multigrid()).
 * x: in x0, out x; res: maxiter doubles.  The V-cycle with nPre == nPost is a symmetric operator. */
int amg1d_pcg(amg1d_t* h, double* x, const double* b, int maxiter, double tol, int nPre, int nPost,
              double alpha, int* iters, double* res);

/* apply_smoother(S, B; alpha) - src/smoother.jl:52-58, :69-81.  Y = alpha * S^-1 * B, B and Y are
 * n_dof_host x n_rhs column-major (the scripts also pass matrices, tests/dg_smoother_test.jl:105). */
int amg1d_apply_smoother(amg1d_t* h, int level, double* Y, const double* B, int64_t n_rhs,
                         double alpha);

/* iterative_smoother_solve(A, smoother, x0, b; maxiter, tol, alpha) - src/solvers.jl:189-213. */
int amg1d_smoother_solve(amg1d_t* h, int level, double* x, const double* b, int maxiter, double tol,
                         double alpha, int* iters, double* res, double* err, const double* u_exact);

/* The stdlib operations the scripts use directly on hierarchy members:
 *   amg1d_matvec        y  = mStiffness[l] * x
 *   amg1d_residual      r  = b - mStiffness[l] * x          (src/solvers.jl:33)
 *   amg1d_restrict      rc = mInterpolation[l]' * rf        (src/solvers.jl:36)
 *   amg1d_prolong       xf = mInterpolation[l] * xc         (src/solvers.jl:42, without the add)
 *   amg1d_coarse_solve  x  = mStiffness[end] \ b            (src/solvers.jl:39) */
int amg1d_matvec(amg1d_t* h, int level, double* y, const double* x);
int amg1d_residual(amg1d_t* h, int level, double* r, const double* x, const double* b);
int amg1d_restrict(amg1d_t* h, int level, double* rc, const double* rf);
int amg1d_prolong(amg1d_t* h, int level, double* xf, const double* xc);
int amg1d_coarse_solve(amg1d_t* h, double* x, const double* b);

/* x = mStiffness[l] \ b for ANY level: the sparse direct solves the reference uses for error histories
 * (u_exact = A \ b, src/solvers.jl:120, :194) and for the coarsest level (:39).  Block cyclic reduction
 * on the GPU; the level is factorised at the first call (about 10 n m^2 doubles of device memory) and
 * the factors are kept.  The coarsest level of the V-cycle itself is solved the same way when it has
 * more than 64 elements (a serial block-Thomas kernel below that). */
int amg1d_direct_solve(amg1d_t* h, int level, double* x, const double* b);

/* ---- device-resident path (no host copies; what bench.py times as `value`) --------------------
 * The problem (x, b on level 0) stays on the device between calls.  The per-level host operations above
 * stage their operands in the levels' own vectors: amg1d_residual and amg1d_smoother_solve on level 0 and
 * amg1d_pcg overwrite the resident right-hand side.  After one of them the amg1d_dev_vcycle /
 * amg1d_dev_residual_norm / amg1d_dev_rhs_norm calls return AMG1D_ERR_STATE until amg1d_dev_set_problem
 * (with b != NULL) or amg1d_dev_fill_rhs_random installs a problem again; amg1d_vcycle / amg1d_solve /
 * amg1d_ldiv upload their own vectors and are not affected. */
int amg1d_dev_set_problem(amg1d_t* h, const double* x0, const double* b); /* host -> device, x0 NULL = 0 */
int amg1d_dev_fill_rhs_random(amg1d_t* h, uint64_t seed);          /* b[i] ~ U(-1,1) on the device, x = 0 */
/* Right-hand side assembled ON THE DEVICE (SURVEY 8f-3): the volume integrals of dg_flux_rhs
 * (src/dg_mesh.jl:342-365) - kind 0, level 0 a DG-type level - or of cg_stiffness_and_rhs / cg_rhs
 * (src/cg_mesh.jl:150-160, :205-215) - kind 1, level 0 a CG level uploaded in group order - for
 *     func(x) = sum_t coef_t x^pow_t g_t(w_t x + phi_t),   g = 1 | cos | sin | exp
 * (terms: 5 doubles per term: kind 0 / 1 / 2 / 3, coef, pow (integer 0..16), w, phi), integrated with the
 * host's quadrature: xi (nq reference nodes) and W (nq x n_basis row-major, W[q][i] = w_q phi_i(xi_q),
 * n_basis = p + 1).  Elements are those of the reference's mesh generator (tests/mesh_generator.jl:20-32:
 * x_i = xin + (i / n)(xout - xin)) or, if `vertices` is not NULL, [vertices[e], vertices[e + 1]] (n + 1 doubles).
 * The boundary terms of the reference (flux / penalty terms at the two end elements, Neumann data, strong
 * Dirichlet rows) are a handful of entries the host computes and passes as a fix list, applied in order:
 * fix_op[k] = 0: b[fix_slot[k]] += fix_val[k]; 1: b[fix_slot[k]] = fix_val[k]; fix_slot are GLOBAL level-0 slots.
 * Sharded handles assemble their own slab (and its ghost elements).  x is set to 0. */
int amg1d_dev_assemble_rhs(amg1d_t* h, int kind, int nq, const double* xi, const double* W, int n_basis,
                           int n_terms, const double* terms, double xin, double xout, const double* vertices,
                           int n_fix, const int64_t* fix_slot, const double* fix_val, const int* fix_op);
int amg1d_dev_get_rhs(amg1d_t* h, double* b);                      /* device -> host (this rank's slab) */
/* multigrid(H, x0, b, maxiter, tol) (src/solvers.jl:116-139) on the device-resident problem: no host vector
 * moves; res[i] = ||A x - b||_2 after cycle i + 1; the solution stays on the device (amg1d_dev_get_solution). */
int amg1d_dev_solve(amg1d_t* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters,
                    double* res);
/* amg1d_pcg on the device-resident problem (initial guess = the resident iterate); the solution becomes the
 * resident iterate, the resident right-hand side is consumed (it becomes the CG residual). */
int amg1d_dev_pcg(amg1d_t* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters,
                  double* res);
/* asynchronous on the stream; with_residual_norm = 1 also leaves ||A x - b||_2 of the new iterate on the
 * device (fused into the last kernel of the cycle), which amg1d_dev_residual_norm then just reads */
int amg1d_dev_vcycle(amg1d_t* h, int nPre, int nPost, double alpha, int with_residual_norm);
int amg1d_dev_residual_norm(amg1d_t* h, double* res);              /* ||A x - b||_2, synchronises */
int amg1d_dev_rhs_norm(amg1d_t* h, double* nb);                    /* ||b||_2, synchronises */
int amg1d_dev_get_solution(amg1d_t* h, double* x);                 /* device -> host */

/* ---- multi-column device-resident problems ----------------------------------------------------------
 * ldiv!(Y, H, B) / multigrid_v_cycle / multigrid (src/solvers.jl:19-50, :63-92, :116-139) for k <= AMG1D_MAX_COLS
 * right-hand sides at once: the reference's ldiv! methods make MeshHierarchy a preconditioner, which block Krylov
 * methods, time steppers and multi-load problems apply to many vectors.  One V-cycle serves all columns: on levels
 * with fused legs (amg1d_get_info("multi_legs:<level>") = 1) each leg reads the level's operator once for all columns;
 * the other levels, the coarse tail and the coarse solve run once per column.  Every column's iterate and residual
 * norm are bit-identical to the single-column calls on that column.  Single GPU handles only (AMG1D_ERR_UNSUPPORTED
 * otherwise).  The column set is separate device storage (three vectors per level and column, counted in
 * "device_bytes", allocated at the first call and grown when k grows): the single-column resident problem of
 * amg1d_dev_set_problem is neither read nor written by these calls, nor the column set by that one.  X0, B, X are
 * n_dof_host x k column-major (level 0's host vector length); X0 == NULL: zero initial guesses. */
#define AMG1D_MAX_COLS 8
int amg1d_dev_set_problems(amg1d_t* h, int k, const double* X0, const double* B);   /* host -> device */
/* column c gets exactly the b of amg1d_dev_fill_rhs_random(h, seed + c); x = 0 */
int amg1d_dev_fill_rhs_random_multi(amg1d_t* h, int k, uint64_t seed);
/* one V-cycle on every column, asynchronous; zero_guess = 1: the ldiv! form of amg1d_ldiv (x0 = 0, not read, the first
 * pre-smoothing sweep skips A); with_residual_norms = 1 leaves ||b - A x||_2 of every column on the device */
int amg1d_dev_vcycle_multi(amg1d_t* h, int nPre, int nPost, double alpha, int zero_guess, int with_residual_norms);
int amg1d_dev_residual_norms(amg1d_t* h, double* res);             /* k values ||b - A x||_2, synchronises */
/* multigrid() per column: iters (k ints), res (maxiter x k, column-major).  A column that meets its own stop rule
 * leaves the set of cycled columns, so its iterate, iters[c] and res history equal amg1d_dev_solve on it alone. */
int amg1d_dev_solve_multi(amg1d_t* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters,
                          double* res);
/* amg1d_dev_pcg on every column of the multi-column set: iters (k ints), res (maxiter x k, column-major).
 * Initial guess = the column's resident iterate; the solution becomes it; the column's right-hand side is consumed
 * (it becomes the CG residual).  Every column's iters[c], res history and solution are bit-identical to
 * amg1d_dev_pcg on it alone; a column that meets its stop rule (or whose residual turns non-finite) leaves the set of
 * cycled columns, one with b = 0 or an x0 that already solves it never enters it.  AMG1D_ERR_ARG for a non-finite
 * column before the first iteration, and after the others finished for a column that broke down (the message names
 * the column).  Afterwards amg1d_dev_vcycle_multi / _residual_norms / _solve_multi / _pcg_multi return
 * AMG1D_ERR_STATE until a set is installed again; amg1d_dev_get_solutions returns the solutions.  The per-column CG
 * vectors (three level-0 vectors) are allocated at the first call and grown with k.  The product A p reads level
 * 0's operator once for all columns, and the CG updates and reductions run one launch for all columns. */
int amg1d_dev_pcg_multi(amg1d_t* h, int maxiter, double tol, int nPre, int nPost, double alpha, int* iters,
                        double* res);
int amg1d_dev_get_solutions(amg1d_t* h, double* X);                /* device -> host, n_dof_host x k */

int amg1d_synchronize(amg1d_t* h);
void* amg1d_stream(amg1d_t* h);                                    /* the cudaStream_t in use */
void* amg1d_dev_ptr(amg1d_t* h, int level, int which);             /* raw device pointer (AMG1D_VEC_*) */

/* ---- options and introspection ------------------------------------------------------------------
 * amg1d_set_option keys: "fused" (1 = fused multi-sweep kernels where available, default 1),
 * "graph" (1 = replay the V-cycle as a CUDA graph, default 1), "pdl" (1 = programmatic dependent
 * launch between the fused kernels, default 1), "coarse_cta_elems" (levels with at most this many
 * elements - capped at 512 - run inside the single-CTA coarse kernel; 0 disables it; default 1024),
 * "profile" (see amg1d_get_profile; setting it clears earlier samples), "pattern_resident" (1 = levels
 * given by amg1d_set_level_pattern take their operator from the pattern table; 2 = in addition the CTAs
 * whose elements all lie in the translation-invariant interior of such a level receive the interior block
 * set as a kernel parameter and use it as constant operands; default 0; bit-identical results in all modes),
 * "rows_window" (elements per CTA of the row-per-thread legs for 5..9-row blocks: 32, 64; 0 = off;
 * default 64), "rows_per_thread" (block rows per thread of those legs: 1, 2, 3; 0 = auto, default);
 * "recompute_dinv" (default 4 = levels with 4 x 4 blocks; v = blocks of v x v up to "recompute_dinv_max" (default
 * 4, at most 5 - larger and smaller blocks were measured slower); 0 = never.  Where non-zero when a level is
 * set, its block-Jacobi inverses - if the uploaded Dinv agrees with inv(A_di) to 1e-8 - are replaced by the
 * device's own Gauss-Jordan inverse of the stored diagonal blocks (without pivoting when every element of the level
 * that would swap rows gets the same inverse to 1e-12 without - the DG blocks of the reference; else with partial
 * pivoting), so that the fused legs can invert A_di in registers instead of streaming the stored inverse from HBM
 * while every other kernel, which reads the stored inverse, produces the same bits.  Changing the value later only
 * selects which levels recompute - same results, other byte counts);
 * "leg_pipeline" (default 1: the recomputing legs of 4 x 4 levels run as persistent CTAs that fetch their next
 * window with TMA bulk copies while they compute the current one - f_down_pp / f_up_pp - on levels of at least
 * "leg_pipeline_min" elements per rank (default 500000); 2: the 2 x 2 levels too; 0: one window per CTA), "dinv_registers" (with "leg_pipeline" = 0: 1 = the recomputed inverse of 4 x 4 levels
 * stays in registers - f_down_dv / f_up_dv; 2 = of 2 x 2 levels too; 0 = it goes through shared memory) - every
 * combination gives the same bits;
 * "p2p_halo" (before amg1d_finalize, multi-GPU handles; default 1: the slab-edge exchanges of the V-cycle go
 * through CUDA-IPC peer memory over NVLink - two small kernels per exchange - instead of NCCL send / recv groups;
 * falls back to NCCL, on every rank alike, if the peer mapping is refused; amg1d_get_info("p2p_halo") tells
 * which one is active; bit-identical results);
 * before the first level is
 * set: "compress" (1 = store only the structurally non-zero column / row of the off-diagonal blocks
 * where every element of the level has that structure, default 1), "shard_min" (elements per rank
 * below which a level is gathered to rank 0, default 8192), "ghost_depth" (ghost elements per slab
 * edge, default 4 = max(nPre, nPost) + 1; CG levels with two-parent transfers need + ratio). */
int amg1d_set_option(amg1d_t* h, const char* key, int64_t value);
int64_t amg1d_get_info(amg1d_t* h, const char* key); /* "kernel_launches", "launches_per_cycle",
                                                        "device_bytes", "n_levels", "local_elements",
                                                        "local_dofs", "gather_level", "tail_start",
                                                        "ghost_depth", "structure:<level>",
                                                        "tile_rows:<level>", "dinv_recompute:<level>" (1 = the fused
                                                        legs of the level invert A_di in registers),
                                                        "leg_pipeline:<level>" (1 = they are the persistent
                                                        pipelined legs), "dinv_pivots:<level>" (1 = that
                                                        inversion keeps the partial-pivoting chain),
                                                        "pattern:<level>" (1 = the
                                                        level has a pattern table), "multi_columns"
                                                        (k of the multi-column set, 0: none),
                                                        "multi_legs:<level>" (1 = the multi-column
                                                        cycle reads the level's operator once for all
                                                        columns), "multi_launches_per_cycle",
                                                        "multi_pcg_launches_per_iteration" (launches
                                                        of the last amg1d_dev_pcg_multi iteration
                                                        outside its V-cycle),
                                                        the option keys,
                                                        ... (-1: unknown key) */

/* With option "profile" = 1 every V-cycle runs un-graphed and brackets each level's down leg (leg 0:
 * pre-smoothing + residual + restriction) and up leg (leg 1: prolongation + post-smoothing) with CUDA
 * events on the handle's stream; this returns the summed device time and the number of brackets. */
int amg1d_get_profile(amg1d_t* h, int level, int leg, double* total_ms, int* launches);

/* Pinned host memory helpers for callers that want asynchronous, full-bandwidth copies. */
int amg1d_host_alloc(void** p, int64_t bytes);
int amg1d_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* AMG1D_H */
