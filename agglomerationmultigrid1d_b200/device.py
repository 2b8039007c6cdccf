"""Python owner of one libamg1d handle: uploads a host-assembled hierarchy and exposes the
hot-path calls.  Thin by design - every numerical operation happens inside libamg1d.so.
"""
import ctypes as C

import numpy as np

from . import _capi as capi
from . import blocks as blk


class DeviceHierarchy:
    def __init__(self, n_levels, device=0, stream=None, dist=None):
        """dist: None or (rank, nranks, nccl_id_bytes) for the slab-sharded variant."""
        self._lib = capi.load()
        self._h = C.c_void_p()
        self.n_levels = n_levels
        self.n_dof = [0] * n_levels
        if dist is None:
            rc = self._lib.amg1d_create(C.byref(self._h), n_levels, device, stream)
        else:
            rank, nranks, nid = dist
            buf = C.create_string_buffer(bytes(nid), 128)
            rc = self._lib.amg1d_create_dist(C.byref(self._h), n_levels, device, stream, rank,
                                             nranks, C.cast(buf, C.c_void_p))
        capi.check(None, rc)

    # ---- life cycle ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.amg1d_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        capi.check(self._h, rc)

    # ---- upload -------------------------------------------------------------------------------
    def set_level_blocks(self, level, lo, di, up, dinv, dinv_is_diagonal, slots=None, n_dof=None):
        """lo / di / up: (n, m, m) in (e, i, j) order; dinv already in ABI layout."""
        n, m = di.shape[0], di.shape[1]
        perm = None
        if slots is not None and not blk.is_identity_slots(slots):
            perm = capi.i64(slots.ravel())
        if n_dof is None:
            n_dof = n * m
        self.n_dof[level] = int(n_dof)
        a_lo, a_di, a_up = blk.to_abi(lo), blk.to_abi(di), blk.to_abi(up)
        dinv = capi.f64(dinv)
        self._ck(self._lib.amg1d_set_level(self._h, level, n, m, capi.dptr(a_lo), capi.dptr(a_di),
                                           capi.dptr(a_up), capi.dptr(dinv), int(dinv_is_diagonal),
                                           capi.iptr(perm), int(n_dof)))

    def set_level_flux(self, level, G, D, C, minv):
        """Device-side set-up of a level from its flux operators: G, D, C are (lo, di, up) triples of
        (n, m, m) blocks in (e, i, j) order, minv the (n, m, m) inverse mass blocks (or one (m, m) block)."""
        n, m = G[1].shape[0], G[1].shape[1]
        arrs = [blk.to_abi(a) for X in (G, D, C) for a in X]
        const = minv.ndim == 2
        mi = blk.to_abi(minv[None] if const else minv)
        self.n_dof[level] = n * m
        self._ck(self._lib.amg1d_set_level_flux(self._h, level, n, m, *[capi.dptr(a) for a in arrs],
                                                capi.dptr(mi), int(const)))

    def coarsen_level(self, level, minv_coarse, n_coarse):
        """level + 1 <- Galerkin coarsening of level on the GPU (transfer `level` must be set)."""
        const = minv_coarse.ndim == 2
        mi = blk.to_abi(minv_coarse[None] if const else minv_coarse)
        self.n_dof[level + 1] = int(n_coarse) * mi.shape[1]
        self._ck(self._lib.amg1d_coarsen_level(self._h, level, capi.dptr(mi), int(const)))

    def coarsen_level_galerkin(self, level, slots_coarse, n_dof_coarse, dinv_is_diagonal=True):
        """level + 1 <- L' A L of level's stiffness matrix on the GPU (one- or two-parent transfer `level`
        must be set): the CG loop of the reference's first constructor.  slots_coarse: the coarse
        level's (element block, row) -> host DOF map (blocks.level_slots)."""
        perm = None if blk.is_identity_slots(slots_coarse) else capi.i64(slots_coarse.ravel())
        self.n_dof[level + 1] = int(n_dof_coarse)
        self._ck(self._lib.amg1d_coarsen_level_galerkin(self._h, level, int(slots_coarse.shape[0]),
                                                        int(dinv_is_diagonal), capi.iptr(perm),
                                                        int(n_dof_coarse)))

    def get_level(self, level, n, m, diag=False):
        """(lo, di, up) as (n, m, m) blocks in (e, i, j) order and Dinv ((n, m, m), or (n, m) if diag)."""
        out = [np.zeros((n, m, m)) for _ in range(3)]
        dinv = np.zeros((n, m) if diag else (n, m, m))
        self._ck(self._lib.amg1d_get_level(self._h, level, *[capi.dptr(a) for a in out], capi.dptr(dinv)))
        tr = lambda a: np.ascontiguousarray(np.transpose(a, (0, 2, 1)))      # noqa: E731  ABI is column-major
        return tr(out[0]), tr(out[1]), tr(out[2]), (dinv if diag else tr(dinv))

    def set_level_smoother(self, level, s_lo, s_di, s_up):
        """Block-tridiagonal smoother operator of a level (Schwarz smoothers); (n, m, m) arrays in (e, i, j) order."""
        a_lo, a_di, a_up = blk.to_abi(s_lo), blk.to_abi(s_di), blk.to_abi(s_up)
        self._ck(self._lib.amg1d_set_level_smoother(self._h, level, capi.dptr(a_lo), capi.dptr(a_di),
                                                    capi.dptr(a_up)))

    def set_level_pattern(self, level, n_elem, lo, di, up, dinv, dinv_is_diagonal, n_head, n_tail):
        m = di.shape[1]
        self.n_dof[level] = int(n_elem) * m
        a_lo, a_di, a_up = blk.to_abi(lo), blk.to_abi(di), blk.to_abi(up)
        dinv = capi.f64(dinv)
        self._ck(self._lib.amg1d_set_level_pattern(self._h, level, int(n_elem), m, n_head, n_tail,
                                                   capi.dptr(a_lo), capi.dptr(a_di), capi.dptr(a_up),
                                                   capi.dptr(dinv), int(dinv_is_diagonal)))

    def set_transfer_blocks(self, level, parent, P0, P1=None):
        nf, mf, mc = P0.shape
        p0 = blk.to_abi(P0)
        p1 = blk.to_abi(P1) if P1 is not None else None
        par = capi.i64(parent)
        self._ck(self._lib.amg1d_set_transfer(self._h, level, nf, mf, mc, capi.iptr(par),
                                              capi.dptr(p0), capi.dptr(p1)))

    def set_transfer_pattern(self, level, n_fine, P0, P1=None, ratio=1, shift=0, base=0, period=1,
                             n_head=0, n_tail=0):
        _, mf, mc = P0.shape
        p0 = blk.to_abi(P0)
        p1 = blk.to_abi(P1) if P1 is not None else None
        self._ck(self._lib.amg1d_set_transfer_pattern(self._h, level, int(n_fine), mf, mc, ratio,
                                                      shift, base, period, n_head, n_tail,
                                                      capi.dptr(p0), capi.dptr(p1)))

    def finalize(self):
        self._ck(self._lib.amg1d_finalize(self._h))

    # ---- hot path -------------------------------------------------------------------------------
    def vcycle(self, x0, b, nPre=3, nPost=3, alpha=2.0 / 3.0):
        x = np.array(x0, dtype=np.float64, order="C", copy=True)
        b = capi.f64(b)
        self._check_len(0, x, b)
        self._ck(self._lib.amg1d_vcycle(self._h, capi.dptr(x), capi.dptr(b), nPre, nPost, alpha))
        return x

    def solve(self, x0, b, maxiter, tol, nPre=3, nPost=3, alpha=2.0 / 3.0, u_exact=None):
        x = np.array(x0, dtype=np.float64, order="C", copy=True)
        b = capi.f64(b)
        self._check_len(0, x, b)
        res = np.zeros(max(maxiter, 1))
        err = np.zeros(max(maxiter, 1))
        it = C.c_int(0)
        ue = capi.f64(u_exact) if u_exact is not None else None
        self._ck(self._lib.amg1d_solve(self._h, capi.dptr(x), capi.dptr(b), maxiter, tol, nPre, nPost,
                                       alpha, C.byref(it), capi.dptr(res), capi.dptr(err),
                                       capi.dptr(ue)))
        return x, it.value, res[:it.value].copy(), err[:it.value].copy()

    def ldiv(self, b, nPre=3, nPost=3, alpha=2.0 / 3.0):
        b = capi.f64(b)
        self._check_len(0, b)
        y = np.zeros_like(b)
        self._ck(self._lib.amg1d_ldiv(self._h, capi.dptr(y), capi.dptr(b), nPre, nPost, alpha))
        return y

    def vcycle_batch(self, xs, bs, zero_guess=False, nPre=3, nPost=3, alpha=2.0 / 3.0):
        """One V-cycle per (x, b) pair, pipelined over PCIe (amg1d_vcycle_batch).  xs: list of C-contiguous float64
        arrays, overwritten with the iterates (pinned memory overlaps the copies with the compute); bs likewise."""
        n = len(xs)
        assert len(bs) == n
        for v in list(xs) + list(bs):
            self._check_len(0, v)
            assert v.dtype == np.float64 and v.flags["C_CONTIGUOUS"]
        PD = C.POINTER(C.c_double)
        xa = (PD * n)(*[v.ctypes.data_as(PD) for v in xs])
        ba = (PD * n)(*[v.ctypes.data_as(PD) for v in bs])
        self._ck(self._lib.amg1d_vcycle_batch(self._h, n, xa, ba, int(bool(zero_guess)), nPre, nPost, alpha))
        return xs

    def pcg(self, x0, b, maxiter, tol, nPre=3, nPost=3, alpha=2.0 / 3.0):
        x = np.array(x0, dtype=np.float64, order="C", copy=True)
        b = capi.f64(b)
        self._check_len(0, x, b)
        res = np.zeros(max(maxiter, 1))
        it = C.c_int(0)
        self._ck(self._lib.amg1d_pcg(self._h, capi.dptr(x), capi.dptr(b), maxiter, tol, nPre, nPost, alpha,
                                     C.byref(it), capi.dptr(res)))
        return x, it.value, res[:it.value].copy()

    def apply_smoother(self, level, B, alpha=1.0):
        B = np.asarray(B, dtype=np.float64)
        vec = B.ndim == 1
        Bf = np.asfortranarray(B.reshape(B.shape[0], -1))
        if Bf.shape[0] != self.n_dof[level]:
            raise ValueError("DimensionMismatch")
        Y = np.zeros(Bf.shape, order="F")
        self._ck(self._lib.amg1d_apply_smoother(
            self._h, level, Y.ctypes.data_as(C.POINTER(C.c_double)),
            Bf.ctypes.data_as(C.POINTER(C.c_double)), Bf.shape[1], alpha))
        return Y[:, 0].copy() if vec else np.ascontiguousarray(Y)

    def smoother_solve(self, level, x0, b, maxiter=1000, tol=1e-6, alpha=1.0, u_exact=None):
        x = np.array(x0, dtype=np.float64, order="C", copy=True)
        b = capi.f64(b)
        self._check_len(level, x, b)
        res = np.zeros(max(maxiter, 1))
        err = np.zeros(max(maxiter, 1))
        it = C.c_int(0)
        ue = capi.f64(u_exact) if u_exact is not None else None
        self._ck(self._lib.amg1d_smoother_solve(self._h, level, capi.dptr(x), capi.dptr(b), maxiter,
                                                tol, alpha, C.byref(it), capi.dptr(res),
                                                capi.dptr(err), capi.dptr(ue)))
        return x, it.value, res[:it.value].copy(), err[:it.value].copy()

    def _check_len(self, level, *vecs):
        for v in vecs:
            if v.shape != (self.n_dof[level],):
                raise ValueError(f"DimensionMismatch: expected length {self.n_dof[level]}, got {v.shape}")

    def matvec(self, level, x):
        x = capi.f64(x); self._check_len(level, x)
        y = np.zeros_like(x)
        self._ck(self._lib.amg1d_matvec(self._h, level, capi.dptr(y), capi.dptr(x)))
        return y

    def residual(self, level, x, b):
        x = capi.f64(x); b = capi.f64(b); self._check_len(level, x, b)
        r = np.zeros_like(x)
        self._ck(self._lib.amg1d_residual(self._h, level, capi.dptr(r), capi.dptr(x), capi.dptr(b)))
        return r

    def restrict(self, level, rf):
        rf = capi.f64(rf); self._check_len(level, rf)
        rc = np.zeros(self.n_dof[level + 1])
        self._ck(self._lib.amg1d_restrict(self._h, level, capi.dptr(rc), capi.dptr(rf)))
        return rc

    def prolong(self, level, xc):
        xc = capi.f64(xc); self._check_len(level + 1, xc)
        xf = np.zeros(self.n_dof[level])
        self._ck(self._lib.amg1d_prolong(self._h, level, capi.dptr(xf), capi.dptr(xc)))
        return xf

    def coarse_solve(self, b):
        b = capi.f64(b); self._check_len(self.n_levels - 1, b)
        x = np.zeros_like(b)
        self._ck(self._lib.amg1d_coarse_solve(self._h, capi.dptr(x), capi.dptr(b)))
        return x

    def direct_solve(self, level, b):
        """x = mStiffness[level] \\ b by block cyclic reduction on the GPU (any level, any size)."""
        b = capi.f64(b); self._check_len(level, b)
        x = np.zeros_like(b)
        self._ck(self._lib.amg1d_direct_solve(self._h, level, capi.dptr(x), capi.dptr(b)))
        return x

    # ---- device-resident path -----------------------------------------------------------------
    def dev_set_problem(self, x0, b):
        x0 = capi.f64(x0) if x0 is not None else None
        b = capi.f64(b) if b is not None else None
        self._ck(self._lib.amg1d_dev_set_problem(self._h, capi.dptr(x0), capi.dptr(b)))

    def dev_assemble_rhs(self, kind, xi, W, terms, xin, xout, vertices=None, fixes=()):
        """Right-hand side assembled on the device (amg1d_dev_assemble_rhs).  kind: 0 DG-type level 0, 1 CG level
        0 in group order; xi (nq,), W (nq, p + 1) = w_q phi_i(xi_q); terms: iterable of (kind, coef, pow, w, phi)
        with kind in {"1", "cos", "sin", "exp"} or 0..3; fixes: iterable of (global slot, value, op) with op
        "add" / "set" (the boundary terms, computed by the host)."""
        names = {"1": 0, "const": 0, "cos": 1, "sin": 2, "exp": 3}
        t = np.array([[names.get(k, k) if isinstance(k, str) else k, c, pw, w, ph] for (k, c, pw, w, ph) in terms],
                     dtype=np.float64).reshape(-1, 5)
        xi = capi.f64(xi)
        W = capi.f64(W)
        fs = capi.i64([f[0] for f in fixes])
        fv = capi.f64([f[1] for f in fixes])
        fo = np.ascontiguousarray([1 if f[2] in (1, "set") else 0 for f in fixes], dtype=np.int32)
        vt = capi.f64(vertices) if vertices is not None else None
        self._ck(self._lib.amg1d_dev_assemble_rhs(
            self._h, int(kind), len(xi), capi.dptr(xi), capi.dptr(W), W.shape[1], t.shape[0], capi.dptr(t),
            float(xin), float(xout), capi.dptr(vt), len(fs), capi.iptr(fs) if len(fs) else None,
            capi.dptr(fv) if len(fs) else None, fo.ctypes.data_as(C.POINTER(C.c_int)) if len(fs) else None))

    def dev_get_rhs(self):
        b = np.zeros(self.n_dof[0])
        self._ck(self._lib.amg1d_dev_get_rhs(self._h, capi.dptr(b)))
        return b

    def dev_solve(self, maxiter, tol, nPre=3, nPost=3, alpha=2.0 / 3.0):
        """``multigrid`` on the device-resident problem; returns (iters, res) - the solution stays on the device."""
        res = np.zeros(max(maxiter, 1))
        it = C.c_int(0)
        self._ck(self._lib.amg1d_dev_solve(self._h, maxiter, tol, nPre, nPost, alpha, C.byref(it), capi.dptr(res)))
        return it.value, res[:it.value].copy()

    def dev_pcg(self, maxiter, tol, nPre=3, nPost=3, alpha=2.0 / 3.0):
        """``pcg`` on the device-resident problem; returns (iters, res) - the solution stays on the device."""
        res = np.zeros(max(maxiter, 1))
        it = C.c_int(0)
        self._ck(self._lib.amg1d_dev_pcg(self._h, maxiter, tol, nPre, nPost, alpha, C.byref(it), capi.dptr(res)))
        return it.value, res[:it.value].copy()

    def dev_fill_rhs_random(self, seed=0):
        self._ck(self._lib.amg1d_dev_fill_rhs_random(self._h, seed))

    def dev_vcycle(self, nPre=3, nPost=3, alpha=2.0 / 3.0, with_residual_norm=False):
        self._ck(self._lib.amg1d_dev_vcycle(self._h, nPre, nPost, alpha, int(with_residual_norm)))

    def dev_residual_norm(self):
        v = C.c_double(0.0)
        self._ck(self._lib.amg1d_dev_residual_norm(self._h, C.byref(v)))
        return v.value

    def dev_rhs_norm(self):
        v = C.c_double(0.0)
        self._ck(self._lib.amg1d_dev_rhs_norm(self._h, C.byref(v)))
        return v.value

    def dev_get_solution(self):
        x = np.zeros(self.n_dof[0])
        self._ck(self._lib.amg1d_dev_get_solution(self._h, capi.dptr(x)))
        return x

    # ---- multi-column device-resident set (up to capi.MAX_COLS right-hand sides per V-cycle) ----------------------
    def _check_cols(self, X):
        if X.ndim != 2 or X.shape[0] != self.n_dof[0] or not 1 <= X.shape[1] <= capi.MAX_COLS:
            raise ValueError(f"DimensionMismatch: expected ({self.n_dof[0]}, k) with 1 <= k <= {capi.MAX_COLS}, "
                             f"got {X.shape}")

    def dev_set_problems(self, X0, B):
        """Upload k = B.shape[1] right-hand sides (and initial guesses X0, None = 0), each of shape (n_dof, k)."""
        B = np.asfortranarray(B, dtype=np.float64)
        self._check_cols(B)
        if X0 is not None:
            X0 = np.asfortranarray(X0, dtype=np.float64)
            if X0.shape != B.shape:
                raise ValueError(f"DimensionMismatch: X0 {X0.shape} vs B {B.shape}")
        PD = C.POINTER(C.c_double)
        self._ck(self._lib.amg1d_dev_set_problems(self._h, B.shape[1], X0.ctypes.data_as(PD) if X0 is not None else None,
                                                  B.ctypes.data_as(PD)))

    def dev_fill_rhs_random_multi(self, k, seed=0):
        """Column c gets the right-hand side of dev_fill_rhs_random(seed + c); x = 0."""
        self._ck(self._lib.amg1d_dev_fill_rhs_random_multi(self._h, int(k), seed))

    def dev_vcycle_multi(self, nPre=3, nPost=3, alpha=2.0 / 3.0, zero_guess=False, with_residual_norms=False):
        self._ck(self._lib.amg1d_dev_vcycle_multi(self._h, nPre, nPost, alpha, int(bool(zero_guess)),
                                                  int(bool(with_residual_norms))))

    def dev_residual_norms(self):
        k = self.info("multi_columns")
        res = np.zeros(max(k, 1))
        self._ck(self._lib.amg1d_dev_residual_norms(self._h, capi.dptr(res)))
        return res[:k].copy()

    def dev_solve_multi(self, maxiter, tol, nPre=3, nPost=3, alpha=2.0 / 3.0):
        """``multigrid`` on every column of the set; returns (iters, [res per column])."""
        k = self.info("multi_columns")
        res = np.zeros(max(maxiter, 1) * max(k, 1))
        it = (C.c_int * max(k, 1))()
        self._ck(self._lib.amg1d_dev_solve_multi(self._h, maxiter, tol, nPre, nPost, alpha, it, capi.dptr(res)))
        iters = [int(it[c]) for c in range(k)]
        return iters, [res[c * maxiter:c * maxiter + iters[c]].copy() for c in range(k)]

    def dev_pcg_multi(self, maxiter, tol, nPre=3, nPost=3, alpha=2.0 / 3.0):
        """``pcg`` on every column of the set (each column bit-identical to ``dev_pcg`` on it alone); returns
        (iters, [res per column]).  The solutions stay on the device; the right-hand sides are consumed."""
        k = self.info("multi_columns")
        res = np.zeros(max(maxiter, 1) * max(k, 1))
        it = (C.c_int * max(k, 1))()
        self._ck(self._lib.amg1d_dev_pcg_multi(self._h, maxiter, tol, nPre, nPost, alpha, it, capi.dptr(res)))
        iters = [int(it[c]) for c in range(k)]
        return iters, [res[c * maxiter:c * maxiter + iters[c]].copy() for c in range(k)]

    def dev_get_solutions(self):
        k = self.info("multi_columns")
        X = np.zeros((self.n_dof[0], max(k, 1)), order="F")
        self._ck(self._lib.amg1d_dev_get_solutions(self._h, X.ctypes.data_as(C.POINTER(C.c_double))))
        return X[:, :k]

    def synchronize(self):
        self._ck(self._lib.amg1d_synchronize(self._h))

    def set_option(self, key, value):
        self._ck(self._lib.amg1d_set_option(self._h, key.encode(), int(value)))

    def info(self, key):
        return int(self._lib.amg1d_get_info(self._h, key.encode()))

    def profile(self, level, leg):
        """(total device ms, launches) of one leg of one level since option 'profile' was set."""
        ms, cnt = C.c_double(0.0), C.c_int(0)
        self._ck(self._lib.amg1d_get_profile(self._h, level, leg, C.byref(ms), C.byref(cnt)))
        return ms.value, cnt.value

    @property
    def stream(self):
        return self._lib.amg1d_stream(self._h)
