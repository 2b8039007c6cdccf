"""Oracle (test infrastructure): ctypes driver of oracle/vcycle_ref.c, the plain-C restatement of
src/solvers.jl:19-50.  Feeds it an oracle ``MeshHierarchy`` (scipy operators, LU blocks)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import scipy.sparse as sp

from .smoother import JacobiSmoother

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libvcycle_ref.so")
_pd, _pi = C.POINTER(C.c_double), C.POINTER(C.c_int64)


def load():
    if os.path.exists(_LIB) and os.path.getmtime(_LIB) >= os.path.getmtime(os.path.join(_HERE, "vcycle_ref.c")):
        lib = C.CDLL(_LIB)
    elif os.access(_HERE, os.W_OK):
        subprocess.check_call(["make", "-s", "-C", _HERE])
        lib = C.CDLL(_LIB)
    else:
        # read-only tree: the same Makefile target, built in a temporary directory (the loaded library
        # stays mapped after the directory is removed)
        with tempfile.TemporaryDirectory(prefix="vcycle_ref_") as tmp:
            subprocess.check_call(["make", "-s", "-C", tmp, "-f", os.path.join(_HERE, "Makefile"), f"VPATH={_HERE}"])
            lib = C.CDLL(os.path.join(tmp, "libvcycle_ref.so"))
    lib.ref_create.restype = C.c_void_p
    lib.ref_create.argtypes = [C.c_int]
    lib.ref_set_level.argtypes = [C.c_void_p, C.c_int, C.c_int64, _pi, _pi, _pd, C.c_int, C.c_int64, _pi, _pd, _pd]
    lib.ref_set_transfer.argtypes = [C.c_void_p, C.c_int, C.c_int64, _pi, _pi, _pd, _pi, _pi, _pd]
    lib.ref_set_coarse_dense.argtypes = [C.c_void_p, C.c_int64, _pd]
    lib.ref_vcycle.argtypes = [C.c_void_p, _pd, _pd, C.c_int, C.c_int, C.c_double]
    lib.ref_residual_norm.restype = C.c_double
    lib.ref_residual_norm.argtypes = [C.c_void_p, _pd, _pd]
    lib.ref_destroy.argtypes = [C.c_void_p]
    lib.ref_set_threads.argtypes = [C.c_int]
    lib.ref_set_threads.restype = C.c_int
    lib.ref_set_level_pattern.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, _pd, _pd, _pd,
                                          C.c_int, C.c_int]
    lib.ref_set_transfer_pattern.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _pd, _pd, C.c_int]
    lib.ref_set_coarse_from_pattern.argtypes = [C.c_void_p]
    return lib


def _p(a, t):
    return a.ctypes.data_as(t)


class CRefHierarchy:
    def __init__(self, H):
        self.lib = load()
        self.keep = []
        nL = len(H.mStiffness)
        self.h = self.lib.ref_create(nL)
        for l in range(nL):
            A = sp.csr_matrix(H.mStiffness[l])
            A.sort_indices()
            Ap, Aj, Ax = A.indptr.astype(np.int64), A.indices.astype(np.int64), A.data.astype(np.float64)
            S = H.mSmoothers[l]
            if isinstance(S, JacobiSmoother):
                jac = np.ascontiguousarray(S.mJac, dtype=np.float64)
                self.keep += [Ap, Aj, Ax, jac]
                rc = self.lib.ref_set_level(self.h, l, A.shape[0], _p(Ap, _pi), _p(Aj, _pi), _p(Ax, _pd), 0, 0,
                                            None, None, _p(jac, _pd))
            else:
                inds = np.ascontiguousarray(S.mBlockInds.T, dtype=np.int64)          # (nblocks, m)
                nb, m = inds.shape
                Ac = sp.csc_matrix(H.mStiffness[l])
                blocks = np.ascontiguousarray(
                    np.stack([Ac[i, :][:, i].toarray() for i in inds]) if nb <= 4096 else _diag_blocks(A, inds))
                self.keep += [Ap, Aj, Ax, inds, blocks]
                rc = self.lib.ref_set_level(self.h, l, A.shape[0], _p(Ap, _pi), _p(Aj, _pi), _p(Ax, _pd), m, nb,
                                            _p(inds, _pi), _p(blocks, _pd), None)
            assert rc == 0, rc
            if l < nL - 1:
                L = sp.csr_matrix(H.mInterpolation[l]); L.sort_indices()
                LT = sp.csr_matrix(sp.csc_matrix(H.mInterpolation[l]).T); LT.sort_indices()
                arrs = [L.indptr.astype(np.int64), L.indices.astype(np.int64), L.data.astype(np.float64),
                        LT.indptr.astype(np.int64), LT.indices.astype(np.int64), LT.data.astype(np.float64)]
                self.keep += arrs
                self.lib.ref_set_transfer(self.h, l, L.shape[1], _p(arrs[0], _pi), _p(arrs[1], _pi), _p(arrs[2], _pd),
                                          _p(arrs[3], _pi), _p(arrs[4], _pi), _p(arrs[5], _pd))
        Ad = np.ascontiguousarray(sp.csr_matrix(H.mStiffness[-1]).toarray())
        self.keep.append(Ad)
        assert self.lib.ref_set_coarse_dense(self.h, Ad.shape[0], _p(Ad, _pd)) == 0

    def vcycle(self, x0, b, nPre=3, nPost=3, alpha=2.0 / 3.0):
        x = np.array(x0, dtype=np.float64, copy=True)
        b = np.ascontiguousarray(b, dtype=np.float64)
        self.lib.ref_vcycle(self.h, _p(x, _pd), _p(b, _pd), nPre, nPost, alpha)
        return x

    def residual_norm(self, x, b):
        return self.lib.ref_residual_norm(self.h, _p(np.ascontiguousarray(x), _pd), _p(np.ascontiguousarray(b), _pd))

    def set_threads(self, n):
        """OpenMP threads for the row-parallel loops (0 = leave unchanged); returns the count in use."""
        return self.lib.ref_set_threads(int(n))

    def close(self):
        if self.h:
            self.lib.ref_destroy(self.h)
            self.h = None


class CRefPattern(CRefHierarchy):
    """The same C restatement fed with the block-pattern form of a uniform-mesh hierarchy (vcycle_ref.c header):
    every level as its distinct block rows, every transfer as its periodic blocks - the very arrays that are
    uploaded to the GPU - so that the oracle can run at BASELINE's own sizes (2^20 .. 2^26 elements) where
    global CSR matrices would take tens of GB.  Vectors of CG levels are in the group order of the upload
    ([vertex k, interior nodes of element k], padded closing group); the row walks still follow the
    reference's vertex-first DOF numbering (flag vertex_first).

    levels:    list of dict(n, m, n_head, n_tail, lo, di, up, point_jacobi, vertex_first); lo / di / up are
               (n_head + 1 + n_tail, m, m) arrays in (set, i, j) order
    transfers: list of dict(ratio, shift, base, period, n_head, n_tail, P0, P1) - parent(e) = (e + shift) //
               ratio + base, P0 / P1 of shape (n_head + period + n_tail, m_fine, m_coarse), P1 may be None"""

    def __init__(self, levels, transfers):
        self.lib = load()
        self.keep = []
        nL = len(levels)
        assert len(transfers) == nL - 1
        self.h = self.lib.ref_create(nL)
        self.n_dof = [int(lv["n"]) * int(lv["m"]) for lv in levels]
        for l, lv in enumerate(levels):
            arrs = [np.ascontiguousarray(lv[k], dtype=np.float64) for k in ("lo", "di", "up")]
            ns = lv["n_head"] + 1 + lv["n_tail"]
            assert all(a.shape == (ns, lv["m"], lv["m"]) for a in arrs), (l, [a.shape for a in arrs], ns)
            self.keep += arrs
            rc = self.lib.ref_set_level_pattern(self.h, l, int(lv["n"]), int(lv["m"]), int(lv["n_head"]),
                                                int(lv["n_tail"]), _p(arrs[0], _pd), _p(arrs[1], _pd),
                                                _p(arrs[2], _pd), int(bool(lv["point_jacobi"])),
                                                int(bool(lv["vertex_first"])))
            assert rc == 0, (l, rc)
        for l, t in enumerate(transfers):
            P0 = np.ascontiguousarray(t["P0"], dtype=np.float64)
            P1 = None if t.get("P1") is None else np.ascontiguousarray(t["P1"], dtype=np.float64)
            nb = t["n_head"] + t["period"] + t["n_tail"]
            mf, mc = levels[l]["m"], levels[l + 1]["m"]
            assert P0.shape == (nb, mf, mc) and (P1 is None or P1.shape == P0.shape), (l, P0.shape, nb, mf, mc)
            self.keep += [P0, P1]
            rc = self.lib.ref_set_transfer_pattern(
                self.h, l, int(levels[l]["n"]), int(levels[l + 1]["n"]), mf, mc, int(t["ratio"]), int(t["shift"]),
                int(t["base"]), int(t["period"]), int(t["n_head"]), int(t["n_tail"]), _p(P0, _pd),
                None if P1 is None else _p(P1, _pd), int(bool(levels[l + 1]["vertex_first"])))
            assert rc == 0, (l, rc)
        assert self.lib.ref_set_coarse_from_pattern(self.h) == 0

    def multigrid(self, x0, b, maxiter, tol, nPre=3, nPost=3, alpha=2.0 / 3.0):
        """src/solvers.jl:116-139 without the error history: (x, iter, res)."""
        x = np.array(x0, dtype=np.float64, copy=True)
        b = np.ascontiguousarray(b, dtype=np.float64)
        nb = float(np.linalg.norm(b))
        res = []
        for _ in range(maxiter):
            self.lib.ref_vcycle(self.h, _p(x, _pd), _p(b, _pd), nPre, nPost, alpha)
            res.append(self.lib.ref_residual_norm(self.h, _p(x, _pd), _p(b, _pd)))
            if res[-1] < tol * nb:
                break
        return x, len(res), np.array(res)


def pattern_arrays(U):
    """(levels, transfers) for CRefPattern from a uniform-mesh hierarchy object of the product's host package
    (duck-typed: ``levels`` with ``n, m, explicit, ops['A']`` and ``is_cg``; ``transfers`` as (P, ratio);
    ``cg_transfers`` as dicts) - the arrays its ``upload`` hands to amg1d_set_level_pattern /
    amg1d_set_transfer_pattern, unchanged."""
    levels = []
    for lv in U.levels:
        A = lv.ops["A"]
        cg = bool(getattr(lv, "is_cg", False))
        if lv.explicit:
            lo, di, up = (np.concatenate([a, a[-1:]]) for a in A)    # every block row explicit (+ an unused "interior" one)
            levels.append(dict(n=lv.n, m=lv.m, n_head=lv.n, n_tail=0, lo=lo, di=di, up=up, point_jacobi=cg,
                               vertex_first=cg))
        else:
            nb = (A.di.shape[0] - 1) // 2
            levels.append(dict(n=lv.n, m=lv.m, n_head=nb, n_tail=nb, lo=A.lo, di=A.di, up=A.up, point_jacobi=cg,
                               vertex_first=cg))
    transfers = [dict(t) for t in getattr(U, "cg_transfers", [])]
    for P, ratio in U.transfers:
        transfers.append(dict(ratio=ratio, shift=0, base=0, period=P.shape[0], n_head=0, n_tail=0, P0=P, P1=None))
    return levels, transfers


def _diag_blocks(A, inds):
    """Dense diagonal blocks of a CSR matrix for contiguous element index sets (vectorised)."""
    nb, m = inds.shape
    coo = A.tocoo()
    elem = np.full(A.shape[0], -1, dtype=np.int64)
    loc = np.zeros(A.shape[0], dtype=np.int64)
    elem[inds.ravel()] = np.repeat(np.arange(nb), m)
    loc[inds.ravel()] = np.tile(np.arange(m), nb)
    same = elem[coo.row] == elem[coo.col]
    out = np.zeros((nb, m, m))
    np.add.at(out, (elem[coo.row[same]], loc[coo.row[same]], loc[coo.col[same]]), coo.data[same])
    return out
