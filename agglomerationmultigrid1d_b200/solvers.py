"""Solver entry points: host mirror of src/solvers.jl and of ``apply_smoother`` (src/smoother.jl).

Same names, argument meaning and return values as the reference; every one of them is a call into
libamg1d.so (the GPU).  There is no CPU implementation behind them.

    multigrid_v_cycle(H, x0, b; nPre=3, nPost=3, alpha=2/3) -> x            src/solvers.jl:19-50
    ldiv(H, b) -> b overwritten / ldiv(y, H, b) -> y overwritten            src/solvers.jl:63-92
        (b, y may be n_dof x k matrices: the columns share V-cycles, up to 8 at a time)
    pcg(H, x0, b, maxiter, tol) -> (x, iter, res)      CG with ldiv! as preconditioner (the hook's purpose)
        (x0, b may be n_dof x k matrices: every column its own CG, up to 8 columns sharing V-cycles)
    multigrid(H, x0, b, maxiter, tol) -> (x, iter, res, err)                src/solvers.jl:116-139
    iterative_smoother_solve(A, smoother, x0, b; maxiter, tol, alpha)       src/solvers.jl:189-213
    apply_smoother(S, B; alpha) -> alpha * S^-1 B                           src/smoother.jl:52-81
"""
import numpy as np
import scipy.sparse as sp

from . import blocks as blk
from ._capi import MAX_COLS
from .device import DeviceHierarchy
from .smoother import AbstractSmoother, AdditiveSchwarzSmoother, schwarz_tridiag_blocks, smoother_inverse


def _device_of(H):
    if H.device is None:
        raise RuntimeError("MeshHierarchy was built with upload=False; call H.upload() first")
    return H.device


def multigrid_v_cycle(H, x0, b, nPre=3, nPost=3, alpha=2.0 / 3.0):
    return _device_of(H).vcycle(x0, b, nPre=nPre, nPost=nPost, alpha=alpha)


def ldiv(*args):
    """``ldiv!(H, b)``: b <- one V-cycle from a zero guess; ``ldiv!(y, H, b)``: y <- the same.  A 2-D b (n_dof x k,
    any k) is ``ldiv!(Y, H, B)``: every column as by the 1-D call, up to 8 columns per V-cycle.  On a slab-sharded
    hierarchy b / y are this rank's slabs, as for the 1-D call."""
    if len(args) == 2:
        H, b = args
        out = b
    elif len(args) == 3:
        out, H, b = args
    else:
        raise TypeError("ldiv(H, b) or ldiv(y, H, b)")
    dev = _device_of(H)
    if np.ndim(b) == 2:
        # ldiv!(Y, H, B): the columns in sets of up to 8 through the multi-column cycle, each column bit-identical
        # to ldiv!(y, H, b) on it alone
        B = np.asarray(b, dtype=np.float64)
        if np.shape(out) != B.shape:
            raise ValueError(f"DimensionMismatch: Y {np.shape(out)} vs B {B.shape}")
        Y = np.empty(B.shape, order="F")
        for c0 in range(0, B.shape[1], MAX_COLS):
            dev.dev_set_problems(None, B[:, c0:c0 + MAX_COLS])
            dev.dev_vcycle_multi(zero_guess=True)
            Y[:, c0:c0 + MAX_COLS] = dev.dev_get_solutions()
        out[:] = Y
        return None
    out[:] = dev.ldiv(b)          # zero guess inside the library: no x0 upload, first sweep skips A
    return None


def pcg(H, x0, b, maxiter, tol, nPre=3, nPost=3, alpha=2.0 / 3.0):
    """Conjugate gradients preconditioned with ``ldiv!(z, H, r)`` - the use the reference's ``ldiv!``
    methods are written for (src/solvers.jl:63-92: MeshHierarchy as the ``Pl`` of a Krylov solver); the
    reference itself ships no driver.  Returns (x, iter, res) with res[i] = ||r_i||_2 and the stop rule of
    ``multigrid`` (res < tol ||b||).  A 2-D b (n_dof x k, any k; x0 of the same shape) runs every column as
    the 1-D call would, up to 8 columns at a time through the multi-column set, and returns (X, iters, res) with
    iters a list and res a list of per-column histories.  On a slab-sharded hierarchy x0 / b are this rank's
    slabs, as for the 1-D call."""
    dev = _device_of(H)
    if np.ndim(b) == 2:
        B = np.asarray(b, dtype=np.float64)
        X0 = np.asarray(x0, dtype=np.float64)
        if X0.shape != B.shape:
            raise ValueError(f"DimensionMismatch: x0 {X0.shape} vs b {B.shape}")
        X = np.empty(B.shape, order="F")
        iters, res = [], []
        for c0 in range(0, B.shape[1], MAX_COLS):
            dev.dev_set_problems(X0[:, c0:c0 + MAX_COLS], B[:, c0:c0 + MAX_COLS])
            it, r = dev.dev_pcg_multi(maxiter, tol, nPre=nPre, nPost=nPost, alpha=alpha)
            X[:, c0:c0 + MAX_COLS] = dev.dev_get_solutions()
            iters += it
            res += r
        return X, iters, res
    return dev.pcg(x0, b, maxiter, tol, nPre=nPre, nPost=nPost, alpha=alpha)


def multigrid(H, x0, b, maxiter, tol, u_exact=None, with_error=True):
    """Always cycles with nPre = nPost = 3, alpha = 2/3 like the reference (src/solvers.jl:125).
    ``err`` needs u_exact = A \\ b (GPU direct solve, ~10 n m^2 doubles of factors); pass
    ``with_error=False`` to skip it (err is then filled with NaN)."""
    b = np.asarray(b, dtype=np.float64)
    if maxiter <= 0:
        return np.zeros(len(x0)), 0, np.zeros(0), np.zeros(0)
    if u_exact is None and with_error:
        # src/solvers.jl:120: u_exact = A \\ b - block cyclic reduction on the GPU (amg1d_direct_solve)
        u_exact = _device_of(H).direct_solve(0, b)
    return _device_of(H).solve(x0, b, maxiter, tol, u_exact=u_exact)


def _single_level(A, smoother):
    """One-level device hierarchy for a stand-alone (operator, smoother) pair, cached on the smoother."""
    if smoother._device is not None and smoother._device_A is A:
        return smoother._device
    slots = smoother._slots
    if slots is None:
        raise ValueError("smoother was not built by cg_smoother / dg_smoother")
    lo, di, up = blk.csc_to_blocks(A, slots)
    dinv, is_diag = smoother_inverse(smoother, slots)
    dev = DeviceHierarchy(1)
    dev.set_level_blocks(0, lo, di, up, dinv, is_diag, slots, A.shape[0])
    if isinstance(smoother, AdditiveSchwarzSmoother):       # also HybridSchwarzSmoother
        dev.set_level_smoother(0, *schwarz_tridiag_blocks(smoother, slots))
    dev.finalize()
    smoother._device = dev
    smoother._device_A = A
    return dev


def apply_smoother(A, B, alpha=1.0):
    """``apply_smoother(A::AbstractSmoother, B; alpha)``; B may be a vector, a dense matrix or a
    sparse matrix (the scripts pass the operator itself, tests/dg_smoother_test.jl:105)."""
    if not isinstance(A, AbstractSmoother):
        raise TypeError("apply_smoother needs a smoother")
    if sp.issparse(B):
        B = B.toarray()
    if A._owner is not None:
        dev, level = A._owner
        return dev.apply_smoother(level, B, alpha)
    if A._A is None:
        raise ValueError("smoother was not built by cg_smoother / dg_smoother")
    return _single_level(A._A, A).apply_smoother(0, B, alpha)


def iterative_smoother_solve(A, smoother, x0, b, maxiter=1000, tol=1e-6, alpha=1.0, u_exact=None,
                             with_error=True):
    b = np.asarray(b, dtype=np.float64)
    if maxiter <= 0:
        return np.zeros(len(x0)), 0, np.zeros(0), np.zeros(0)
    dev = _single_level(A, smoother)
    if u_exact is None and with_error:
        u_exact = dev.direct_solve(0, b)          # src/solvers.jl:194, on the GPU
    return dev.smoother_solve(0, x0, b, maxiter=maxiter, tol=tol, alpha=alpha, u_exact=u_exact)
