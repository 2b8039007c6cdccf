"""Preconditioned CG on the multi-column set (amg1d_dev_pcg_multi, solvers.pcg with a 2-D b).

Every column runs the textbook PCG of amg1d_dev_pcg; the columns share each V-cycle (the multi-column cycle), the
product A p (f_matvec_dot_multi reads level 0's operator once for all columns) and one launch per CG vector update or
reduction.  Per column the arithmetic and its order are those of amg1d_dev_pcg, so every column's iteration count,
residual history and solution must be BIT-IDENTICAL to amg1d_dev_pcg on that column alone - compared with
np.array_equal / ==, never with a tolerance."""
import math

import numpy as np
import pytest

import agglomerationmultigrid1d_b200 as aggmg
from agglomerationmultigrid1d_b200 import _capi as capi
from agglomerationmultigrid1d_b200 import blocks as blk
from agglomerationmultigrid1d_b200 import uniform
from agglomerationmultigrid1d_b200.device import DeviceHierarchy
from agglomerationmultigrid1d_b200.smoother import cg_smoother, schwarz_tridiag_blocks, smoother_inverse
from shapes import SHAPES, build_package
from test_gpu_leg_variants import VARIANTS
from test_gpu_multi import _columns, _graded_hierarchy, _uniform

pytestmark = pytest.mark.gpu

CYC = (3, 3, 2.0 / 3.0)
TOL = 1e-10


def _single(dev, x0, b, maxiter, tol, cyc=CYC):
    dev.dev_set_problem(x0, b)
    it, res = dev.dev_pcg(maxiter, tol, *cyc)
    return it, res, dev.dev_get_solution()


def _assert_columns_match(dev, X0, B, maxiter=25, tol=TOL, cyc=CYC, tag=""):
    dev.dev_set_problems(X0, B)
    iters, res = dev.dev_pcg_multi(maxiter, tol, *cyc)
    X = dev.dev_get_solutions()
    for c in range(B.shape[1]):
        it, r, x = _single(dev, X0[:, c], B[:, c], maxiter, tol, cyc)
        assert iters[c] == it, (tag, c, iters, it)
        assert np.array_equal(res[c], r), (tag, c)
        assert np.array_equal(X[:, c], x), (tag, c)
    return iters


@pytest.mark.parametrize("name", ["cg_heirarchy", "dg_heirarchy", "dg_cg_heirarchy", "full_heirarchy", "C2_dg3_agg",
                                  "C3_dg4_agg", "C4_cg3_dg1_agg", "bcr_dg3_agg_n512", "factor3_n24"])
def test_columns_bit_identical_to_single_column_pcg(name):
    H, _, b = build_package(**SHAPES[name])
    dev = H.device
    try:
        for k in (1, 3, 8):
            X0, B = _columns(len(b), k, seed=20 + k)
            B[:, 0] = b
            _assert_columns_match(dev, X0, B, tag=(name, k))
            assert dev.info("multi_columns") == k
        X0, B = _columns(len(b), 3, seed=40)
        B[:, 0] = b
        _assert_columns_match(dev, X0, B, cyc=(2, 2, 0.6), tag=(name, "2/2/0.6"))
    finally:
        dev.close()


def test_columns_leave_at_different_iterations():
    U, _ = _uniform(40960)
    dev = U.upload()
    try:
        w = 2.0 * math.pi / 64.0
        U.device_rhs([("cos", w * w, 0, w, 0.0)], [0.0, math.cos(w * 40960)], dev)
        smooth = dev.dev_get_rhs()
        n = len(smooth)
        rng = np.random.default_rng(7)
        X0 = rng.standard_normal((n, 4))
        X0[:, 0] = 0.0
        B = np.stack([smooth, rng.standard_normal(n), np.zeros(n), dev.matvec(0, X0[:, 3])], axis=1)
        iters = _assert_columns_match(dev, X0, B, maxiter=60, tag="leave")
        assert len(set(iters)) > 1, iters
        assert iters[2] == 0 and iters[3] == 0, iters
        dev.dev_set_problems(X0, B)
        dev.dev_pcg_multi(60, TOL)
        assert np.array_equal(dev.dev_get_solutions()[:, 2], X0[:, 2])      # b = 0 returns x0
    finally:
        dev.close()


def _schwarz_device():
    H, _, b = build_package(**SHAPES["cg_heirarchy"], upload=False)
    nL = len(H.mMeshes)
    dev = DeviceHierarchy(nL)
    slots = [blk.level_slots(m) for m in H.mMeshes]
    for l in range(nL):
        lo, di, up = blk.csc_to_blocks(H.mStiffness[l], slots[l])
        smoother = cg_smoother(H.mMeshes[l], H.mStiffness[l], "addSchwarz") if l == 0 else H.mSmoothers[l]
        dinv, is_diag = smoother_inverse(smoother, slots[l])
        dev.set_level_blocks(l, lo, di, up, dinv, is_diag, slots[l], H.mStiffness[l].shape[0])
        if l == 0:
            dev.set_level_smoother(0, *schwarz_tridiag_blocks(smoother, slots[0]))
    for l in range(nL - 1):
        dev.set_transfer_blocks(l, *blk.transfer_to_blocks(H.mInterpolation[l], slots[l], slots[l + 1]))
    dev.finalize()
    return dev, b


@pytest.mark.parametrize("case", ["uniform_40960", "graded"])
def test_leg_forms_and_options(case):
    if case == "graded":
        dev, b = _graded_hierarchy()
    else:
        U, b = _uniform(40960)
        dev = U.upload()
    try:
        dev.set_option("leg_pipeline_min", 0)
        X0, B = _columns(len(b), 3, seed=13)
        B[:, 1] = b
        settings = [(name, opts) for name, opts in VARIANTS] + [("unfused", dict(fused=0)), ("ungraphed", dict(graph=0))]
        for name, opts in settings:
            for key, val in opts.items():
                dev.set_option(key, val)
            _assert_columns_match(dev, X0, B, maxiter=15, tag=(case, name))
            for key in opts:
                dev.set_option(key, {"fused": 1, "graph": 1}.get(key, opts[key]))
        if case != "graded":
            for mode in (1, 2):
                dev.set_option("pattern_resident", mode)
                _assert_columns_match(dev, X0, B, maxiter=15, tag=(case, "pattern", mode))
            dev.set_option("pattern_resident", 0)
    finally:
        dev.close()


def test_row_tier_and_schwarz_levels():
    U, b = _uniform(6144, orders=(8, 4, 2, 1))
    dev = U.upload()
    try:
        assert dev.info("multi_legs:0") == 0
        X0, B = _columns(len(b), 3, seed=15)
        B[:, 0] = b
        _assert_columns_match(dev, X0, B, maxiter=15, tag="p8")
    finally:
        dev.close()
    dev, b = _schwarz_device()
    try:
        assert dev.info("multi_legs:0") == 0
        X0, B = _columns(len(b), 3, seed=16)
        B[:, 2] = b
        _assert_columns_match(dev, X0, B, maxiter=15, tag="schwarz")
    finally:
        dev.close()


def test_launches_per_iteration_do_not_grow_with_columns_on_a_fused_level():
    U, b = _uniform(40960)
    dev = U.upload()
    try:
        def launches(k):
            X0, B = _columns(len(b), k, seed=k)
            dev.dev_set_problems(X0, B)
            iters, _ = dev.dev_pcg_multi(3, 1e-15)
            assert iters == [3] * k, iters
            return dev.info("multi_pcg_launches_per_iteration")
        fused = launches(2)
        assert fused > 0 and launches(8) == fused
        dev.set_option("fused", 0)
        assert launches(8) > launches(2)
    finally:
        dev.close()


def test_state_and_errors():
    H, _, b = build_package(**SHAPES["C2_dg3_agg"])
    dev = H.device
    lib = capi.load()
    try:
        with pytest.raises(capi.Amg1dError) as e:
            dev.dev_pcg_multi(10, TOL)
        assert e.value.code == capi.ERR_STATE
        X0, B = _columns(len(b), 3, seed=17)
        dev.dev_set_problems(X0, B)
        with pytest.raises(capi.Amg1dError) as e:
            dev.dev_pcg_multi(-1, TOL)
        assert e.value.code == capi.ERR_ARG
        bytes0 = dev.info("device_bytes")
        # the single-column resident problem is unchanged across an interleaved multi PCG ...
        x0 = np.random.default_rng(3).standard_normal(len(b))
        dev.dev_set_problem(x0, b)
        dev.dev_vcycle(with_residual_norm=True)
        before = dev.dev_get_solution(), dev.dev_residual_norm()
        dev.dev_set_problem(x0, b)
        dev.dev_set_problems(X0, B)
        iters, res = dev.dev_pcg_multi(20, TOL)
        assert dev.info("device_bytes") > bytes0                      # the per-column CG vectors are counted
        X = dev.dev_get_solutions()
        dev.dev_vcycle(with_residual_norm=True)
        assert np.array_equal(dev.dev_get_solution(), before[0]) and dev.dev_residual_norm() == before[1]
        # ... the right-hand sides are consumed: the set refuses to cycle until it is installed again
        for call in (dev.dev_vcycle_multi, dev.dev_residual_norms, lambda: dev.dev_solve_multi(5, TOL),
                     lambda: dev.dev_pcg_multi(5, TOL)):
            with pytest.raises(capi.Amg1dError) as e:
                call()
            assert e.value.code == capi.ERR_STATE
        assert np.array_equal(dev.dev_get_solutions(), X)
        # ... and the set is unchanged across an interleaved single-column PCG
        dev.dev_set_problems(X0, B)
        dev.dev_set_problem(x0, b)
        dev.dev_pcg(20, TOL)
        iters2, res2 = dev.dev_pcg_multi(20, TOL)
        assert iters2 == iters and all(np.array_equal(r, q) for r, q in zip(res, res2))
        assert np.array_equal(dev.dev_get_solutions(), X)
        # a NaN in one column is rejected before the first iteration, naming the column
        Bn = B.copy()
        Bn[5, 1] = np.nan
        dev.dev_set_problems(X0, Bn)
        with pytest.raises(capi.Amg1dError) as e:
            dev.dev_pcg_multi(20, TOL)
        assert e.value.code == capi.ERR_ARG and "column 1" in str(e.value)
        assert np.array_equal(dev.dev_get_solutions(), X0)            # no iteration ran
        dev.dev_set_problems(X0, B)
        assert lib.amg1d_dev_pcg_multi(dev._h, 5, TOL, 3, 3, 2.0 / 3.0, None, None) == capi.ERR_ARG
    finally:
        dev.close()


def test_solvers_pcg_with_eleven_columns():
    H, _, b = build_package(**SHAPES["C2_dg3_agg"])
    try:
        rng = np.random.default_rng(19)
        B = rng.standard_normal((len(b), 11))
        B[:, 4] = b
        X0 = rng.standard_normal((len(b), 11))
        X, iters, res = aggmg.pcg(H, X0, B, 30, TOL)
        assert len(iters) == 11 and len(res) == 11
        for c in range(11):
            x, it, r = aggmg.pcg(H, X0[:, c].copy(), B[:, c].copy(), 30, TOL)
            assert iters[c] == it, (c, iters, it)
            assert np.array_equal(res[c], r), c
            assert np.array_equal(X[:, c], x), c
    finally:
        H.device.close()


def test_at_scale_t_chain_random_columns():
    """T's level chain at 2^24 elements, k = 4 right-hand sides filled on the device."""
    n = 1 << 24
    U = uniform.UniformDgHierarchy(n, [3, 1], [2] * 24, xin=0.0, xout=float(n), CDir=1000.0)
    dev = U.upload()
    try:
        seed = 91
        dev.dev_fill_rhs_random_multi(4, seed)
        iters, res = dev.dev_pcg_multi(8, TOL)
        X = dev.dev_get_solutions()
        for c in (0, 3):
            dev.dev_fill_rhs_random(seed + c)
            it, r = dev.dev_pcg(8, TOL)
            assert iters[c] == it, (c, iters, it)
            assert np.array_equal(res[c], r), c
            assert np.array_equal(X[:, c], dev.dev_get_solution()), c
    finally:
        dev.close()


def test_at_scale_c4_chain_uploaded_columns():
    """C4's chain (CG p = 3 -> CG 1 -> DG 1 -> agglomerated) at 2^22 elements: the permuted CG-first level 0."""
    n = 1 << 22
    U = uniform.UniformCgHierarchy(n, [3, 1], [1], [2] * 22, xin=0.0, xout=float(n), CDir=1000.0)
    dev = U.upload()
    try:
        X0, B = _columns(dev.n_dof[0], 2, seed=23)
        _assert_columns_match(dev, X0, B, maxiter=8, tag="C4 2^22")
    finally:
        dev.close()
