"""Multi-column device-resident problems (amg1d_dev_set_problems ... amg1d_dev_get_solutions, kernels_multi.cuh).

One V-cycle serves up to 8 right-hand sides: levels with fused legs read their operator once for all columns
(f_down_multi / f_up_multi), every other level, the single-CTA tail and the coarse solve run their single-column code
once per column.  Per column the arithmetic and its order are those of the single-column cycle, so every column's
iterate, residual norm and solve history must be BIT-IDENTICAL to the single-column calls on that column alone -
compared with np.array_equal / ==, never with a tolerance."""
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

pytestmark = pytest.mark.gpu

CYCLES = ((3, 3, 2.0 / 3.0), (0, 2, 0.7), (2, 0, 0.5), (1, 1, 1.0))


def _columns(n_dof, k, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n_dof, k)), rng.standard_normal((n_dof, k))


def _single(dev, x0, b, cyc, zero_guess=False):
    a, c, al = cyc
    if zero_guess:
        return dev.ldiv(b, nPre=a, nPost=c, alpha=al), None
    dev.dev_set_problem(x0, b)
    dev.dev_vcycle(a, c, al, with_residual_norm=True)
    return dev.dev_get_solution(), dev.dev_residual_norm()


def _multi(dev, X0, B, cyc, zero_guess=False):
    a, c, al = cyc
    dev.dev_set_problems(None if zero_guess else X0, B)
    dev.dev_vcycle_multi(a, c, al, zero_guess=zero_guess, with_residual_norms=not zero_guess)
    return dev.dev_get_solutions(), (None if zero_guess else dev.dev_residual_norms())


def _assert_columns_match(dev, X0, B, cycles=CYCLES, zero_guess=True, tag=""):
    for cyc in cycles:
        X, R = _multi(dev, X0, B, cyc)
        for c in range(B.shape[1]):
            x, r = _single(dev, X0[:, c], B[:, c], cyc)
            assert np.array_equal(X[:, c], x), (tag, cyc, c)
            assert R[c] == r, (tag, cyc, c, R[c], r)
    if zero_guess:
        Y, _ = _multi(dev, X0, B, CYCLES[0], zero_guess=True)
        for c in range(B.shape[1]):
            assert np.array_equal(Y[:, c], _single(dev, None, B[:, c], CYCLES[0], zero_guess=True)[0]), (tag, "ldiv", c)


@pytest.mark.parametrize("name", ["cg_heirarchy", "dg_heirarchy", "dg_cg_heirarchy", "full_heirarchy", "C2_dg3_agg",
                                  "C3_dg4_agg", "C4_cg3_dg1_agg", "bcr_dg3_agg_n512", "factor3_n24"])
def test_columns_bit_identical_to_single_column(name):
    H, _, b = build_package(**SHAPES[name])
    dev = H.device
    try:
        for k in (1, 2, 3, 8):
            X0, B = _columns(len(b), k, seed=k)
            B[:, 0] = b
            _assert_columns_match(dev, X0, B, cycles=CYCLES if k in (3, 8) else CYCLES[:1], tag=(name, k))
            assert dev.info("multi_columns") == k
        assert dev.info("multi_launches_per_cycle") > 0
    finally:
        dev.close()


def _graded_hierarchy():
    """Explicit per-element blocks on a graded mesh (the mesh of test_gpu_leg_variants)."""
    n = 3 * 2 ** 12
    rng = np.random.default_rng(0)
    x = np.concatenate([[0.0], np.cumsum(0.5 + rng.random(n))])
    xout = float(x[-1])
    w = 2.0 * math.pi / 64.0
    mesh = aggmg.Mesh(x)
    bd = aggmg.set_boundary(mesh, 0.0, xout, [("neu", 0.0), ("dir", math.cos(w * xout))])
    meshes = [aggmg.DgMesh(mesh, 3), aggmg.DgMesh(mesh, 1)]
    cur = n
    for i in range(10):
        agg = [[2 * j, 2 * j + 1] for j in range(cur // 2)]
        cur //= 2
        meshes.append(aggmg.AgglomeratedDgMesh1(1, agg, mesh, meshes[1]) if i == 0
                      else aggmg.AgglomeratedDgMeshN(1, agg, meshes[-1], meshes[1]))
    G, D, C = aggmg.dg_flux_operators(meshes[0], mesh, bd, 1000.0)
    A = (C - D @ meshes[0].mMassMatrixLU.solve(G)).tocsc()
    f, r = aggmg.dg_flux_rhs(meshes[0], mesh, lambda t: w * w * np.cos(w * t), bd, 1000.0)
    b = f - D @ meshes[0].mMassMatrixLU.solve(r)
    H = aggmg.MeshHierarchy(meshes, [bd] * len(meshes), A, G, D, C, nDG=2, nAgg=10, upload=False)
    return H.upload(), b


def _uniform(n, orders=(3, 1)):
    k = (n & -n).bit_length() - 1
    U = uniform.UniformDgHierarchy(n, list(orders), [2] * k, xin=0.0, xout=float(n), CDir=1000.0)
    w = 2.0 * math.pi / 64.0
    return U, U.rhs(lambda x: w * w * np.cos(w * x), [0.0, math.cos(w * n)])


@pytest.mark.parametrize("case", ["uniform_40960", "uniform_786432", "graded"])
def test_leg_forms_and_options(case):
    if case == "graded":
        dev, b = _graded_hierarchy()
    else:
        U, b = _uniform(int(case.split("_")[1]))
        dev = U.upload()
    try:
        dev.set_option("leg_pipeline_min", 0)
        X0, B = _columns(len(b), 3, seed=11)
        B[:, 1] = b
        cycles = CYCLES[:2]
        settings = [(name, opts) for name, opts in VARIANTS] + [("unfused", dict(fused=0)), ("ungraphed", dict(graph=0))]
        for name, opts in settings:
            for key, val in opts.items():
                dev.set_option(key, val)
            assert dev.info("multi_legs:0") == (0 if name == "unfused" else 1), name
            _assert_columns_match(dev, X0, B, cycles=cycles, zero_guess=name != "ungraphed", tag=(case, name))
            for key in opts:
                dev.set_option(key, {"fused": 1, "graph": 1}.get(key, opts[key]))
        # an option changed between two multi cycles takes effect: the graphs are rebuilt, the launches change
        dev.dev_set_problems(X0, B)
        dev.dev_vcycle_multi()
        fused_launches = dev.info("multi_launches_per_cycle")
        dev.set_option("fused", 0)
        dev.dev_vcycle_multi()
        assert dev.info("multi_launches_per_cycle") > fused_launches
        dev.set_option("fused", 1)
    finally:
        dev.close()


def test_pattern_resident_modes():
    U, b = _uniform(40960)
    dev = U.upload()
    try:
        assert dev.info("pattern:0") == 1
        X0, B = _columns(len(b), 4, seed=3)
        for mode in (1, 2):
            dev.set_option("pattern_resident", mode)
            assert dev.info("multi_legs:0") == 1
            _assert_columns_match(dev, X0, B, cycles=CYCLES[:2], tag=("pattern", mode))
    finally:
        dev.close()


def test_row_tier_level_falls_back_per_column():
    """p = 8 level 0: 9 x 9 blocks run the row-per-thread legs, once per column."""
    U, b = _uniform(6144, orders=(8, 4, 2, 1))
    dev = U.upload()
    try:
        assert dev.info("multi_legs:0") == 0
        X0, B = _columns(len(b), 3, seed=5)
        _assert_columns_match(dev, X0, B, cycles=CYCLES[:2], tag="p8")
    finally:
        dev.close()


def test_schwarz_smoothed_level_falls_back_per_column():
    """Level 0 smoothed by the additive Schwarz smoother (block-tridiagonal smoother operator, generic kernels)."""
    H, _, b = build_package(**SHAPES["cg_heirarchy"], upload=False)
    nL = len(H.mMeshes)
    dev = DeviceHierarchy(nL)
    try:
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
        assert dev.info("multi_legs:0") == 0
        X0, B = _columns(len(b), 3, seed=9)
        B[:, 2] = b
        _assert_columns_match(dev, X0, B, cycles=CYCLES[:2], tag="schwarz")
    finally:
        dev.close()


def test_solve_multi_matches_per_column_solves():
    U, _ = _uniform(40960)
    dev = U.upload()
    try:
        w = 2.0 * math.pi / 64.0
        U.device_rhs([("cos", w * w, 0, w, 0.0)], [0.0, math.cos(w * 40960)], dev)
        smooth = dev.dev_get_rhs()
        rng = np.random.default_rng(1)
        # b = 0 never meets the relative stop rule (0 < tol * 0 is false) and cycles maxiter times
        B = np.stack([rng.standard_normal(len(smooth)), smooth, np.zeros(len(smooth))], axis=1)
        tol = 1e-9
        dev.dev_set_problems(None, B)
        iters, res = dev.dev_solve_multi(40, tol)
        X = dev.dev_get_solutions()
        assert len(set(iters)) > 1, iters                              # the columns leave the set at different cycles
        for c in range(B.shape[1]):
            dev.dev_set_problem(None, B[:, c])
            it, r = dev.dev_solve(40, tol)
            assert iters[c] == it, (c, iters, it)
            assert np.array_equal(res[c], r), c
            assert np.array_equal(X[:, c], dev.dev_get_solution()), c
    finally:
        dev.close()


def test_state_and_errors():
    H, _, b = build_package(**SHAPES["C2_dg3_agg"])
    dev = H.device
    try:
        with pytest.raises(capi.Amg1dError) as e:
            dev.dev_vcycle_multi()
        assert e.value.code == capi.ERR_STATE
        lib = capi.load()
        for k in (0, 9):
            assert lib.amg1d_dev_fill_rhs_random_multi(dev._h, k, 1) == capi.ERR_ARG
            assert lib.amg1d_dev_set_problems(dev._h, k, None, capi.dptr(np.zeros(len(b) * 9))) == capi.ERR_ARG
        assert dev.info("multi_columns") == 0
        bytes0 = dev.info("device_bytes")
        # the resident single-column problem is the same before and after an interleaved multi run
        x0 = np.random.default_rng(2).standard_normal(len(b))
        dev.dev_set_problem(x0, b)
        dev.dev_vcycle(with_residual_norm=True)
        before = dev.dev_get_solution(), dev.dev_residual_norm()
        dev.dev_set_problem(x0, b)
        X0, B = _columns(len(b), 5, seed=4)
        dev.dev_set_problems(X0, B)
        dev.dev_vcycle_multi(with_residual_norms=True)
        assert dev.info("device_bytes") > bytes0                      # the column storage is counted
        dev.dev_vcycle(with_residual_norm=True)
        assert np.array_equal(dev.dev_get_solution(), before[0]) and dev.dev_residual_norm() == before[1]
        # ... and the column set survives single-column cycles
        dev.dev_vcycle_multi(with_residual_norms=True)
        X2 = dev.dev_get_solutions()
        dev.dev_set_problems(X0, B)
        dev.dev_vcycle_multi()
        dev.dev_vcycle_multi()
        assert np.array_equal(dev.dev_get_solutions(), X2)
        with pytest.raises(ValueError):
            dev.dev_set_problems(None, np.zeros((len(b) + 1, 2)))
        # ldiv!(Y, H, B) with 11 columns: two sets, each column as the 1-D ldiv!
        B11 = np.random.default_rng(6).standard_normal((len(b), 11))
        Y = np.zeros_like(B11)
        aggmg.ldiv(Y, H, B11)
        for c in range(11):
            y = np.zeros(len(b))
            aggmg.ldiv(y, H, B11[:, c].copy())
            assert np.array_equal(Y[:, c], y), c
    finally:
        dev.close()


def test_at_scale_random_columns():
    """T's level chain at 2^24 elements, k = 4 right-hand sides filled on the device."""
    n = 1 << 24
    U = uniform.UniformDgHierarchy(n, [3, 1], [2] * 24, xin=0.0, xout=float(n), CDir=1000.0)
    dev = U.upload()
    try:
        seed = 77
        dev.dev_fill_rhs_random_multi(4, seed)
        dev.dev_vcycle_multi(with_residual_norms=True)
        X = dev.dev_get_solutions()
        R = dev.dev_residual_norms()
        for c in (0, 3):
            dev.dev_fill_rhs_random(seed + c)
            dev.dev_vcycle(with_residual_norm=True)
            assert np.array_equal(X[:, c], dev.dev_get_solution()), c
            assert R[c] == dev.dev_residual_norm(), c
    finally:
        dev.close()
