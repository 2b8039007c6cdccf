"""Ragged agglomerations on the GPU (tests/ragged_shapes.py): aggregates of several sizes, a last coarse
element with fewer children than the others, shifted and non-closed parent maps, two-parent maps without a
closed form.  Each of these takes its own kernel path (the transfer class decides between the fused legs,
the single-CTA tail f_tail and the generic tier), and every one is judged here against a reference that
does not share its code:

  - the path itself: info "multi_legs:<l>" and "tail_start" against the class each shape claims;
  - every level operation against an extended-precision reference, ROW BY ROW: a dropped or doubled child
    of a partial aggregate changes one row by far more than its own rounding bound, even when that row's
    entries are small next to ||A||;
  - V-cycles, multigrid, ldiv and PCG against the oracle with the tolerance rules of test_gpu_parity.py;
  - every kernel tier, leg form and storage class bit for bit against the generic tier;
  - the multi-column set bit for bit against the single-column calls;
  - device-side set-up on the single-parent shapes, and its refusal on the others;
  - at 2^17 + 1 and 3 * 2^16 + 5 elements, the C oracle fed the very host hierarchy that is uploaded."""
import math

import numpy as np
import pytest
import scipy.sparse as sp

import agglomerationmultigrid1d_b200 as aggmg
from oracle import solvers as osolv
from ragged_shapes import SHAPES, build_kwargs, build_oracle, build_package, transfer_classes
from test_gpu_leg_variants import VARIANTS
from test_gpu_multi import CYCLES, _assert_columns_match
from test_gpu_parity import dense_coarse_solver, rounding_floor
from test_gpu_pcg_multi import _assert_columns_match as _assert_pcg_columns_match

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps
LD = np.longdouble
SWEEPS = ((3, 3, 2.0 / 3.0), (1, 2, 0.5), (0, 3, 2.0 / 3.0), (2, 0, 0.8), (0, 0, 1.0))
DEFAULT_TAIL = 1024


@pytest.fixture(scope="module", params=sorted(SHAPES))
def case(request):
    kw = build_kwargs(request.param)
    Ho, bo = build_oracle(**kw)
    Hp, bp = build_package(**kw)
    yield request.param, Ho, bo, Hp, bp
    Hp.device.close()


DEFAULTS = (("fused", 1), ("graph", 1), ("coarse_cta_elems", DEFAULT_TAIL), ("leg_pipeline_min", 500000),
            ("recompute_dinv", 4), ("leg_pipeline", 1), ("dinv_registers", 0))


def _reset(dev):
    for key, val in DEFAULTS:
        dev.set_option(key, val)


# ---- a. path pinning ------------------------------------------------------------------------------
def test_paths_are_pinned(case):
    name, Ho, bo, Hp, bp = case
    dev = Hp.device
    s = SHAPES[name]
    nT = len(Hp.mMeshes) - 1
    try:
        dev.set_option("coarse_cta_elems", 0)
        assert dev.info("tail_start") < 0
        got = [dev.info(f"multi_legs:{l}") for l in range(nT)]
        assert got == s["multi_legs"], (name, got)
        dev.set_option("coarse_cta_elems", DEFAULT_TAIL)
        ts = dev.info("tail_start")
        assert ts == s["tail_start"], (name, ts)
        got = [dev.info(f"multi_legs:{l}") for l in range(nT)]
        assert got == [v if l < ts else 0 for l, v in enumerate(s["multi_legs"])], (name, got)
        # the classes the multi-column legs and the tail rely on agree with the host replay
        tc = transfer_classes(Hp)
        assert all(tc[l]["single_parent_uniform"] for l in range(ts, nT)), name
        assert all(got[l] == 0 for l in range(nT) if not tc[l]["fusable"]), name
    finally:
        _reset(dev)


# ---- b. level operations, row by row --------------------------------------------------------------
def _rows(M, v):
    """(M v in long double, |M| |v| in long double, terms per row) for a sparse M."""
    M = sp.csr_matrix(M)
    M.sort_indices()
    prod = M.data.astype(LD) * np.asarray(v, dtype=LD)[M.indices]
    k = np.diff(M.indptr)
    ref = np.zeros(M.shape[0], dtype=LD)
    mag = np.zeros(M.shape[0], dtype=LD)
    nz = k > 0
    ref[nz] = np.add.reduceat(prod, M.indptr[:-1][nz])
    mag[nz] = np.add.reduceat(np.abs(prod), M.indptr[:-1][nz])
    return ref, mag, k


def _assert_rows(got, ref, mag, k, what):
    err = np.abs(np.asarray(got, dtype=LD) - ref)
    bound = (k + 2) * LD(EPS) * mag
    bad = np.nonzero(err > bound)[0]
    assert bad.size == 0, (what, bad[:8], [float(err[i]) for i in bad[:4]], [float(bound[i]) for i in bad[:4]])


def test_level_operations_row_bounds(case):
    name, Ho, bo, Hp, bp = case
    dev = Hp.device
    rng = np.random.default_rng(0)
    nL = len(Hp.mMeshes)
    for fused in (1, 0):
        dev.set_option("fused", fused)
        for l in range(nL):
            A = Hp.mStiffness[l]
            N = A.shape[0]
            x = rng.standard_normal(N)
            b = rng.standard_normal(N)
            ref, mag, k = _rows(A, x)
            _assert_rows(dev.matvec(l, x), ref, mag, k, (name, fused, l, "matvec"))
            _assert_rows(dev.residual(l, x, b), b.astype(LD) - ref, mag + np.abs(b.astype(LD)), k + 1,
                         (name, fused, l, "residual"))
            # apply_smoother with the device's own block inverses (element blocks, (e, i, j) order)
            slots = Hp.mSlots[l]
            n, m = slots.shape
            dinv = Hp.level_blocks(l)[3]
            valid = slots >= 0
            be = np.zeros((n, m), dtype=LD)
            be[valid] = b[slots[valid]]
            alpha = 2.0 / 3.0
            if dinv.ndim == 2:
                ye, me, ke = dinv.astype(LD) * be, np.abs(dinv.astype(LD) * be), np.ones((n, m))
            else:
                D = dinv.astype(LD)
                ye = np.einsum("eij,ej->ei", D, be)
                me = np.einsum("eij,ej->ei", np.abs(D), np.abs(be))
                ke = np.full((n, m), m)
            ref, mag, k = np.zeros(N, dtype=LD), np.zeros(N, dtype=LD), np.zeros(N)
            ref[slots[valid]], mag[slots[valid]], k[slots[valid]] = LD(alpha) * ye[valid], LD(alpha) * me[valid], ke[valid] + 1
            _assert_rows(dev.apply_smoother(l, b, alpha=alpha), ref, mag, k, (name, fused, l, "apply_smoother"))
            if l < nL - 1:
                L = sp.csc_matrix(Hp.mInterpolation[l])
                ref, mag, k = _rows(L.T, x)
                _assert_rows(dev.restrict(l, x), ref, mag, k, (name, fused, l, "restrict"))
                xc = rng.standard_normal(L.shape[1])
                ref, mag, k = _rows(L, xc)
                _assert_rows(dev.prolong(l, xc), ref, mag, k, (name, fused, l, "prolong"))
    dev.set_option("fused", 1)
    # A_l \ b on every level: backward error of the GPU's direct solver
    for l in range(nL):
        A = sp.csr_matrix(Hp.mStiffness[l])
        b = rng.standard_normal(A.shape[0])
        x = dev.direct_solve(l, b)
        r, _, _ = _rows(A, x)
        berr = float(np.abs(b.astype(LD) - r).max()) / (abs(A).sum(axis=1).max() * np.abs(x).max())
        assert berr <= 64 * EPS * math.sqrt(A.shape[0]), (name, l, berr)


# ---- c. cycles against the oracle -----------------------------------------------------------------
def _assert_iterate_close(Ho, bo, x, x_or):
    """Two iterates that both stopped at 1e-10 ||b|| may differ by more than 1e-10 in the smoothest modes
    (cond(A) reaches 1e9 here); the GPU's must be within 1e-9, or as close to A \\ b as the oracle's is."""
    u = np.linalg.solve(sp.csc_matrix(Ho.mStiffness[0]).toarray(), bo)
    d = np.abs(x - x_or).max()
    assert d <= max(1e-9 * np.abs(x_or).max(), 2 * np.abs(x_or - u).max()), (d, np.abs(x_or - u).max())


def test_vcycles_match_the_oracle(case):
    name, Ho, bo, Hp, bp = case
    x_or = osolv.multigrid_v_cycle(Ho, np.zeros(len(bo)), bo)
    with dense_coarse_solver():
        noise = np.abs(osolv.multigrid_v_cycle(Ho, np.zeros(len(bo)), bo) - x_or).max() / np.abs(x_or).max()
    x0 = np.random.default_rng(1).standard_normal(len(bo)) * np.abs(x_or).max()
    for nPre, nPost, alpha in SWEEPS:
        for guess in (np.zeros(len(bo)), x0):
            x_or = osolv.multigrid_v_cycle(Ho, guess, bo, nPre=nPre, nPost=nPost, alpha=alpha)
            x = aggmg.multigrid_v_cycle(Hp, guess, bp, nPre=nPre, nPost=nPost, alpha=alpha)
            assert np.abs(x - x_or).max() <= max(1e-10, 20 * noise) * np.abs(x_or).max(), (name, nPre, nPost, alpha)
        # ldiv starts from zero inside the library: the same bits as the V-cycle from an explicit zero guess
        assert np.array_equal(Hp.device.ldiv(bp, nPre, nPost, alpha),
                              Hp.device.vcycle(np.zeros(len(bp)), bp, nPre, nPost, alpha)), (name, nPre, nPost)
    y = np.zeros(len(bp))
    aggmg.ldiv(y, Hp, bp)
    assert np.array_equal(y, aggmg.multigrid_v_cycle(Hp, np.zeros(len(bp)), bp))


def test_multigrid_matches_the_oracle(case):
    name, Ho, bo, Hp, bp = case
    x_or, it_or, res_or, _ = osolv.multigrid(Ho, np.zeros(len(bo)), bo, 100, 1e-10)
    x, it, res, _ = aggmg.multigrid(Hp, np.zeros(len(bp)), bp, 100, 1e-10, with_error=False)
    assert it == it_or, (name, it, it_or)
    floor = rounding_floor(Ho, x_or)
    with dense_coarse_solver():
        _, it_d, res_d, _ = osolv.multigrid(Ho, np.zeros(len(bo)), bo, 100, 1e-10)
    k = min(it_d, it_or)
    noise = np.zeros(it_or)
    noise[:k] = 20 * np.abs(res_d[:k] - res_or[:k])
    assert np.all(np.abs(res - res_or) <= np.maximum(np.maximum(1e-10 * res_or, floor), noise)), (name, res, res_or)
    _assert_iterate_close(Ho, bo, x, x_or)


def test_pcg_matches_the_oracle(case):
    name, Ho, bo, Hp, bp = case
    x_or, it_or, res_or = osolv.pcg(Ho, np.zeros(len(bo)), bo, 100, 1e-10)
    x, it, res = aggmg.pcg(Hp, np.zeros(len(bp)), bp, 100, 1e-10)
    floor = rounding_floor(Ho, x_or)
    with dense_coarse_solver():
        _, it_d, res_d = osolv.pcg(Ho, np.zeros(len(bo)), bo, 100, 1e-10)
    assert abs(it - it_or) <= (0 if it_d == it_or else 1), (name, it, it_or, it_d)
    k = min(it, it_or, it_d)
    noise = 20 * np.abs(res_d[:k] - res_or[:k])
    assert np.all(np.abs(res[:k] - res_or[:k]) <= np.maximum(np.maximum(1e-8 * res_or[:k], floor), noise)), (res, res_or)
    assert res[-1] < 1e-10 * np.linalg.norm(bp)
    assert np.abs(x - x_or).max() <= 1e-8 * np.abs(x_or).max()


# ---- d. tier matrix, bit for bit ------------------------------------------------------------------
def _tier_run(dev, x0, b, maxiter=30):
    out = [dev.vcycle(x0, b, *cyc) for cyc in SWEEPS[:2]] + [dev.ldiv(b)]
    x, it, res, _ = dev.solve(np.zeros(len(b)), b, maxiter, 1e-10)
    return out + [x, np.array([it]), np.asarray(res)]


def _assert_same(got, ref, tag, floor):
    """Iterates, ldiv and the solve's iterate and cycle count bit for bit.  The reported residual norms are
    two-stage reductions whose partition depends on the tier (fused into f_up or stand-alone), so they are
    held to 1e-11 as in test_gpu_parity.test_fused_and_generic_tiers_agree."""
    for i, (g, r) in enumerate(zip(got[:-1], ref[:-1])):
        assert np.array_equal(g, r), (tag, i)
    assert np.allclose(got[-1], ref[-1], rtol=1e-11, atol=floor), (tag, got[-1], ref[-1])


def _tier_matrix(H, b, tag, maxiter=30):
    dev = H.device
    x0 = np.random.default_rng(7).standard_normal(len(b))
    try:
        dev.set_option("leg_pipeline_min", 0)
        dev.set_option("fused", 0)
        dev.set_option("coarse_cta_elems", 0)
        ref = _tier_run(dev, x0, b, maxiter)
        floor = rounding_floor(H, ref[3])
        for fused in (0, 1):
            for tail in (0, DEFAULT_TAIL):
                for graph in (0, 1):
                    for key, val in (("fused", fused), ("coarse_cta_elems", tail), ("graph", graph)):
                        dev.set_option(key, val)
                    _assert_same(_tier_run(dev, x0, b, maxiter), ref, (tag, fused, tail, graph), floor)
        dev.set_option("fused", 1)
        for tail in (0, DEFAULT_TAIL):
            dev.set_option("coarse_cta_elems", tail)
            for vname, opts in VARIANTS:
                for key, val in opts.items():
                    dev.set_option(key, val)
                _assert_same(_tier_run(dev, x0, b, maxiter), ref, (tag, vname, tail), floor)
    finally:
        _reset(dev)
    return x0, ref, floor


def test_tier_matrix_bit_identical(case):
    name, Ho, bo, Hp, bp = case
    x0, ref, floor = _tier_matrix(Hp, bp, name)
    # uncompressed storage (every block dense, ST_DENSE) through the default tiers
    Hd, _ = build_package(upload=False, **build_kwargs(name))
    dense = Hd.upload(options={"compress": 0})
    try:
        assert all(dense.info(f"structure:{l}") == 0 for l in range(len(Hd.mMeshes)))
        _assert_same(_tier_run(dense, x0, bp), ref, (name, "compress=0"), floor)
        dense.set_option("fused", 0)
        dense.set_option("coarse_cta_elems", 0)
        _assert_same(_tier_run(dense, x0, bp), ref, (name, "compress=0, generic"), floor)
    finally:
        dense.close()


# ---- e. multi-column set ----------------------------------------------------------------------------
def test_multi_column_set_bit_identical(case):
    name, Ho, bo, Hp, bp = case
    dev = Hp.device
    N = len(bp)
    for k in (3, 8):
        rng = np.random.default_rng(k)
        X0, B = rng.standard_normal((N, k)), rng.standard_normal((N, k))
        B[:, 0] = bp
        B[:, k - 1] = 0.0
        for tail in (DEFAULT_TAIL, 0):
            dev.set_option("coarse_cta_elems", tail)
            _assert_columns_match(dev, X0, B, cycles=CYCLES if k == 3 else CYCLES[:2], tag=(name, k, tail))
            assert dev.info("multi_columns") == k
            assert dev.info("multi_launches_per_cycle") > 0
            # multigrid on every column (the zero column never meets the relative rule and runs maxiter cycles)
            maxiter, tol = 40, 1e-10
            dev.dev_set_problems(None, B)
            iters, res = dev.dev_solve_multi(maxiter, tol)
            X = dev.dev_get_solutions()
            for c in range(k):
                dev.dev_set_problem(None, B[:, c])
                it, r = dev.dev_solve(maxiter, tol)
                assert iters[c] == it, (name, k, tail, c, iters, it)
                assert np.array_equal(res[c], r), (name, k, tail, c)
                assert np.array_equal(X[:, c], dev.dev_get_solution()), (name, k, tail, c)
            assert iters[k - 1] == maxiter
            _assert_pcg_columns_match(dev, X0, B, maxiter=40, tag=(name, k, tail))
    dev.set_option("coarse_cta_elems", DEFAULT_TAIL)


# ---- f. device-side set-up ----------------------------------------------------------------------------
@pytest.mark.parametrize("name", [n for n, s in SHAPES.items() if s["pattern"] == "last1" and not s.get("cg_orders")])
def test_device_side_setup_single_parent(name):
    kw = build_kwargs(name)
    Ho, bo = build_oracle(**kw)
    Hh, bp = build_package(**kw)
    Hd, _ = build_package(**kw, device_setup=True)
    try:
        nL = len(Ho.mMeshes)
        for l in range(nL):
            got, ref = Hd.level_blocks(l), Hh.level_blocks(l)
            scale = np.abs(ref[1]).max()
            for g, r_, what in zip(got[:3], ref[:3], ("lo", "di", "up")):
                assert np.abs(g - r_).max() <= 1e-12 * scale, (name, l, what)
            assert np.abs(got[3] - ref[3]).max() <= 1e-10 * np.abs(ref[3]).max(), (name, l)
            assert Hd.device.info(f"structure:{l}") == Hh.device.info(f"structure:{l}"), l
        x_or, it_or, res_or, _ = osolv.multigrid(Ho, np.zeros(len(bo)), bo, 100, 1e-10)
        x, it, res, _ = aggmg.multigrid(Hd, np.zeros(len(bp)), bp, 100, 1e-10, with_error=False)
        assert it == it_or, (name, it, it_or)
        floor = rounding_floor(Ho, x_or)
        assert np.all(np.abs(res - res_or) <= np.maximum(1e-9 * res_or, floor)), (res, res_or)
        _assert_iterate_close(Ho, bo, x, x_or)
    finally:
        Hh.device.close()
        Hd.device.close()


@pytest.mark.parametrize("name", ["dg3_first1_n37", "dg3_mixed_n50", "pagg0_mixed_n50", "cg3_dg1_mixed_n50"])
def test_device_side_setup_refuses_other_maps(name):
    with pytest.raises(aggmg.Amg1dError, match="single-parent transfer"):
        build_package(**build_kwargs(name), device_setup=True)


# ---- g. at scale, judged by the C oracle fed the same host hierarchy ---------------------------------
@pytest.mark.parametrize("n", [2 ** 17 + 1, 3 * 2 ** 16 + 5])
def test_at_scale_against_the_c_oracle(n):
    from oracle import cref
    H, b = build_package(n, dg_orders=[3, 1], pattern="last1", upload=False)
    classes = [t["cls"] for t in transfer_classes(H)]
    assert classes[1] == "partial" and set(classes) == {"full", "partial"}, classes
    dev = H.upload()
    try:
        cycles = 6
        x, it, res, _ = dev.solve(np.zeros(len(b)), b, cycles, 0.0)
        assert it == cycles
        c = cref.CRefHierarchy(H)
        try:
            x_or = np.zeros(len(b))
            res_or = []
            for _ in range(cycles):
                x_or = c.vcycle(x_or, b)
                res_or.append(c.residual_norm(x_or, b))
        finally:
            c.close()
        res_or = np.array(res_or)
        A = sp.csr_matrix(H.mStiffness[0])
        floor = 8 * EPS * abs(A).sum(axis=1).max() * np.abs(x_or).max() * math.sqrt(len(b))
        assert np.all(np.abs(res - res_or) <= np.maximum(1e-10 * res_or, floor)), (n, res, res_or, floor)
        assert np.all(np.diff(res_or) < 0)
        # every tier and leg form, the pipelined legs running many windows per CTA over the partial elements
        _tier_matrix(H, b, n, maxiter=8)
    finally:
        dev.close()
