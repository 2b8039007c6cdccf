"""Repeated-column / repeated-row storage of the agglomerated 2 x 2 levels (structure class 3, ST_REPEAT in
csrc/layout.cuh).

Below a DG p = 1 level, every pAgg = 1 agglomerated level has off-diagonal blocks whose columns (A_lo) and rows
(A_up) are bitwise equal, so the device keeps one column and one row instead of the whole blocks (12 instead of 16
doubles per element).  The dense FMA chains then run on the same operand values, so every result must be
BIT-IDENTICAL to the dense storage (option compress = 0) - compared with np.array_equal / ==, never with a
tolerance.  The class is detected bitwise on levels uploaded as patterns: one ulp off in one element keeps the level
dense."""
import numpy as np
import pytest

import bench
from agglomerationmultigrid1d_b200 import blocks as blk
from agglomerationmultigrid1d_b200.device import DeviceHierarchy

pytestmark = pytest.mark.gpu

# workload shape, elements, first agglomerated level (its structure class is 3 down to the last level with more
# than one element)
SHAPES = {"T": (1 << 14, 2), "C4": (1 << 14, 3)}


def _zero_pattern_class(lo, up):
    """The class the compressed storage had before ST_REPEAT: structural zeros only (blocks in (e, i, j) order)."""
    lo_col, lo_row = (lo != 0).any(axis=(0, 1)), (lo != 0).any(axis=(0, 2))
    up_col, up_row = (up != 0).any(axis=(0, 1)), (up != 0).any(axis=(0, 2))
    if lo.shape[1] >= 2 and lo_col.sum() <= 1 and up_row.sum() <= 1:
        return 1
    if lo.shape[1] >= 2 and lo_row.sum() <= 1 and up_col.sum() <= 1:
        return 2
    return 0


def _problem(U, n):
    pr = bench.problem(n)
    return bench.rhs_slab(U, pr, 0, 1)


@pytest.fixture(scope="module", params=sorted(SHAPES))
def pair(request):
    name = request.param
    n, first_agg = SHAPES[name]
    U = bench.build_hierarchy(name, n)
    dev = U.upload()
    dense = U.upload(options={"compress": 0})
    yield name, U, first_agg, dev, dense, _problem(U, n)
    dev.close()
    dense.close()


def test_agglomerated_levels_store_one_column_and_one_row(pair):
    name, U, first_agg, dev, dense, _ = pair
    for l, lv in enumerate(U.levels):
        lo, _, up = U.level_blocks(l)
        st, rows = dev.info(f"structure:{l}"), dev.info(f"tile_rows:{l}")
        assert dense.info(f"structure:{l}") == 0
        if l >= first_agg and lv.n > 1 and dev.info(f"pattern:{l}") == 1:
            assert lv.m == 2
            assert st == 3 and rows == 12, (name, l, st, rows)
            assert dense.info(f"tile_rows:{l}") == 16
        else:
            assert st == _zero_pattern_class(lo, up), (name, l, st)
    assert dev.info(f"pattern:{first_agg}") == 1


def test_dense_p1_levels_keep_their_class():
    """P8 shape: the DG p = 1 level is assembled dense (entries of 5e-17 instead of zeros) and no level below it
    has bitwise-repeated columns and rows."""
    U = bench.build_hierarchy("P8", 1 << 10)
    dev = U.upload()
    try:
        for l in range(len(U.levels)):
            lo, _, up = U.level_blocks(l)
            assert dev.info(f"structure:{l}") == _zero_pattern_class(lo, up), l
            assert dev.info(f"structure:{l}") != 3, l
    finally:
        dev.close()


def _upload_level(lo, di, up, diag=False, pattern=True):
    """One level; pattern: every element's blocks as a block set of its own (n_head = n - 1, n_tail = 0)."""
    dev = DeviceHierarchy(1)
    dinv = (1.0 / np.einsum("eii->ei", di)) if diag else blk.to_abi(np.linalg.inv(di))
    n = di.shape[0]
    if pattern:
        dev.set_level_pattern(0, n, lo, di, up, dinv, diag, n - 1, 0)
    else:
        dev.set_level_blocks(0, lo, di, up, dinv, diag)
    return dev


def test_detection_is_bitwise():
    U = bench.build_hierarchy("T", 1 << 10)
    lo, di, up = (np.array(a, copy=True) for a in U.level_blocks(3))
    assert lo.shape[1] == 2
    cases = [("as assembled", lo, up, False, 3), ("point Jacobi", lo, up, True, 0)]
    dev = _upload_level(lo, di, up, pattern=False)                 # explicit levels keep the zero-pattern classes
    try:
        assert dev.info("structure:0") == 0
    finally:
        dev.close()
    e = lo.shape[0] // 2
    lo1 = lo.copy()
    lo1[e, 0, 1] = np.nextafter(lo1[e, 0, 1], np.inf)              # one A_lo entry one ulp off in one element
    cases.append(("A_lo one ulp", lo1, up, False, 0))
    up1 = up.copy()
    up1[e, 1, 0] = np.nextafter(up1[e, 1, 0], -np.inf)             # one A_up entry one ulp off in one element
    cases.append(("A_up one ulp", lo, up1, False, 0))
    for what, a_lo, a_up, diag, want in cases:
        dev = _upload_level(a_lo, di, a_up, diag)
        try:
            assert dev.info("structure:0") == want, what
        finally:
            dev.close()


def _same_level0_tier(dev, dense):
    """compress = 0 also changes level 0 of C4 (CG p = 3 groups, point Jacobi): its dense form has no fused leg and
    takes the generic tier, whose ||b - A x|| and dot products are summed in another order.  Residual histories and
    conjugate gradients are compared where level 0 runs the same kernels in both handles."""
    return dev.info("multi_legs:0") == dense.info("multi_legs:0")


def test_bit_identical_to_dense_storage(pair):
    name, U, first_agg, dev, dense, b = pair
    norms = _same_level0_tier(dev, dense)
    rng = np.random.default_rng(17)
    x0 = rng.standard_normal(len(b))
    for fused in (0, 1):
        dev.set_option("fused", fused)
        dense.set_option("fused", fused)
        assert np.array_equal(dev.vcycle(x0, b), dense.vcycle(x0, b)), (name, fused)
        assert np.array_equal(dev.vcycle(x0, b, nPre=1, nPost=2, alpha=0.7),
                              dense.vcycle(x0, b, nPre=1, nPost=2, alpha=0.7)), (name, fused)
        x_c, it_c, res_c, _ = dev.solve(np.zeros(len(b)), b, 30, 1e-10)
        x_d, it_d, res_d, _ = dense.solve(np.zeros(len(b)), b, 30, 1e-10)
        assert it_c == it_d and np.array_equal(x_c, x_d), (name, fused)
        assert np.array_equal(res_c, res_d) or not (norms or fused == 0), (name, fused)
        for l in range(len(U.levels)):
            v = rng.standard_normal(dev.n_dof[l])
            assert np.array_equal(dev.matvec(l, v), dense.matvec(l, v)), (name, fused, l)
    dev.set_option("fused", 1)
    dense.set_option("fused", 1)
    ref = dense.vcycle(x0, b)
    x_ref, it_ref, res_ref, _ = dense.solve(np.zeros(len(b)), b, 30, 1e-10)
    for mode in (1, 2):                                            # pattern-resident legs (table / by-value operand)
        dev.set_option("pattern_resident", mode)
        assert np.array_equal(dev.vcycle(x0, b), ref), (name, mode)
        x, it, res, _ = dev.solve(np.zeros(len(b)), b, 30, 1e-10)
        assert it == it_ref and np.array_equal(x, x_ref) and (np.array_equal(res, res_ref) or not norms), (name, mode)
    dev.set_option("pattern_resident", 0)
    # the legs that invert the 2 x 2 blocks in registers: one window per CTA, and persistent pipelined
    for opts in (dict(dinv_registers=2), dict(leg_pipeline=2, leg_pipeline_min=0)):
        for k, v in opts.items():
            dev.set_option(k, v)
        assert np.array_equal(dev.vcycle(x0, b), ref), (name, opts)
        x, it, res, _ = dev.solve(np.zeros(len(b)), b, 30, 1e-10)
        assert it == it_ref and np.array_equal(x, x_ref) and (np.array_equal(res, res_ref) or not norms), (name, opts)
        dev.set_option("dinv_registers", 0)
        dev.set_option("leg_pipeline", 1)
        dev.set_option("leg_pipeline_min", 500000)


def test_multi_column_bit_identical_to_dense_storage(pair):
    name, U, first_agg, dev, dense, b = pair
    rng = np.random.default_rng(23)
    X0 = rng.standard_normal((len(b), 3))
    B = np.column_stack([b, rng.standard_normal(len(b)), rng.standard_normal(len(b))])
    out = []
    for d in (dev, dense):
        d.dev_set_problems(X0, B)
        d.dev_vcycle_multi(with_residual_norms=True)
        X, norms = d.dev_get_solutions(), d.dev_residual_norms()
        d.dev_set_problems(None, B)
        iters, hist = d.dev_pcg_multi(20, 1e-10)
        out.append((X, norms, iters, hist, d.dev_get_solutions()))
    (X, n1, it1, h1, S1), (Xd, n2, it2, h2, S2) = out
    assert dev.info("multi_columns") == 3
    assert all(dev.info(f"multi_legs:{l}") == dense.info(f"multi_legs:{l}") for l in range(1, len(U.levels)))
    assert np.array_equal(X, Xd), name
    if _same_level0_tier(dev, dense):
        assert np.array_equal(n1, n2), name
        assert it1 == it2 and all(np.array_equal(a, c) for a, c in zip(h1, h2)) and np.array_equal(S1, S2), name
