"""Host set-up parity on ragged agglomerations (tests/ragged_shapes.py): the product's assembly against the
oracle's literal restatement, and the transfer class of every level against the one its shape claims."""
import time

import numpy as np
import pytest
import scipy.sparse as sp

from agglomerationmultigrid1d_b200 import blocks as blk
from ragged_shapes import SHAPES, build_kwargs, build_oracle, build_package, size_chain, transfer_classes


@pytest.fixture(scope="module", params=sorted(SHAPES))
def pair(request):
    kw = build_kwargs(request.param)
    Ho, bo = build_oracle(**kw)
    Hp, bp = build_package(upload=False, **kw)
    return request.param, Ho, bo, Hp, bp


def test_sizes_are_ragged():
    for name, s in SHAPES.items():
        chain = size_chain(s["n"], s["pattern"])
        assert len(chain[-1]) == 1
        assert any(len(set(sizes)) > 1 for sizes in chain), name


def test_index_maps_bit_exact(pair):
    name, Ho, bo, Hp, bp = pair
    assert len(Ho.mMeshes) == len(Hp.mMeshes)
    for mo, mp in zip(Ho.mMeshes, Hp.mMeshes):
        nodes_o = np.stack([np.asarray(el.mNodesInd) for el in mo.mElements])
        assert np.array_equal(nodes_o, mp.mNodesInd)
        assert mo.mNumNodes == mp.mNumNodes
        if hasattr(mo.mElements[0], "mBaseElementInds"):
            for k, el in enumerate(mo.mElements):
                ep = mp.mElements[k]
                assert np.array_equal(np.asarray(el.mBaseElementInds) - 1, ep.mBaseElementInds)
                assert np.array_equal(np.asarray(el.mSubAggElementInds) - 1, ep.mSubAggElementInds)
    for So, Sp in zip(Ho.mSmoothers, Hp.mSmoothers):
        if hasattr(So, "mBlockInds"):
            assert np.array_equal(So.mBlockInds, Sp.mBlockInds)


def test_operators_agree(pair):
    name, Ho, bo, Hp, bp = pair
    assert np.abs(bo - bp).max() <= 1e-13 * np.abs(bo).max()
    for l, (So, Sp) in enumerate(zip(Ho.mStiffness, Hp.mStiffness)):
        assert So.shape == Sp.shape
        assert abs(So - Sp).max() <= 1e-13 * abs(So).max(), (name, l)
    for l, (Io, Ip) in enumerate(zip(Ho.mInterpolation, Hp.mInterpolation)):
        assert abs(sp.csc_matrix(Io) - sp.csc_matrix(Ip)).max() <= 1e-13, (name, l)


def test_transfer_classes_are_the_claimed_ones(pair):
    """The host replay of amg1d_set_transfer / amg1d_finalize puts every transfer in the class its shape
    names, and the block form of every transfer reproduces L (the arrays the library receives)."""
    name, Ho, bo, Hp, bp = pair
    tc = transfer_classes(Hp)
    assert [t["cls"] for t in tc] == SHAPES[name]["classes"], name
    for t in tc:
        assert t["fusable"] == (t["cls"] in ("full", "partial", "two_parent"))
        assert t["single_parent_uniform"] == (t["cls"] in ("full", "partial"))
        if t["cls"] == "partial":         # the last coarse element really is short of children
            assert np.count_nonzero(t["parent"] == t["n_coarse"] - 1) < t["ratio"]
    slots = [blk.level_slots(m) for m in Hp.mMeshes]
    for l, L in enumerate(Hp.mInterpolation):
        parent, P0, P1 = blk.transfer_to_blocks(L, slots[l], slots[l + 1])
        nc, mc = slots[l + 1].shape
        xc_host = np.random.default_rng(l).standard_normal(L.shape[1])
        xc = np.zeros((nc + 2, mc))
        valid = slots[l + 1] >= 0
        xc[1:-1][valid] = xc_host[slots[l + 1][valid]]
        xf = np.einsum("eij,ej->ei", P0, xc[parent + 1])
        if P1 is not None:
            xf += np.einsum("eij,ej->ei", P1, xc[parent + 2])
        ref = sp.csc_matrix(L) @ xc_host
        vf = slots[l] >= 0
        assert np.abs(xf[vf] - ref[slots[l][vf]]).max() <= 1e-13 * max(1.0, np.abs(ref).max())


def test_detection_rule_on_hand_made_maps():
    from ragged_shapes import detect_closed_form
    assert detect_closed_form([0, 0, 1, 1, 2]) == (True, 2, 0, 0)            # partial last element
    assert detect_closed_form([0, 1, 1, 2, 2]) == (True, 2, 1, 0)            # leading singleton
    assert detect_closed_form([0, 0, 1, 1, 1, 2]) == (True, 3, 1, 0)         # 2, 3, 1 fits a shifted formula
    assert detect_closed_form([0, 0, 1, 1, 1, 2, 3, 3, 3, 3])[0] is False    # 2, 3, 1, 4 does not
    assert detect_closed_form([0, 0, 0]) == (True, 3, 0, 0)
    assert detect_closed_form([-1, 0, 0, 1, 1]) == (True, 2, 1, -1)


def test_host_build_at_scale_feeds_the_c_oracle():
    """The at-scale GPU test builds DG 3 -> 1 with pairs and a trailing singleton on the host and hands that
    hierarchy to oracle/cref.CRefHierarchy: the C oracle accepts the package's objects and its V-cycle agrees
    with the Python oracle's on a small instance; the host build at 2^17 + 1 stays within a minute."""
    from oracle import cref
    from oracle import solvers as osolv
    kw = build_kwargs("dg3_last1_n37")
    Ho, bo = build_oracle(**kw)
    Hp, bp = build_package(upload=False, **kw)
    c = cref.CRefHierarchy(Hp)
    try:
        x = c.vcycle(np.zeros(len(bp)), bp)
        x_or = osolv.multigrid_v_cycle(Ho, np.zeros(len(bo)), bo)
        assert np.abs(x - x_or).max() <= 1e-10 * np.abs(x_or).max()
    finally:
        c.close()
    t0 = time.perf_counter()
    H, b = build_package(2 ** 17 + 1, dg_orders=[3, 1], pattern="last1", upload=False)
    assert time.perf_counter() - t0 < 60.0
    assert [t["cls"] for t in transfer_classes(H)][:3] == ["full", "partial", "partial"]
