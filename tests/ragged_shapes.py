"""Hierarchies whose agglomerates are not all the same size: explicit aggregate-size lists, one per
agglomerated level.  A mesh of 37 elements coarsened by pairs, for example, ends every level with a
one-element aggregate (37 -> 19 -> 10 -> 5 -> 3 -> 2 -> 1).  Each shape is built twice from the same
parameters, as in tests/shapes.py: by the oracle's literal restatement (1-based groups) and by the
product's host package (0-based groups).

The library classifies each transfer when it is uploaded (amg1d_set_transfer / amg1d_finalize), and the
class decides which kernels run.  ``transfer_classes`` replays that rule on the host, and every shape names
the classes it is meant to exercise, so that a shape cannot drift into another code path unnoticed:

  full              parent[e] = e / ratio, no P1, every coarse element has `ratio` children: fused legs, f_tail
  partial           the same with a last coarse element of fewer than `ratio` children
  shifted           parent[e] = (e + shift) / ratio, shift > 0: closed formula, generic tier
  open              no closed formula: generic tier through the child-pointer array
  two_parent        closed formula with P1 (CG -> CG): fused legs, no f_tail
  two_parent_open   P1 and no closed formula: generic two-parent path
"""
import math

import numpy as np

import agglomerationmultigrid1d_b200 as aggmg
from agglomerationmultigrid1d_b200 import blocks as blk
from oracle import aggdg as oagg
from oracle import cg as ocg
from oracle import dg as odg
from oracle import hierarchy as ohier
from oracle import refmesh


# ---- aggregate-size patterns: element count -> sizes of the aggregates of the next level ----------
def last1(cur):
    """Pairs, and a trailing one-element aggregate when the count is odd."""
    return [2] * (cur // 2) + [1] * (cur % 2)


def first1(cur):
    """A leading one-element aggregate, then pairs (and a trailing one when needed); three or fewer: one aggregate."""
    if cur <= 3:
        return [cur]
    return [1] + last1(cur - 1)


def mixed(cur):
    """Sizes cycling 2, 3, 1, 4, 2, the last one cut to what is left."""
    out, pat = [], (2, 3, 1, 4, 2)
    while sum(out) < cur:
        out.append(min(pat[len(out) % len(pat)], cur - sum(out)))
    return out


PATTERNS = {"last1": last1, "first1": first1, "mixed": mixed}


def size_chain(n, pattern):
    """Aggregate sizes of every agglomerated level, down to a single element."""
    fn = PATTERNS[pattern]
    out, cur = [], n
    while cur > 1:
        s = fn(cur)
        assert sum(s) == cur and min(s) >= 1
        out.append(s)
        cur = len(s)
    return out


def groups(sizes, one_based=False):
    out, s = [], 1 if one_based else 0
    for k in sizes:
        out.append(list(range(s, s + k)))
        s += k
    return out


# name -> build parameters, the class of every transfer (level l -> l + 1), and what the library reports
# for them: multi_legs (info "multi_legs:<l>" with the coarse tail off, one entry per transfer) and tail_start
# (info "tail_start" with the default coarse_cta_elems; -1 with it set to 0)
SHAPES = {
    "dg3_last1_n37": dict(
        n=37, dg_orders=[3, 1], pattern="last1",
        classes=["full", "partial", "partial", "full", "partial", "partial", "full"],
        multi_legs=[1] * 7, tail_start=1),
    "dg3_first1_n37": dict(
        n=37, dg_orders=[3, 1], pattern="first1",
        classes=["full"] + ["shifted"] * 5 + ["full"],
        multi_legs=[1] + [0] * 5 + [1], tail_start=6),
    "dg3_mixed_n50": dict(
        n=50, dg_orders=[3, 1], pattern="mixed",
        classes=["full"] + ["open"] * 3 + ["full"] * 2,
        multi_legs=[1, 0, 0, 0, 1, 1], tail_start=4),
    "cg3_dg1_mixed_n50": dict(
        n=50, cg_orders=[3, 1], dg_orders=[1], pattern="mixed",
        classes=["two_parent", "two_parent_open"] + ["open"] * 3 + ["full"] * 2,
        multi_legs=[1, 0, 0, 0, 0, 1, 1], tail_start=5),
    "cg1_last1_n37": dict(
        n=37, cg_orders=[1], pattern="last1",
        classes=["two_parent_open", "partial", "full", "partial", "partial", "full"],
        multi_legs=[0] + [1] * 5, tail_start=1),
    "dg4_last1_n481": dict(
        n=481, dg_orders=[4, 2, 1], pattern="last1",
        classes=["full"] * 2 + ["partial"] * 5 + ["full"] * 4,
        multi_legs=[1] * 11, tail_start=3),
    "dg3_last1_n961": dict(
        n=961, dg_orders=[3, 1], pattern="last1",
        classes=["full"] + ["partial"] * 6 + ["full"] * 4,
        multi_legs=[1] * 11, tail_start=3),
    "dg8_last1_n97": dict(
        n=97, dg_orders=[8, 4, 2, 1], pattern="last1",
        classes=["full"] * 3 + ["partial"] * 5 + ["full"] * 2,
        multi_legs=[0] + [1] * 9, tail_start=3),
    "pagg0_mixed_n50": dict(
        n=50, dg_orders=[3, 1], pattern="mixed", pAgg=0,
        classes=["full"] + ["open"] * 3 + ["full"] * 2,
        multi_legs=[1, 0, 0, 0, 1, 1], tail_start=4),
}

BUILD_KEYS = ("n", "cg_orders", "dg_orders", "pattern", "pAgg")


def build_kwargs(name):
    return {k: v for k, v in SHAPES[name].items() if k in BUILD_KEYS}


def _problem(n):
    return dict(xin=0.0, xout=1.0, CDir=1000.0 * n)


def build_oracle(n, cg_orders=(), dg_orders=(), pattern="last1", pAgg=1, sizes=None):
    """oracle/drivers.build_problem with explicit 1-based agglomeration maps."""
    pr = _problem(n)
    sizes = size_chain(n, pattern) if sizes is None else sizes
    mesh = refmesh.create_uniform_mesh(n, pr["xin"], pr["xout"])
    bd = refmesh.set_boundary(mesh, pr["xin"], pr["xout"], [("neu", -math.sin(pr["xin"])), ("dir", math.cos(pr["xout"]))])
    meshes = [ocg.CgMesh(mesh, p) for p in cg_orders] + [odg.DgMesh(mesh, p) for p in dg_orders]
    nCG, nDG = len(cg_orders), len(dg_orders)
    base = meshes[0] if nCG else meshes[nDG - 1]
    for i, s in enumerate(sizes):
        g = groups(s, one_based=True)
        meshes.append(oagg.AgglomeratedDgMesh1(pAgg, g, mesh, base) if i == 0
                      else oagg.AgglomeratedDgMeshN(pAgg, g, meshes[-1], base))
    bds = [bd] * len(meshes)
    if nCG:
        A, b = ocg.cg_stiffness_and_rhs(meshes[0], mesh, math.cos, bd)
        H = ohier.MeshHierarchyCG(meshes, mesh, bds, A, nCG=nCG, nDG=nDG, nAgg=len(sizes), CDir=pr["CDir"])
    else:
        A, b, G, D, C = odg.dg_operator_and_rhs(meshes[0], mesh, math.cos, bd, pr["CDir"])
        H = ohier.MeshHierarchyDG(meshes, bds, A, G, D, C, nDG=nDG, nAgg=len(sizes))
    return H, b


def build_package(n, cg_orders=(), dg_orders=(), pattern="last1", pAgg=1, sizes=None, upload=True,
                  device_setup=False):
    """The product's host path with explicit 0-based agglomeration maps."""
    pr = _problem(n)
    sizes = size_chain(n, pattern) if sizes is None else sizes
    mesh = aggmg.create_uniform_mesh(n, pr["xin"], pr["xout"])
    bd = aggmg.set_boundary(mesh, pr["xin"], pr["xout"], [("neu", -math.sin(pr["xin"])), ("dir", math.cos(pr["xout"]))])
    meshes = [aggmg.CgMesh(mesh, p) for p in cg_orders] + [aggmg.DgMesh(mesh, p) for p in dg_orders]
    nCG, nDG = len(cg_orders), len(dg_orders)
    base = meshes[0] if nCG else meshes[nDG - 1]
    for i, s in enumerate(sizes):
        g = groups(s)
        meshes.append(aggmg.AgglomeratedDgMesh1(pAgg, g, mesh, base) if i == 0
                      else aggmg.AgglomeratedDgMeshN(pAgg, g, meshes[-1], base))
    bds = [bd] * len(meshes)
    if nCG:
        A, b = aggmg.cg_stiffness_and_rhs(meshes[0], mesh, np.cos, bd)
        H = aggmg.MeshHierarchy(meshes, mesh, bds, A, nCG=nCG, nDG=nDG, nAgg=len(sizes), CDir=pr["CDir"],
                                upload=upload, device_setup=device_setup)
    else:
        G, D, C = aggmg.dg_flux_operators(meshes[0], mesh, bd, pr["CDir"])
        A = (C - D @ meshes[0].mMassMatrixLU.solve(G)).tocsc()
        f, r = aggmg.dg_flux_rhs(meshes[0], mesh, np.cos, bd, pr["CDir"])
        b = f - D @ meshes[0].mMassMatrixLU.solve(r)
        H = aggmg.MeshHierarchy(meshes, bds, A, G, D, C, nDG=nDG, nAgg=len(sizes), upload=upload,
                                device_setup=device_setup)
    return H, b


# ---- host replay of the library's transfer classification ----------------------------------------
def detect_closed_form(parent):
    """amg1d_set_transfer: fit parent[e] = (e + shift) / ratio + base from the first two runs of equal
    parents.  Returns (closed, ratio, shift, base); ratio 1, shift 0, base 0 when there is no closed form."""
    parent = np.asarray(parent, dtype=np.int64)
    n = len(parent)
    base = int(parent[0])
    c0 = 1
    while c0 < n and parent[c0] == base:
        c0 += 1
    c1 = 0
    while c0 + c1 < n and parent[c0 + c1] == base + 1:
        c1 += 1
    ratio = c1 if c0 + c1 < n else max(c0, c1)
    ratio = max(ratio, 1)
    shift = ratio - c0
    closed = ratio <= 1024 and 0 <= shift < ratio
    if closed:
        closed = bool(np.array_equal(parent, (np.arange(n) + shift) // ratio + base))
    return (closed, ratio, shift, base) if closed else (False, 1, 0, 0)


def transfer_classes(H):
    """Per transfer of a host hierarchy (upload=False): dict(cls, closed, ratio, shift, base, two_parent,
    fusable, single_parent_uniform, n_fine, n_coarse) - the rule of amg1d_set_transfer and amg1d_finalize."""
    slots = [blk.level_slots(m) for m in H.mMeshes]
    out = []
    for l, L in enumerate(H.mInterpolation):
        parent, P0, P1 = blk.transfer_to_blocks(L, slots[l], slots[l + 1])
        closed, ratio, shift, base = detect_closed_form(parent)
        n_fine, n_coarse = len(parent), slots[l + 1].shape[0]
        two = P1 is not None
        fusable = closed and -base * ratio - shift >= 0 and (n_coarse - 1 - base) * ratio - shift < n_fine
        spu = closed and not two and shift == 0 and base == 0
        if two:
            cls = "two_parent" if closed else "two_parent_open"
        elif not closed:
            cls = "open"
        elif shift or base:
            cls = "shifted"
        else:
            cls = "full" if n_coarse * ratio == n_fine else "partial"
        out.append(dict(cls=cls, closed=closed, ratio=ratio, shift=shift, base=base, two_parent=two,
                        fusable=fusable, single_parent_uniform=spu, n_fine=n_fine, n_coarse=n_coarse,
                        parent=parent))
    return out
