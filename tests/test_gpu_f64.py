"""BVHAccel<double> on the GPU (nrt_build_f64 / nrt_traverse_f64).  Checker: the unmodified reference's fp64
instantiation, through its results recorded in tests/golden (fingerprints in reference_digests.json, the reference's
regression program in regression30.npz) and through the oracle's double restatement pinned to them."""
import os

import numpy as np
import pytest

from helpers import REF_DIFF, hits_digest, reference_golden, tree_digest

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _ray64(org, d, min_t=0.0, max_t=1e30):
    from nanort_b200 import api

    r = np.zeros(1, api.RAY64_DTYPE)
    r["org"], r["dir"], r["min_t"], r["max_t"] = org, d, min_t, max_t
    return r


def test_regression30_in_double_matches_the_reference_bits():
    """test/regression/possible-accuracy-problem-30/main.cc:24-76 in its native precision: hit, u = 0.68,
    v = 0.131201, and t / u / v bit-equal to what the reference computed (tests/golden/regression30.npz)."""
    from nanort_b200 import api

    d = np.load(os.path.join(G, "regression30.npz"))
    acc = api.BVHAccelF64()
    assert acc.Build(1, d["verts"], d["faces"])
    org = np.array([-0.36, 7.93890843, 1.2160368])
    for k, dx in (("plain", 0.0), ("bug", -5.30287619e-17)):
        dd = np.array([dx, -8.66025404e-01, -0.5])
        dd = dd / np.sqrt((dd * dd).sum())
        h, m = acc.Traverse(_ray64(org, dd))
        want = d[f"f64_{k}"]  # [hit, t, u, v, prim]
        assert m[0] == 1 == int(want[0])
        assert (h["t"][0], h["u"][0], h["v"][0]) == (want[1], want[2], want[3]) and h["prim_id"][0] == int(want[4])
        assert abs(h["u"][0] - 0.68) < 1e-6 and abs(h["v"][0] - 0.131201) < 1e-6


def _scene64(seed=3):
    """Sphere grid with coordinates that do not survive a round trip through float."""
    from nanort_b200 import scenes as S

    v, f = S.sphere_grid(nx=3, nz=3)
    rng = np.random.default_rng(seed)
    v64 = v.astype(np.float64) * (1.0 + 1e-9 * rng.standard_normal(v.shape)) + 1e-11 * rng.standard_normal(v.shape)
    assert not np.array_equal(v64.astype(np.float32).astype(np.float64), v64)
    return v64, f


def _rays64(v64, n, seed):
    from nanort_b200 import api, scenes as S

    r32 = S.incoherent_rays(v64.min(axis=0).astype(np.float32), v64.max(axis=0).astype(np.float32), n, seed=seed)
    rng = np.random.default_rng(seed)
    r = np.zeros(n, api.RAY64_DTYPE)
    r["org"] = r32["org"].astype(np.float64) + 1e-10 * rng.standard_normal((n, 3))
    d = r32["dir"].astype(np.float64)
    nz = d != 0.0
    d = np.where(nz, d + 1e-12 * rng.standard_normal((n, 3)), d)  # keep the exact zeros / -0.0 of the family
    r["dir"] = d
    r["min_t"], r["max_t"] = r32["min_t"], r32["max_t"]
    return r


def test_f64_tree_is_valid_and_exact():
    from nanort_b200 import api

    v64, f = _scene64()
    acc = api.BVHAccelF64()
    acc.Build(len(f), v64, f)
    nodes, idx = acc.GetNodes(), acc.GetIndices()
    st = acc.GetStatistics()
    assert st["num_leaf_nodes"] == st["num_branch_nodes"] + 1 == (nodes["flag"] == 1).sum()
    assert np.array_equal(np.sort(idx), np.arange(len(f), dtype=np.uint32))
    tri = v64[f]  # (n, 3, 3)
    tmin, tmax = tri.min(axis=1), tri.max(axis=1)
    for i in np.nonzero(nodes["flag"] == 1)[0]:  # leaf boxes: exact double min / max of their triangles
        p = idx[nodes["data"][i, 1]: nodes["data"][i, 1] + nodes["data"][i, 0]]
        assert np.array_equal(nodes["bmin"][i], tmin[p].min(axis=0)) and np.array_equal(nodes["bmax"][i], tmax[p].max(axis=0))
    br = np.nonzero(nodes["flag"] == 0)[0]
    l, r = nodes["data"][br, 0], nodes["data"][br, 1]  # branch boxes: exact unions of their children
    assert np.array_equal(nodes["bmin"][br], np.minimum(nodes["bmin"][l], nodes["bmin"][r]))
    assert np.array_equal(nodes["bmax"][br], np.maximum(nodes["bmax"][l], nodes["bmax"][r]))
    a, b = acc.BoundingBox()
    assert np.array_equal(a, v64[f.ravel()].min(axis=0)) and np.array_equal(b, v64[f.ravel()].max(axis=0))


@pytest.mark.parametrize("cpp11", [True, False])
def test_f64_hits_match_the_reference(cpp11):
    from nanort_b200 import api
    from oracle import orc

    port = orc.Port64()
    v64, f = _scene64()
    rays = _rays64(v64, 60000, seed=4)
    acc = api.BVHAccelF64()
    acc.Build(len(f), v64, f)
    flags = api.TRAVERSE_CONFORMANCE | (0 if cpp11 else api.TRAVERSE_CPP03_INVERSE)
    gh, gm = acc.Traverse(rays, flags=flags)
    # (1) the reference's own Build + Traverse in double (the restatement's, checked against the reference's recorded
    # result): same hits; same bits for the same primitive
    rn, ri, _ = port.build(v64, f, None, orc.MODE_CPP11 if cpp11 else 0)
    rh, rm = port.traverse(rn, ri, v64, f, rays, cpp11=cpp11, threads=8)
    assert hits_digest(rh, rm) == reference_golden()[f"gpu_f64_hits/{cpp11}"], REF_DIFF
    assert rm.sum() > 5000 and np.array_equal(rm, gm)
    hit = rm == 1
    same = hit & (rh["prim_id"] == gh["prim_id"])
    for k in ("t", "u", "v"):
        assert np.array_equal(rh[k][same].view(np.uint64), gh[k][same].view(np.uint64)), k
    other = hit & ~same  # a different primitive only at exactly the same distance (shared edges)
    assert other.sum() <= 0.002 * hit.sum() and np.array_equal(rh["t"][other], gh["t"][other])
    # (2) the reference's Traverse walking the GPU's node array: everything bit-equal, ties included
    gn, gi = acc.GetNodes(), acc.GetIndices()
    ah, am = port.traverse(gn, gi, v64, f, rays, cpp11=cpp11, threads=8)
    assert np.array_equal(am, gm)
    for k in ("t", "u", "v", "prim_id"):
        assert ah[k][hit].tobytes() == gh[k][hit].tobytes(), k
    # (3) trace options
    o = orc.trace_options(cull_back_face=1, skip_prim_id=int(gh["prim_id"][hit][0]))
    gh2, gm2 = acc.Traverse(rays[:8000], options=o, flags=flags)
    ah2, am2 = port.traverse(gn, gi, v64, f, rays[:8000], topts=o, cpp11=cpp11, threads=4)
    assert np.array_equal(am2, gm2) and ah2[am2 == 1].tobytes() == gh2[gm2 == 1].tobytes()
    assert gm2.sum() < gm[:8000].sum()


@pytest.mark.parametrize("cpp11", [True, False])
def test_f64_adopted_reference_tree_is_bit_exact(cpp11):
    """BVHAccel<double>::Load path (nrt_adopt_f64): the CPU reference's own double tree walked on the GPU gives the
    reference's records bit for bit -- hit flag, prim_id (ties included), t, u, v.  The tree is the restatement's,
    which is the reference's (tests/golden/reference_digests.json)."""
    from nanort_b200 import api
    from oracle import orc

    want = reference_golden()[f"gpu_f64_adopted/{cpp11}"]
    port = orc.Port64()
    v64, f = _scene64(seed=9)
    rays = _rays64(v64, 40000, seed=10)
    rn, ri, _ = port.build(v64, f, None, orc.MODE_CPP11 if cpp11 else 0)
    assert tree_digest(rn, ri) == want["tree"], REF_DIFF
    rh, rm = port.traverse(rn, ri, v64, f, rays, cpp11=cpp11, threads=8)
    assert hits_digest(rh, rm) == want["hits"], REF_DIFF
    acc = api.BVHAccelF64()
    assert acc.Adopt(rn, ri, v64, f)
    gh, gm = acc.Traverse(rays, flags=api.TRAVERSE_CONFORMANCE | (0 if cpp11 else api.TRAVERSE_CPP03_INVERSE))
    assert rm.sum() > 3000 and np.array_equal(rm, gm)
    hit = rm == 1
    for k in ("t", "u", "v", "prim_id"):
        assert rh[k][hit].tobytes() == gh[k][hit].tobytes(), k
    a, b = acc.BoundingBox()
    assert a.tolist() == want["bbox"][0] and b.tolist() == want["bbox"][1]
    with pytest.raises(api.NanortB200Error):  # foreign data is validated
        bad = rn.copy()
        bad["data"][np.nonzero(bad["flag"] == 0)[0][0], 0] = len(bad) + 3
        api.BVHAccelF64().Adopt(bad, ri, v64, f)


@pytest.mark.parametrize("cpp11", [True, False])
def test_f64_against_the_c_restatement(cpp11):
    """The same checks with the oracle proper (oracle/liborc64.so, pinned to the reference by tests/test_oracle_f64.py):
    the port walking the GPU's BVHNode<double> array must reproduce the GPU's records bit for bit, and the GPU walking
    the port's own (reference-identical) tree must reproduce the port's."""
    from nanort_b200 import api
    from oracle import orc

    port = orc.Port64()
    v64, f = _scene64(seed=13)
    rays = _rays64(v64, 30000, seed=14)
    flags = api.TRAVERSE_CONFORMANCE | (0 if cpp11 else api.TRAVERSE_CPP03_INVERSE)
    acc = api.BVHAccelF64()
    acc.Build(len(f), v64, f)
    gh, gm = acc.Traverse(rays, flags=flags)
    ph, pm = port.traverse(acc.GetNodes(), acc.GetIndices(), v64, f, rays, cpp11=cpp11, threads=8)
    assert pm.sum() > 2000 and np.array_equal(pm, gm)
    for k in ("t", "u", "v", "prim_id"):
        assert ph[k][pm == 1].tobytes() == gh[k][gm == 1].tobytes(), k
    nodes, idx, _ = port.build(v64, f, None, orc.MODE_CPP11 if cpp11 else 0)
    adopted = api.BVHAccelF64()
    adopted.Adopt(nodes, idx, v64, f)
    ah, am = adopted.Traverse(rays, flags=flags)
    qh, qm = port.traverse(nodes, idx, v64, f, rays, cpp11=cpp11, threads=8)
    assert np.array_equal(qm, am)
    for k in ("t", "u", "v", "prim_id"):
        assert qh[k][qm == 1].tobytes() == ah[k][am == 1].tobytes(), k


def conformance_cases():
    from nanort_b200 import scenes as S
    from oracle import orc

    cases = [(_scene64(seed=21), None), (_scene64(seed=22), orc.build_options_f64(min_leaf_primitives=1, bin_size=16)),
             (_scene64(seed=23), orc.build_options_f64(max_tree_depth=6))]
    v, f = S.make_scene("cornell")
    cases.append(((v.astype(np.float64) * (1.0 + 1e-13), f), None))
    v, f = S.sphere_grid(nx=6, nz=5)  # 30,000 triangles: above min_primitives_for_parallel_build -> joined node order
    rng = np.random.default_rng(5)
    cases.append(((v.astype(np.float64) + 1e-10 * rng.standard_normal(v.shape), f), None))
    return cases


@pytest.mark.parametrize("cpp11", [True, False])
def test_f64_conformance_build_writes_the_references_arrays(cpp11):
    """nrt_build_f64_ex(NRT_BUILD_REFERENCE_TREE): the device writes the very BVHNode<double> array and indices_ that
    BVHAccel<double>::Build writes -- checked against the oracle's double instantiation (pinned to the unmodified
    reference's BVHAccel<double> by tests/test_oracle_f64.py) and against the reference's own trees (recorded fingerprints):
    every field of every node, every index, the statistics, for several scenes and option sets -- coordinates that do not
    survive a round trip through float, so a float-precision split decision would show."""
    from nanort_b200 import api, scenes as S
    from oracle import orc

    port = orc.Port64()
    mode = orc.MODE_CPP11 if cpp11 else 0
    flags = api.BUILD_REFERENCE_TREE | (0 if cpp11 else api.BUILD_REFERENCE_CPP03_ORDER)
    cases = conformance_cases()
    ref_trees = reference_golden()[f"gpu_f64_conformance/{cpp11}"]
    assert len(ref_trees) == len(cases)
    for ((v64, f), opts), ref_tree in zip(cases, ref_trees):
        want_nodes, want_idx, _ = port.build(v64, f, opts, mode)
        acc = api.BVHAccelF64()
        assert acc.Build(len(f), v64, f, options=opts, flags=flags)
        nodes, idx = acc.GetNodes(), acc.GetIndices()
        assert len(nodes) == len(want_nodes), (len(nodes), len(want_nodes))
        assert np.array_equal(idx, want_idx)
        for k in ("bmin", "bmax", "flag", "data"):
            assert nodes[k].tobytes() == want_nodes[k].tobytes(), k
        br = nodes["flag"] == 0
        assert np.array_equal(nodes["axis"][br], want_nodes["axis"][br])  # the reference leaves leaf.axis uninitialised
        st = acc.GetStatistics()
        assert st["num_leaf_nodes"] == int((nodes["flag"] == 1).sum()) and st["num_branch_nodes"] == int(br.sum())
        assert tree_digest(nodes, idx) == ref_tree, REF_DIFF
        # and the conformance walk over it gives the oracle's records, ties included
        rays = _rays64(v64, 5000, seed=31)
        tf = api.TRAVERSE_CONFORMANCE | (0 if cpp11 else api.TRAVERSE_CPP03_INVERSE)
        gh, gm = acc.Traverse(rays, flags=tf)
        ph, pm = port.traverse(want_nodes, want_idx, v64, f, rays, cpp11=cpp11, threads=8)
        assert np.array_equal(pm, gm)
        for k in ("t", "u", "v", "prim_id"):
            assert ph[k][pm == 1].tobytes() == gh[k][gm == 1].tobytes(), k


def _assert_fast_equals_conformance(rays, fh, fm, ch, cm, max_tie_fraction=0.002):
    """Same hit flags; the same primitive carries the same bits; a different primitive only at EXACTLY the same t."""
    assert np.array_equal(fm, cm)
    hit = cm == 1
    same = hit & (fh["prim_id"] == ch["prim_id"])
    for k in ("t", "u", "v"):
        assert np.array_equal(fh[k][same].view(np.uint64), ch[k][same].view(np.uint64)), k
    other = hit & ~same
    assert other.sum() <= max_tie_fraction * max(1, hit.sum()), (int(other.sum()), int(hit.sum()))
    assert np.array_equal(fh["t"][other].view(np.uint64), ch["t"][other].view(np.uint64))
    miss = ~hit
    assert np.all(fh["prim_id"][miss] == 0xFFFFFFFF)
    assert np.array_equal(fh["t"][miss].view(np.uint64), ch["t"][miss].view(np.uint64))  # max_t, NaN payloads included


@pytest.mark.parametrize("cpp11", [True, False])
@pytest.mark.parametrize("tree", ["production", "reference", "adopted"])
def test_f64_fast_kernel_matches_the_reference_order_kernel(cpp11, tree):
    """nrt_traverse_f64 default (persistent warps over PairNodeD / TriD, csrc/f64_fast.cuh) against
    NRT_TRAVERSE_CONFORMANCE on the same accel -- which the tests above pin to the reference's BVHAccel<double>: the
    production tree, the reference's own tree built on the device (depth > 64: the deep-stack instantiation) and an
    adopted CPU tree; trace options; hostile rays."""
    from nanort_b200 import api
    from oracle import orc

    v64, f = _scene64(seed=21)
    rays = _rays64(v64, 50000, seed=22)
    # hostile rays: NaN / inverted ranges, zero and axis-parallel directions, huge and denormal components, min_t > 0
    # (NaN / inf ray COMPONENTS make the reference's own answer depend on its visiting order: a NaN t is accepted and then
    # poisons its box test; they are left to the reference-order kernel)
    h = rays[:64].copy()
    h["min_t"][0], h["max_t"][1] = np.nan, np.nan
    h["min_t"][2], h["max_t"][2] = 5.0, 1.0
    h["dir"][3] = 0.0
    h["dir"][4] = (1.0, 0.0, 0.0)
    h["dir"][5] = (0.0, -0.0, 1.0)
    h["dir"][6] = (1e-320, 1.0, 0.0)
    h["org"][7] = (1e300, 0.0, 0.0)
    h["dir"][8] *= 1e-8
    h["min_t"][9:20] = 0.75
    h["max_t"][20:30] = 0.5
    rays = np.concatenate([rays, h])
    acc = api.BVHAccelF64()
    if tree == "production":
        assert acc.Build(len(f), v64, f)
    elif tree == "reference":
        assert acc.Build(len(f), v64, f, flags=api.BUILD_REFERENCE_TREE)
    else:
        port = orc.Port64()
        nodes, idx, _ = port.build(v64, f, None, orc.MODE_CPP11 if cpp11 else 0)
        assert acc.Adopt(nodes, idx, v64, f)
    inv = 0 if cpp11 else api.TRAVERSE_CPP03_INVERSE
    ch, cm = acc.Traverse(rays, flags=api.TRAVERSE_CONFORMANCE | inv)
    fh, fm = acc.Traverse(rays, flags=api.TRAVERSE_FAST | inv)
    assert cm.sum() > 3000
    _assert_fast_equals_conformance(rays, fh, fm, ch, cm)
    # trace options: back-face culling, a skipped primitive, a primitive id window
    hit_prims = ch["prim_id"][cm == 1]
    for o in (orc.trace_options(cull_back_face=1), orc.trace_options(skip_prim_id=int(hit_prims[0])),
              orc.trace_options(prim_ids_range=(len(f) // 4, len(f) // 2))):
        ch2, cm2 = acc.Traverse(rays[:12000], options=o, flags=api.TRAVERSE_CONFORMANCE | inv)
        fh2, fm2 = acc.Traverse(rays[:12000], options=o, flags=inv)
        _assert_fast_equals_conformance(rays[:12000], fh2, fm2, ch2, cm2)
    # more rays than one pipeline chunk (three stream slots): every record lands in its place
    big = np.tile(rays[:40000], 30)[: (1 << 20) + 12345]
    bh, bm = acc.Traverse(big, flags=inv)
    assert np.array_equal(bm[: len(fm[:40000])], fm[:40000]) and np.array_equal(bm[40000:80000], fm[:40000])
    assert bh[1 << 20:].tobytes() == np.tile(fh[:40000], 30)[1 << 20: (1 << 20) + 12345].tobytes()


def test_f64_fast_kernel_on_a_single_leaf_tree_and_empty_input():
    from nanort_b200 import api

    v64 = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], np.float64)
    f = np.array([[0, 1, 2], [0, 1, 3]], np.uint32)
    acc = api.BVHAccelF64()
    assert acc.Build(len(f), v64, f)
    rays = np.zeros(3, api.RAY64_DTYPE)
    rays["org"] = [(0.2, 0.2, 1.0), (0.2, -1.0, 0.2), (5.0, 5.0, 5.0)]
    rays["dir"] = [(0, 0, -1.0), (0, 1.0, 0), (0, 0, 1.0)]
    rays["max_t"] = 1e30
    fh, fm = acc.Traverse(rays)
    ch, cm = acc.Traverse(rays, flags=api.TRAVERSE_CONFORMANCE)
    assert fm.tolist() == [1, 1, 0] and fh.tobytes() == ch.tobytes()
    eh, em = acc.Traverse(rays[:0])
    assert len(eh) == 0
