"""CPU: the C restatement instantiated for double (oracle/liborc64.so) against the unmodified reference's
BVHAccel<double>: record sizes, node array, indices_, and every hit record, bit for bit, in both build modes /
vsafe_inverse conventions (the reference's results as fingerprints, tests/golden/reference_digests.json); plus the
reference's regression program in its native precision."""
import os

import numpy as np
import pytest

from helpers import REF_DIFF, hits_digest, reference_golden, tree_digest
from nanort_b200 import scenes as S
from oracle import orc

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SCENES = [("cornell", {}), ("sphere_grid", dict(nx=3, nz=3)), ("terrain", dict(n=80))]
BUILD_VARIANTS = (dict(min_leaf_primitives=1), dict(bin_size=8, min_leaf_primitives=8), dict(max_tree_depth=6),
                  dict(shallow_depth=2, min_primitives_for_parallel_build=1000))
TRACE_VARIANTS = (dict(cull_back_face=1), dict(skip_prim_id=17), dict(prim_ids_range=(100, 900)))


def _scene64(name, kw, seed):
    v, f = S.make_scene(name, **kw)
    rng = np.random.default_rng(seed)
    v64 = v.astype(np.float64) * (1.0 + 1e-9 * rng.standard_normal(v.shape)) + 1e-11 * rng.standard_normal(v.shape)
    return v64, f


def _rays64(v64, n, seed, hostile=False):
    if hostile:
        from edge_cases import hostile_rays

        r32 = hostile_rays(v64.min(axis=0).astype(np.float32) - 1, v64.max(axis=0).astype(np.float32) + 1, n=n, seed=seed)
    else:
        r32 = S.incoherent_rays(v64.min(axis=0).astype(np.float32), v64.max(axis=0).astype(np.float32), n, seed=seed)
    rng = np.random.default_rng(seed)
    r = np.zeros(n, orc.RAY64_DTYPE)
    r["org"] = r32["org"].astype(np.float64) * (1.0 + 1e-12 * rng.standard_normal((n, 3)))
    d = r32["dir"].astype(np.float64)
    r["dir"] = np.where((d != 0.0) & np.isfinite(d), d * (1.0 + 1e-13 * rng.standard_normal((n, 3))), d)
    r["min_t"], r["max_t"] = r32["min_t"], r32["max_t"]
    return r


@pytest.mark.parametrize("name,kw", SCENES)
@pytest.mark.parametrize("cpp11", [True, False])
def test_port64_equals_reference_double(name, kw, cpp11):
    g = reference_golden()
    port = orc.Port64()
    assert g["ref64_sizes"] == port.sizes() == [64, 72, 32, 32, 16]
    want = g[f"f64_vs_ref/{name}/{cpp11}"]
    v64, f = _scene64(name, kw, seed=2)
    nodes, idx, st = port.build(v64, f, None, orc.MODE_CPP11 if cpp11 else 0)
    assert tree_digest(nodes, idx) == want["tree"], REF_DIFF
    assert st["num_leaf_nodes"] == st["num_branch_nodes"] + 1
    for hostile in (False, True):
        rays = _rays64(v64, 12000, seed=6, hostile=hostile)
        ph, pm = port.traverse(nodes, idx, v64, f, rays, cpp11=cpp11, threads=4)
        assert hits_digest(ph, pm) == want[f"hits/{hostile}"], (hostile, REF_DIFF)
    assert pm.sum() > 100


def test_port64_build_options_and_trace_options():
    g = reference_golden()
    port = orc.Port64()
    v64, f = _scene64("sphere_grid", dict(nx=2, nz=2), seed=4)
    for okw in BUILD_VARIANTS:
        nodes, idx, _ = port.build(v64, f, orc.build_options_f64(**okw), orc.MODE_CPP11)
        assert tree_digest(nodes, idx) == g[f"f64_vs_ref_options/{sorted(okw.items())}"], (okw, REF_DIFF)
    rays = _rays64(v64, 6000, seed=8)
    for tkw in TRACE_VARIANTS:  # on the tree of the last build option set
        ph, pm = port.traverse(nodes, idx, v64, f, rays, topts=orc.trace_options(**tkw))
        assert hits_digest(ph, pm) == g[f"f64_vs_ref_options/{sorted(tkw.items())}"], (tkw, REF_DIFF)


def test_port64_regression30_native_precision():
    """test/regression/possible-accuracy-problem-30/main.cc:24-76: hit, u = 0.68, v = 0.131201 -- against the golden
    values the reference produced (tests/golden/regression30.npz)."""
    d = np.load(os.path.join(G, "regression30.npz"))
    port = orc.Port64()
    nodes, idx, _ = port.build(d["verts"], d["faces"], None, orc.MODE_CPP11)
    org = np.array([-0.36, 7.93890843, 1.2160368])
    for k, dx in (("plain", 0.0), ("bug", -5.30287619e-17)):
        dd = np.array([dx, -8.66025404e-01, -0.5])
        dd = dd / np.sqrt((dd * dd).sum())
        r = np.zeros(1, orc.RAY64_DTYPE)
        r["org"], r["dir"], r["min_t"], r["max_t"] = org, dd, 0.0, 1e30
        h, m = port.traverse(nodes, idx, d["verts"], d["faces"], r)
        want = d[f"f64_{k}"]
        assert m[0] == 1 and (h["t"][0], h["u"][0], h["v"][0]) == (want[1], want[2], want[3])
