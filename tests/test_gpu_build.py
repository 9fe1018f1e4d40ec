"""GPU builder: structural invariants, statistics, cross-walks against the oracle."""
import numpy as np
import pytest

from helpers import REF_DIFF, assert_parity, check_tree_structure, compare_hits, hits_digest, reference_golden

pytestmark = pytest.mark.gpu


def _degenerate(kind):
    if kind == "one":
        v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
        return v, np.array([[0, 1, 2]], np.uint32)
    if kind == "five":
        v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [2, 0, 1], [3, 1, 1], [2, 2, 2], [5, 5, 5]], np.float32)
        return v, np.array([[0, 1, 2], [1, 2, 3], [2, 3, 4], [3, 4, 5], [4, 5, 6]], np.uint32)
    if kind == "identical":  # 3000 copies of one triangle: no plane separates the centroids -> median cuts
        v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
        return v, np.tile(np.array([[0, 1, 2]], np.uint32), (3000, 1))
    if kind == "line":  # centroids on a line along x only
        k = 700
        x = np.arange(k, dtype=np.float32)
        v = np.stack([np.stack([x, 0 * x, 0 * x], 1), np.stack([x + 0.5, 0 * x, 0 * x + 1], 1),
                      np.stack([x, 0 * x + 1, 0 * x], 1)], 1).reshape(-1, 3)
        return v.astype(np.float32), np.arange(3 * k, dtype=np.uint32).reshape(k, 3)
    raise KeyError(kind)


CASES = [
    ("cornell", {}, {}),
    ("sphere_grid", dict(nx=3, nz=3), {}),
    ("sphere_grid", dict(nx=3, nz=3), dict(min_leaf_primitives=1)),
    ("sphere_grid", dict(nx=3, nz=3), dict(min_leaf_primitives=8, bin_size=8)),
    ("sphere_grid", dict(nx=3, nz=3), dict(max_tree_depth=5)),
    ("terrain", dict(n=96), dict(bin_size=16)),
    ("terrain", dict(n=96), dict(bin_size=256)),          # largest bin count: 47 KB of shared memory in the middle phase
    ("terrain", dict(n=30), {}),                          # 1,682 triangles: the root itself is a middle-phase node
    ("terrain", dict(n=40), dict(min_leaf_primitives=1)),  # one level-synchronous pass, then middle-phase nodes; 1-primitive leaves
    ("terrain", dict(n=96), dict(max_tree_depth=9)),      # the depth limit is reached inside the middle phase
    ("terrain", dict(n=96), dict(max_tree_depth=13)),     # ... and inside the warp-built subtrees
    ("sphere_grid", {}, {}),
    ("deg:one", {}, {}),
    ("deg:five", {}, {}),
    ("deg:identical", {}, {}),
    ("deg:line", {}, dict(min_leaf_primitives=2)),
]


def _scene(name, kw):
    from nanort_b200 import scenes as S

    if name.startswith("deg:"):
        return _degenerate(name[4:])
    return S.make_scene(name, **kw)


@pytest.mark.parametrize("name,kw,okw", CASES)
def test_built_tree_structure_and_stats(name, kw, okw):
    from nanort_b200 import api

    v, f = _scene(name, kw)
    opts = api.BVHBuildOptions(**okw)
    acc = api.BVHAccel()
    assert acc.Build(len(f), v, f, opts)
    nodes, idx = acc.GetNodes(), acc.GetIndices()
    st = check_tree_structure(nodes, idx, v, f, min_leaf=int(opts["min_leaf_primitives"][0]),
                              max_depth=int(opts["max_tree_depth"][0]))
    got = acc.GetStatistics()
    for k in ("max_tree_depth", "num_leaf_nodes", "num_branch_nodes"):
        assert got[k] == st[k], (k, got, st)
    assert got["build_secs"] > 0
    bmin, bmax = acc.BoundingBox()
    assert np.array_equal(bmin, nodes["bmin"][0]) and np.array_equal(bmax, nodes["bmax"][0])
    # deterministic: a second build gives the same arrays (every rank of a multi-GPU job rebuilds)
    acc2 = api.BVHAccel()
    acc2.Build(len(f), v, f, opts)
    assert np.array_equal(acc2.GetNodes().view(np.uint8), nodes.view(np.uint8))
    assert np.array_equal(acc2.GetIndices(), idx)


def test_build_zero_primitives_returns_false():
    from nanort_b200 import api

    acc = api.BVHAccel()
    assert acc.Build(0, np.zeros((3, 3), np.float32), np.zeros((0, 3), np.uint32)) is False
    assert not acc.IsValid()
    bmin, bmax = acc.BoundingBox()
    assert np.all(bmin == np.finfo(np.float32).max) and np.all(bmax == -np.finfo(np.float32).max)


@pytest.mark.parametrize("name,kw", [("cornell", {}), ("sphere_grid", dict(nx=4, nz=4)), ("terrain", dict(n=128))])
def test_cross_walk_oracle_over_gpu_tree_and_gpu_over_gpu_tree(port, name, kw):
    """(1) the oracle's Traverse over the GPU-built arrays and (2) the GPU kernels over them both give the
    hits the oracle finds on the CPU-built reference tree (hits do not depend on topology, SURVEY.md F1)."""
    from oracle import orc
    from nanort_b200 import api, scenes as S

    v, f = S.make_scene(name, **kw)
    cam = S.scene_camera(name, 256, 192)
    rays = np.concatenate([S.primary_rays(cam, 256, 192, spp=1, seed=3),
                           S.incoherent_rays(v.min(axis=0), v.max(axis=0), 80000, seed=9)])
    rn, ri, _ = port.build(v, f, mode=orc.MODE_CPP11)
    want_h, want_m = port.traverse(rn, ri, v, f, rays, threads=8)
    acc = api.BVHAccel()
    acc.Build(len(f), v, f)
    gn, gi = acc.GetNodes(), acc.GetIndices()
    o_h, o_m = port.traverse(gn, gi, v, f, rays, threads=8)
    assert_parity(compare_hits(port, v, f, rays, o_h, o_m, want_h, want_m))
    for flags in (api.TRAVERSE_FAST, api.TRAVERSE_CONFORMANCE):
        g_h, g_m = acc.Traverse(rays, flags=flags)
        assert_parity(compare_hits(port, v, f, rays, g_h, g_m, want_h, want_m))
    # conformance walk of the GPU tree == oracle walk of the GPU tree, bit for bit, ties included
    c_h, c_m = acc.Traverse(rays, flags=api.TRAVERSE_CONFORMANCE)
    assert np.array_equal(c_m, o_m)
    hit = o_m.astype(bool)
    assert np.array_equal(c_h[hit].view(np.uint32), o_h[hit].view(np.uint32))


def test_reference_traverses_gpu_built_tree(port):
    """The reference's Traverse (the oracle's restatement of it), walking the GPU-built arrays, finds the same hits as
    the unmodified reference on its own tree (recorded in tests/golden/reference_digests.json)."""
    from nanort_b200 import api, scenes as S

    v, f = S.make_scene("sphere_grid", nx=3, nz=3)
    cam = S.scene_camera("sphere_grid", 200, 150)
    rays = S.primary_rays(cam, 200, 150, spp=1, seed=4)
    rn, ri, _ = port.build(v, f)
    want_h, want_m = port.traverse(rn, ri, v, f, rays, threads=4)
    assert hits_digest(want_h, want_m) == reference_golden()["gpu_build_own_tree_hits"], REF_DIFF
    acc = api.BVHAccel()
    acc.Build(len(f), v, f)
    got_h, got_m = port.traverse(acc.GetNodes(), acc.GetIndices(), v, f, rays, threads=4)
    assert_parity(compare_hits(port, v, f, rays, got_h, got_m, want_h, want_m))


def _random_soup(rng, n):
    """Clustered triangle soup: cluster centres on very different scales, many coincident centroids, some slivers."""
    k = int(rng.integers(1, 6))
    centres = rng.normal(0, 10.0 ** rng.uniform(-2, 2), (k, 3))
    which = rng.integers(0, k, n)
    spread = 10.0 ** rng.uniform(-3, 0.5, k)
    c = centres[which] + rng.normal(0, 1, (n, 3)) * spread[which][:, None]
    dup = rng.random(n) < 0.15  # exact duplicates of another triangle's centroid position
    c[dup] = c[rng.integers(0, n, int(dup.sum()))]
    size = 10.0 ** rng.uniform(-3, 0, (n, 1, 1))
    tri = c[:, None, :] + rng.normal(0, 1, (n, 3, 3)) * size
    flat = rng.random(n) < 0.1  # axis-aligned flat triangles: zero-thickness boxes
    tri[flat, :, int(rng.integers(0, 3))] = c[flat, int(rng.integers(0, 3))][:, None]
    v = tri.reshape(-1, 3).astype(np.float32)
    return v, np.arange(3 * n, dtype=np.uint32).reshape(n, 3)


@pytest.mark.parametrize("seed", range(24))
def test_random_soups_and_options(port, seed):
    """Sizes around every class boundary of the builder (one warp-built subtree <= 128 < one-CTA node <= 2048 <
    level-synchronous), random leaf sizes / bin counts / depth limits, clustered and degenerate centroid distributions:
    the tree is structurally valid (exact boxes, leaf rule, pre-order, statistics), deterministic, and walking it in the
    reference's order on the device gives what the oracle finds walking the same arrays, bit for bit."""
    from nanort_b200 import api, scenes as S

    rng = np.random.default_rng(1000 + seed)
    sizes = [2, 5, 31, 33, 64, 127, 128, 129, 400, 1000, 2047, 2048, 2049, 3000, 5000, 9000]
    n = sizes[seed % len(sizes)] if seed < 16 else int(rng.integers(2, 12000))
    v, f = _random_soup(rng, n)
    okw = dict(min_leaf_primitives=int(rng.choice([1, 1, 2, 4, 4, 8, 13])), bin_size=int(rng.choice([2, 4, 8, 16, 64, 64, 128])),
               max_tree_depth=int(rng.choice([3, 8, 20, 256, 256])))
    opts = api.BVHBuildOptions(**okw)
    acc = api.BVHAccel()
    assert acc.Build(len(f), v, f, opts)
    nodes, idx = acc.GetNodes(), acc.GetIndices()
    st = check_tree_structure(nodes, idx, v, f, min_leaf=okw["min_leaf_primitives"], max_depth=okw["max_tree_depth"])
    got = acc.GetStatistics()
    for k in ("max_tree_depth", "num_leaf_nodes", "num_branch_nodes"):
        assert got[k] == st[k], (k, got, st, n, okw)
    acc2 = api.BVHAccel()
    acc2.Build(len(f), v, f, opts)
    assert np.array_equal(acc2.GetNodes().view(np.uint8), nodes.view(np.uint8)) and np.array_equal(acc2.GetIndices(), idx)
    rays = S.incoherent_rays(v.min(axis=0) - 1, v.max(axis=0) + 1, 3000, seed=seed)
    # aim half of them at triangles so that they hit something
    tgt = v.reshape(-1, 3, 3).mean(axis=1)[rng.integers(0, n, 1500)]
    d = tgt - rays["org"][:1500]
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-20)
    rays["dir"][:1500] = d.astype(np.float32)
    rays["max_t"][:1500] = 1e30
    o_h, o_m = port.traverse(nodes, idx, v, f, rays, threads=8)
    c_h, c_m = acc.Traverse(rays, flags=api.TRAVERSE_CONFORMANCE)
    assert np.array_equal(c_m, o_m)
    hit = o_m.astype(bool)
    assert np.array_equal(c_h[hit].view(np.uint32), o_h[hit].view(np.uint32))
    if st["max_tree_depth"] + 2 <= 512:
        g_h, g_m = acc.Traverse(rays, flags=api.TRAVERSE_FAST)
        assert_parity(compare_hits(port, v, f, rays, g_h, g_m, o_h, o_m))
