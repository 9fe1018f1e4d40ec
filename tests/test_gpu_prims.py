"""Non-triangle primitives (csrc/prims.cu): the device kinds of nanort's Prim / Pred / Intersector concept against the
reference's own models running on the unmodified nanort.h, through their results recorded in tests/golden
(tests/golden/make_reference_golden.py).

  * spheres: examples/particle_primitive/main.cc's SphereGeometry / SpherePred / SphereIntersector.  The trees differ
             (the reference builds its own), hits do not depend on the topology: hit flag identical and t bit-identical
             on every ray (fingerprints); prim_id identical and u / v within 1e-6 (atan2 / acos of two libms) on a
             seeded sample of the hits (spheres_ref.npz).
  * boxes:   BVHAccel::ListNodeIntersections with nanosg's NodeBBoxIntersector: the same nearest-first list of pierced
             boxes, bit for bit."""
import os

import numpy as np
import pytest

from helpers import GOLDEN, REF_DIFF, digest, list_digest, reference_golden, tree_digest

pytestmark = pytest.mark.gpu
SPHERE_COUNTS = [1, 7, 5000, 200000]
MAX_HITS = [64, 5, 1]


def _spheres(n, seed, rmax=0.35):
    rng = np.random.default_rng(seed)
    centers = rng.uniform(-6, 6, size=(n, 3)).astype(np.float32)
    radii = rng.uniform(0.02, rmax, size=n).astype(np.float32)
    return centers, radii


def _rays(n, seed, lo=-8.0, hi=8.0):
    from nanort_b200 import scenes as S

    r = S.incoherent_rays(np.float32([lo] * 3), np.float32([hi] * 3), n, seed=seed, axis_parallel_fraction=1.0 / 64)
    r["min_t"] = 0.0
    return r


def sphere_case_rays(centers, n_spheres):
    rays = _rays(60000, seed=3)
    # rays starting inside spheres and rays with a short range exercise the t0 < 0 and the `t > t_inout` branches
    rays["org"][:2000] = centers[np.arange(2000) % n_spheres] + np.float32(0.01)
    rays["max_t"][2000:6000] = np.float32(3.0)
    return rays


@pytest.mark.parametrize("n_spheres", SPHERE_COUNTS)
def test_spheres_match_the_reference_particle_primitive_model(n_spheres):
    from nanort_b200 import api

    want = reference_golden()[f"spheres/{n_spheres}"]
    sample = np.load(os.path.join(GOLDEN, "spheres_ref.npz"))
    centers, radii = _spheres(n_spheres, seed=n_spheres)
    acc = api.BVHAccel()
    assert acc.BuildSpheres(centers, radii)
    gb = acc.BoundingBox()
    assert gb[0].tolist() == want["bbox"][0] and gb[1].tolist() == want["bbox"][1]
    st = acc.GetStatistics()
    assert st["num_leaf_nodes"] == st["num_branch_nodes"] + 1
    rays = sphere_case_rays(centers, n_spheres)
    got_h, got_m = acc.Traverse(rays)
    assert digest(got_m) == want["mask"], REF_DIFF
    hit = got_m.astype(bool)
    assert hit.sum() > (100 if n_spheres > 100 else 0)
    assert digest(got_h["t"][hit]) == want["t"], ("t must be bit-identical", REF_DIFF)
    j = sample[f"n{n_spheres}_ray"]
    assert len(j) == min(1536, int(hit.sum()))
    same_prim = got_h["prim_id"][j] == sample[f"n{n_spheres}_prim"]
    # overlapping spheres can be hit at exactly the same distance: the reference keeps whichever it tested last (t is
    # bit-identical on every ray, so a different prim_id can only be such a tie)
    ok = j[same_prim]
    assert np.max(np.abs(got_h["u"][ok] - sample[f"n{n_spheres}_u"][same_prim]), initial=0.0) <= 1e-6
    assert np.max(np.abs(got_h["v"][ok] - sample[f"n{n_spheres}_v"][same_prim]), initial=0.0) <= 1e-6


def test_sphere_prim_id_range_filter():
    from nanort_b200 import api

    want = reference_golden()["spheres_prim_range"]
    centers, radii = _spheres(3000, seed=5)
    acc = api.BVHAccel()
    acc.BuildSpheres(centers, radii)
    rays = _rays(20000, seed=9)
    opt = api.BVHTraceOptions(prim_ids_range=(500, 1500))
    got_h, got_m = acc.Traverse(rays, options=opt)
    assert digest(got_m) == want["mask"], REF_DIFF
    hit = got_m.astype(bool)
    assert hit.any() and got_h["prim_id"][hit].min() >= 500 and got_h["prim_id"][hit].max() < 1500
    assert digest(got_h["t"][hit]) == want["t"], REF_DIFF


def test_sphere_build_of_nothing_fails_like_the_reference():
    from nanort_b200 import api

    acc = api.BVHAccel()
    assert acc.BuildSpheres(np.zeros((0, 3), np.float32), np.zeros(0, np.float32)) is False


def list_case_rays(node_states):
    from nanort_b200 import scenes as S

    boxes = np.concatenate([node_states["xbmin"], node_states["xbmax"]], axis=1).astype(np.float32)
    bmin, bmax = boxes[:, :3].min(axis=0), boxes[:, 3:].max(axis=0)
    rays = S.incoherent_rays(bmin - 1, bmax + 1, 3000, seed=4, axis_parallel_fraction=0.25)
    # rays down the row (both ways, slightly tilted, some starting inside it): these pierce tens of boxes, more than 64
    # for the long ones, and meet the coincident instances at exactly equal distances
    k = np.arange(240)
    down = np.zeros(len(k), S.RAY_DTYPE)
    fwd = (k % 2) == 0
    down["org"][:, 0] = np.where(fwd, -2.0 + 0.37 * (k % 60), 82.0 - 0.41 * (k % 50))
    down["org"][:, 1] = 0.3 * np.sin(k * 0.7)
    down["org"][:, 2] = 0.3 * np.cos(k * 1.3)
    d = np.stack([np.where(fwd, 1.0, -1.0), 0.004 * np.sin(k * 2.1), 0.004 * np.cos(k * 0.9)], axis=1)
    down["dir"] = (d / np.linalg.norm(d, axis=1)[:, None]).astype(np.float32)
    down["max_t"] = np.where(k % 3 == 0, 30.0, 1e30)
    rays = np.concatenate([rays, down])
    rays["min_t"] = 0.0
    return rays


@pytest.mark.parametrize("max_hits", MAX_HITS)
def test_list_node_intersections_matches_the_reference(max_hits):
    """The boxes are the world boxes of a reference nanosg scene's nodes.  BVHAccel::ListNodeIntersections is a property
    of the TREE, not only of the boxes: the leaf-level NodeBBoxIntersector has no [min_t, max_t] clamp (nanosg.h:597-634),
    so a box behind the origin is listed iff it shares a leaf with a box the range-clamped node test lets through.  The
    device list is therefore compared, bit for bit, with the reference algorithm walking the DEVICE's tree (the oracle's
    restatement, itself pinned to the unmodified nanosg.h on the reference's tree -- re-checked below), and with the
    reference's own list on every ray whose answer cannot depend on the leaves (all listed boxes start in front of
    min_t)."""
    from oracle import orc
    from nanort_b200 import api, scenes as S

    want = reference_golden()["list_nodes"]
    insts = S.instances_row(80)  # a row of overlapping instances: rays along the row pierce > 64 boxes
    ref = orc.PortScene(insts, cpp11=True)  # the restatement, pinned to the reference's scene by the fingerprints
    port = ref.port
    st, ref_nodes, ref_idx = ref.sg, ref.top, ref.top_idx
    assert digest(st) == want["node_states"] and tree_digest(ref_nodes, ref_idx) == want["top"], REF_DIFF
    boxes = np.concatenate([st["xbmin"], st["xbmax"]], axis=1).astype(np.float32)
    acc = api.BVHAccel()
    assert acc.BuildBoxes(boxes)
    dev_nodes, dev_idx = acc.GetNodes(), acc.GetIndices()
    rays = list_case_rays(st)
    # the reference's lists: the reference algorithm on the reference's tree, equal to the recorded ones
    ref_lists = [orc.list_node_intersections_on_tree(port, ref_nodes, ref_idx, st, r, max_hits) for r in rays]
    assert list_digest(ref_lists) == want[str(max_hits)], REF_DIFF
    hits, counts = acc.ListNodeIntersections(rays, max_intersections=max_hits)
    many = tree_independent = 0
    for i in range(len(rays)):
        r_tmin, r_tmax, r_ids = ref_lists[i]
        tmin, tmax, ids = orc.list_node_intersections_on_tree(port, dev_nodes, dev_idx, st, rays[i], max_hits)
        assert counts[i] == len(ids), (i, counts[i], len(ids))
        g = hits[i, : counts[i]]
        assert np.array_equal(g["t_min"].view(np.uint32), tmin.view(np.uint32)), i
        assert np.array_equal(g["node_id"], ids), i  # same tree, same heap: same order, ties included
        assert np.array_equal(g["t_max"].view(np.uint32), tmax.view(np.uint32)), i
        if len(r_ids) == len(ids) and len(ids) < max_hits and (len(ids) == 0 or (tmin.min() > 0.0 and r_tmin.min() > 0.0)):
            # nothing was dropped and nothing lies behind the origin: the set of boxes is the same in any tree
            assert sorted(ids) == sorted(r_ids), i
            tree_independent += 1
        many += int(counts[i] >= min(max_hits, 10))
    assert many > 20 and tree_independent > 100
