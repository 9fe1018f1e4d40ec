"""The two-level scene restatement (oracle/nanort_oracle.c, "two-level scene" section) against the unmodified
reference scene graph (examples/nanosg/nanosg.h via oracle/ref_sg_shim.cc): per-instance matrices and boxes,
the top-level tree, the sorted node-hit list and Scene::Traverse's records, all bit for bit.  The reference's results
are recorded as fingerprints in tests/golden/reference_digests.json (tests/golden/make_reference_golden.py)."""
import numpy as np
import pytest

from helpers import REF_DIFF, digest, hits_digest, list_digest, reference_golden, tree_digest
from nanort_b200 import scenes as S
from oracle import orc

LIST_RAYS = list(range(0, 300)) + list(range(5000, 5100))


def _scene_rays(insts, n, seed):
    lo = np.min([np.min(v @ x[:3, :3] + x[3, :3], axis=0) for v, f, x in insts], axis=0)
    hi = np.max([np.max(v @ x[:3, :3] + x[3, :3], axis=0) for v, f, x in insts], axis=0)
    pad = 0.25 * (hi - lo) + 0.5
    rays = S.incoherent_rays(lo - pad, hi + pad, n, seed=seed)
    rays["min_t"] = 0.0
    return rays


def scene_case_rays(kind, insts):
    rays = _scene_rays(insts, 20000, seed=5)
    if kind == "row":  # rays down the row: > 64 boxes pierced, exact entry ties at the duplicates
        k = np.arange(2000)
        rays["org"][:2000] = np.stack([-3.0 - 0.01 * (k % 7), 0.3 * S.rand01(k, 0, 9) - 0.15,
                                       0.3 * S.rand01(k, 1, 9) - 0.15], axis=1)
        d = np.stack([np.ones(2000), 0.002 * (S.rand01(k, 2, 9) - 0.5), 0.002 * (S.rand01(k, 3, 9) - 0.5)], axis=1)
        rays["dir"][:2000] = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
        rays["dir"][:50, 1:] = 0.0
        rays["dir"][:50, 0] = 1.0
        rays["max_t"][:2000] = 1e30
    return rays


def blas_checked(insts):
    return (0, 1, 2, len(insts) - 1)


def short_max_t_rays(insts):
    rays = _scene_rays(insts, 4000, seed=8)
    rays["max_t"] = 0.75  # far smaller than most hit distances
    return rays


def hostile_scene_rays():
    from edge_cases import hostile_rays

    rays = hostile_rays(np.float32([-8, -4, -8]), np.float32([8, 4, 8]), n=8000, seed=5)
    rays["min_t"] = np.where(np.isnan(rays["min_t"]), rays["min_t"], 0.0)
    return rays


@pytest.mark.parametrize("cpp11", [True, False])
@pytest.mark.parametrize("kind", ["mixed", "row"])
def test_port_scene_matches_reference(kind, cpp11):
    want = reference_golden()[f"scene/{kind}/{cpp11}"]
    insts = S.instances_mixed() if kind == "mixed" else S.instances_row()
    port = orc.PortScene(insts, cpp11)
    # Node::Update: matrices, local and world boxes
    assert digest(port.sg) == want["node_states"], REF_DIFF
    # top-level tree + every bottom-level tree
    assert tree_digest(port.top, port.top_idx) == want["top"], REF_DIFF
    assert [tree_digest(*port.blas[i][:2]) for i in blas_checked(insts)] == want["blas"], REF_DIFF
    rays = scene_case_rays(kind, insts)
    # first stage: the node-hit list in its exact order
    lists = [port.list_node_intersections(rays[r]) for r in LIST_RAYS]
    assert list_digest(lists) == want["lists"], REF_DIFF
    if kind == "row":
        assert any(len(ids) == 64 for _, _, ids in lists)
    # Scene::Traverse
    ph, pm = port.traverse(rays, threads=4)
    assert pm.sum() > 500
    assert hits_digest(ph, pm) == want["hits"], REF_DIFF


def test_cull_back_face_flag_is_inert_and_local_ray_is_unbounded():
    """S2 / S4 of the restatement header: the world ray's min_t/max_t gate only the top-level walk."""
    insts = S.instances_mixed(6)
    port = orc.PortScene(insts)
    ph, pm = port.traverse(short_max_t_rays(insts))
    assert hits_digest(ph, pm) == reference_golden()["scene_short_max_t"], REF_DIFF
    assert (ph["t"][pm == 1] > 0.75).any()  # hits beyond the world max_t are still reported


def test_port_scene_matches_reference_on_hostile_rays():
    """Non-finite, zero-length and far-from-unit directions through Scene::Traverse: raw bits must match."""
    insts = S.instances_mixed(12)
    port = orc.PortScene(insts)
    ph, pm = port.traverse(hostile_scene_rays(), threads=4)
    assert hits_digest(ph, pm) == reference_golden()["scene_hostile"], REF_DIFF
    assert pm.sum() > 300
