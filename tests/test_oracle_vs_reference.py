"""CPU: the oracle port against the unmodified reference -- bit-for-bit, both build modes.  The reference's results are
recorded as fingerprints in tests/golden/reference_digests.json (tests/golden/make_reference_golden.py)."""
import numpy as np
import pytest

from helpers import REF_DIFF, hits_digest, reference_golden, tree_digest

SCENES = [("cornell", {}), ("sphere_grid", dict(nx=3, nz=3)), ("terrain", dict(n=80))]
BUILD_VARIANTS = (dict(min_leaf_primitives=1), dict(bin_size=8), dict(max_tree_depth=6), dict(min_leaf_primitives=16))
TRACE_VARIANTS = (dict(cull_back_face=1), dict(skip_prim_id=17), dict(prim_ids_range=(1000, 3000)))


def scene_rays(name, v):
    from nanort_b200 import scenes as S

    cam = S.scene_camera(name, 128, 96)
    return np.concatenate([S.primary_rays(cam, 128, 96, spp=1, seed=5),
                           S.incoherent_rays(v.min(axis=0), v.max(axis=0), 30000, seed=6)])


@pytest.mark.parametrize("name,kw", SCENES)
@pytest.mark.parametrize("cpp11", [True, False])
def test_port_equals_reference(port, name, kw, cpp11):
    from oracle import orc
    from nanort_b200 import scenes as S

    g = reference_golden()
    assert g["ref_sizes"] == [40, 36, 16, 28, 16]
    assert [d.itemsize for d in (orc.NODE_DTYPE, orc.RAY_DTYPE, orc.HIT_DTYPE, orc.BUILD_OPT_DTYPE,
                                 orc.TRACE_OPT_DTYPE)] == g["ref_sizes"]
    want = g[f"vs_ref/{name}/{cpp11}"]
    v, f = S.make_scene(name, **kw)
    pn, pi, ps = port.build(v, f, mode=orc.MODE_CPP11 if cpp11 else 0)
    assert tree_digest(pn, pi) == want["tree"], REF_DIFF
    assert list(ps.values()) == want["stats"]
    rays = scene_rays(name, v)
    ph, pm, ctr = port.traverse(pn, pi, v, f, rays, cpp11=cpp11, threads=4, counters=True)
    assert hits_digest(ph, pm) == want["hits"], REF_DIFF
    assert ctr["nodes_popped"] >= len(rays)


def test_reference_option_variants(port):
    """Non-default build / trace options go through the same code paths in port and reference."""
    from oracle import orc
    from nanort_b200 import scenes as S

    g = reference_golden()
    v, f = S.make_scene("sphere_grid", nx=2, nz=2)
    rays = S.incoherent_rays(v.min(axis=0), v.max(axis=0), 20000, seed=8)
    for okw in BUILD_VARIANTS:
        pn, pi, ps = port.build(v, f, orc.build_options(**okw))
        want = g[f"vs_ref_options/{sorted(okw.items())}"]
        assert tree_digest(pn, pi) == want["tree"], (okw, REF_DIFF)
        assert list(ps.values()) == want["stats"], okw
    pn, pi, _ = port.build(v, f)
    for tkw in TRACE_VARIANTS:
        ph, pm = port.traverse(pn, pi, v, f, rays, topts=orc.trace_options(**tkw))
        assert hits_digest(ph, pm) == g[f"vs_ref_options/{sorted(tkw.items())}"], (tkw, REF_DIFF)


@pytest.mark.parametrize("cpp11", [True, False])
def test_port_equals_reference_on_hostile_rays_and_degenerate_triangles(port, cpp11):
    """Non-finite / zero / denormal ray components, inverted ranges, zero-area triangles: the restatement must
    follow the reference through every IEEE corner (raw bits, NaN payloads included)."""
    from oracle import orc
    from edge_cases import degenerate_mesh, hostile_rays

    want = reference_golden()[f"vs_ref_hostile/{cpp11}"]
    v, f = degenerate_mesh()
    nodes, idx, _ = port.build(v, f, None, orc.MODE_CPP11 if cpp11 else 0)
    assert tree_digest(nodes, idx) == want["tree"], REF_DIFF
    rays = hostile_rays(v[:34 * 3].min(axis=0) - 1, v[:34 * 3].max(axis=0) + 1)
    ph, pm = port.traverse(nodes, idx, v, f, rays, cpp11=cpp11)
    assert hits_digest(ph, pm) == want["hits"], REF_DIFF
