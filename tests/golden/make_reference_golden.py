"""Records what the unmodified reference computes for the tests that compare with it, so that they run without it:

    tests/golden/reference_digests.json   SHA-256 fingerprints (tests/helpers.py:digest) of bit-exact results: trees,
                                          hit records, node-hit lists of the reference's BVHAccel<float / double> and
                                          of its two-level scene (examples/nanosg), plus a few small exact values
    tests/golden/spheres_ref.npz          the particle_primitive example's hits where a tolerance applies (u / v):
                                          a fixed, seeded sample of the rays
    tests/golden/path_ref_<scene>.npz     the path_tracer example's shading, bounce by bounce, for a fixed, seeded
                                          sample of camera paths followed through every bounce

Needs oracle/_ref (oracle/Makefile builds it from a checkout of the reference); run from the repository root:

    python tests/golden/make_reference_golden.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]
from oracle import orc  # noqa: E402
from nanort_b200 import scenes as S  # noqa: E402
from edge_cases import degenerate_mesh, hostile_rays  # noqa: E402
from helpers import digest, hits_digest, list_digest, tree_digest  # noqa: E402
import test_gpu_f64 as tf64  # noqa: E402
import test_gpu_path as tpath  # noqa: E402
import test_gpu_prims as tprims  # noqa: E402
import test_oracle_f64 as tof64  # noqa: E402
import test_oracle_scene as tscene  # noqa: E402
import test_oracle_vs_reference as tvs  # noqa: E402


def key(*parts):
    return "/".join(str(p) for p in parts)


def oracle_vs_reference(D):
    D["ref_sizes"] = orc.Reference(True).sizes()
    for name, kw in tvs.SCENES:
        for cpp11 in (True, False):
            v, f = S.make_scene(name, **kw)
            ra = orc.Reference(cpp11).build(v, f)
            rh, rm = ra.traverse(tvs.scene_rays(name, v), threads=4)
            D[key("vs_ref", name, cpp11)] = {"tree": tree_digest(ra.nodes(), ra.indices()),
                                             "stats": list(ra.stats().values()), "hits": hits_digest(rh, rm)}
    ref = orc.Reference(True)
    v, f = S.make_scene("sphere_grid", nx=2, nz=2)
    rays = S.incoherent_rays(v.min(axis=0), v.max(axis=0), 20000, seed=8)
    for okw in tvs.BUILD_VARIANTS:
        ra = ref.build(v, f, orc.build_options(**okw))
        D[key("vs_ref_options", sorted(okw.items()))] = {"tree": tree_digest(ra.nodes(), ra.indices()),
                                                         "stats": list(ra.stats().values())}
    ra = ref.build(v, f)
    for tkw in tvs.TRACE_VARIANTS:
        D[key("vs_ref_options", sorted(tkw.items()))] = hits_digest(*ra.traverse(rays, topts=orc.trace_options(**tkw)))
    for cpp11 in (True, False):
        v, f = degenerate_mesh()
        acc = orc.Reference(cpp11).build(v, f)
        rays = hostile_rays(v[:34 * 3].min(axis=0) - 1, v[:34 * 3].max(axis=0) + 1)
        D[key("vs_ref_hostile", cpp11)] = {"tree": tree_digest(acc.nodes(), acc.indices()),
                                           "hits": hits_digest(*acc.traverse(rays))}


def oracle_f64(D):
    D["ref64_sizes"] = orc.ReferenceF64(True).sizes()
    for name, kw in tof64.SCENES:
        for cpp11 in (True, False):
            v64, f = tof64._scene64(name, kw, seed=2)
            racc = orc.ReferenceF64(cpp11).build(v64, f)
            d = {"tree": tree_digest(racc.nodes(), racc.indices())}
            for hostile in (False, True):
                rays = tof64._rays64(v64, 12000, seed=6, hostile=hostile)
                d[key("hits", hostile)] = hits_digest(*racc.traverse(rays, threads=4))
            D[key("f64_vs_ref", name, cpp11)] = d
    ref = orc.ReferenceF64(True)
    v64, f = tof64._scene64("sphere_grid", dict(nx=2, nz=2), seed=4)
    for okw in tof64.BUILD_VARIANTS:
        racc = ref.build(v64, f, orc.build_options_f64(**okw))
        D[key("f64_vs_ref_options", sorted(okw.items()))] = tree_digest(racc.nodes(), racc.indices())
    rays = tof64._rays64(v64, 6000, seed=8)
    for tkw in tof64.TRACE_VARIANTS:  # on the tree of the last build option set, as the test walks it
        D[key("f64_vs_ref_options", sorted(tkw.items()))] = hits_digest(*racc.traverse(rays,
                                                                                         topts=orc.trace_options(**tkw)))


def oracle_scene(D):
    for kind in ("mixed", "row"):
        for cpp11 in (True, False):
            insts = S.instances_mixed() if kind == "mixed" else S.instances_row()
            ref = orc.ReferenceScene(insts, cpp11)
            tn, ti = ref.top()
            rays = tscene.scene_case_rays(kind, insts)
            D[key("scene", kind, cpp11)] = {
                "node_states": digest(ref.node_states()), "top": tree_digest(tn, ti),
                "blas": [tree_digest(*ref.node_tree(i)) for i in tscene.blas_checked(insts)],
                "lists": list_digest([ref.list_node_intersections(rays[r]) for r in tscene.LIST_RAYS]),
                "hits": hits_digest(*ref.traverse(rays, threads=4))}
    insts = S.instances_mixed(6)
    D["scene_short_max_t"] = hits_digest(*orc.ReferenceScene(insts).traverse(tscene.short_max_t_rays(insts)))
    insts = S.instances_mixed(12)
    D["scene_hostile"] = hits_digest(*orc.ReferenceScene(insts).traverse(tscene.hostile_scene_rays(), threads=4))


def gpu_build(D):
    v, f = S.make_scene("sphere_grid", nx=3, nz=3)
    rays = S.primary_rays(S.scene_camera("sphere_grid", 200, 150), 200, 150, spp=1, seed=4)
    D["gpu_build_own_tree_hits"] = hits_digest(*orc.Reference(True).build(v, f).traverse(rays, threads=4))


def gpu_f64(D):
    for cpp11 in (True, False):
        ref = orc.ReferenceF64(cpp11)
        v64, f = tf64._scene64()
        D[key("gpu_f64_hits", cpp11)] = hits_digest(*ref.build(v64, f).traverse(tf64._rays64(v64, 60000, seed=4),
                                                                                 threads=8))
        v64, f = tf64._scene64(seed=9)
        racc = ref.build(v64, f)
        rh, rm = racc.traverse(tf64._rays64(v64, 40000, seed=10), threads=8)
        D[key("gpu_f64_adopted", cpp11)] = {"tree": tree_digest(racc.nodes(), racc.indices()), "hits": hits_digest(rh, rm),
                                            "bbox": [x.tolist() for x in racc.bounding_box()]}
        D[key("gpu_f64_conformance", cpp11)] = [tree_digest(a.nodes(), a.indices()) for a in
                                                (ref.build(v64, f, opts) for (v64, f), opts in tf64.conformance_cases())]


def gpu_prims(D):
    samples = {}
    rng = np.random.default_rng(2024)
    for n in tprims.SPHERE_COUNTS:
        centers, radii = tprims._spheres(n, seed=n)
        ref = orc.ReferenceSpheres(centers, radii)
        h, m = ref.traverse(tprims.sphere_case_rays(centers, n))
        hit = m == 1
        D[key("spheres", n)] = {"bbox": [x.tolist() for x in ref.bounding_box()], "mask": digest(m),
                                "t": digest(h["t"][hit])}
        idx = np.sort(rng.choice(np.nonzero(hit)[0], min(1536, int(hit.sum())), replace=False)).astype(np.uint32)
        samples.update({f"n{n}_ray": idx, f"n{n}_prim": h["prim_id"][idx], f"n{n}_u": h["u"][idx], f"n{n}_v": h["v"][idx]})
    np.savez_compressed(os.path.join(HERE, "spheres_ref.npz"), **samples)
    centers, radii = tprims._spheres(3000, seed=5)
    h, m = orc.ReferenceSpheres(centers, radii).traverse(tprims._rays(20000, seed=9), prim_range=(500, 1500))
    D["spheres_prim_range"] = {"mask": digest(m), "t": digest(h["t"][m == 1])}
    insts = S.instances_row(80)
    ref = orc.ReferenceScene(insts, cpp11=True)
    rays = tprims.list_case_rays(ref.node_states())
    tn, ti = ref.top()
    D["list_nodes"] = {"node_states": digest(ref.node_states()), "top": tree_digest(tn, ti)}
    for max_hits in tprims.MAX_HITS:
        D["list_nodes"][str(max_hits)] = list_digest([ref.list_node_intersections(r, max_hits) for r in rays])


def gpu_path(scene, n_paths, per_bounce=48, emitting=256):
    """Follows a seeded sample of the camera paths through every bounce of the reference's own shading, with the hits
    of the reference's own Traverse; the continuation rays of bounce b are the input of bounce b + 1.  Long paths and
    paths that reach an emitter are rare, so the sample is drawn by depth: (up to) `per_bounce` paths that hit something
    at each bounce, (up to) `emitting` paths with an emission event, the rest uniformly -- all in one seeded order."""
    v, f, mats, ids, emissive, W, H, spp, bounces, seed = tpath.scene_setup(scene)
    ref = orc.ReferencePathTracer(v, f, ids, mats)
    assert np.array_equal(ref.emissive_faces(), emissive)
    acc = orc.Reference(True).build(v, f)
    pix_of_slot, smp_of_slot, pid0, rays0 = tpath.camera_paths(scene, W, H, spp, seed)

    def follow(k):
        out = {}
        pid, org, dirs, w = pid0[k], rays0["org"][k], rays0["dir"][k], np.ones((len(k), 4), np.float32)
        for b in range(bounces):
            if len(pid) == 0:
                break
            r = np.zeros(len(pid), S.RAY_DTYPE)
            r["org"], r["dir"], r["min_t"], r["max_t"] = org, dirs, np.float32(1e-3), np.float32(1e30)
            hits, mask = acc.traverse(r)
            h = np.nonzero(mask)[0]
            draws = tpath.draws(pix_of_slot[pid], smp_of_slot[pid], b, seed)
            want = ref.shade(b, bounces, org[h], dirs[h], np.stack([hits["u"][h], hits["v"][h], hits["t"][h]], axis=1),
                             hits["prim_id"][h], w[h], draws[h])
            out.update({f"b{b}_pid": pid.astype(np.uint32), f"b{b}_mask": mask, f"b{b}_prim": hits["prim_id"][h],
                        f"b{b}_t": hits["t"][h]})
            out.update({f"b{b}_{name}": a for name, a in want.items()})
            cont = (want["flags"] & 1) != 0
            pid, org, dirs, w = pid[h][cont], want["next_org"][cont], want["next_dir"][cont], want["weight"][cont]
        return out

    every = follow(np.arange(len(pid0)))
    position = np.zeros(int(pid0.max()) + 1, np.int64)
    position[pid0] = np.arange(len(pid0))
    priority = np.argsort(np.random.default_rng(77).permutation(len(pid0)))
    chosen = np.zeros(len(pid0), bool)

    def take(cands, quota):
        cands = cands[np.argsort(priority[cands], kind="stable")]
        chosen[cands[~chosen[cands]][:max(0, quota - int(chosen[cands].sum()))]] = True

    for b in reversed(range(bounces)):
        if f"b{b}_pid" in every:
            take(position[every[f"b{b}_pid"][every[f"b{b}_mask"] == 1]], per_bounce)
    take(np.concatenate([position[every[f"b{b}_pid"][every[f"b{b}_mask"] == 1][(every[f"b{b}_flags"] & 4) != 0]]
                         for b in range(bounces) if f"b{b}_pid" in every]), emitting)
    take(np.arange(len(pid0)), n_paths)
    k = np.nonzero(chosen)[0]
    out = {"sample": k.astype(np.uint32), **follow(k)}
    if scene == "cornell":  # the face normals the example's loader makes (calcNormal), for the device's normal input
        out["fvn"] = ref.fvn
    np.savez_compressed(os.path.join(HERE, f"path_ref_{scene}.npz"), **out)


def main():
    D = {}
    for fn in (oracle_vs_reference, oracle_f64, oracle_scene, gpu_build, gpu_f64, gpu_prims):
        fn(D)
        print(fn.__name__, "done", flush=True)
    with open(os.path.join(HERE, "reference_digests.json"), "w") as f:
        json.dump(D, f, indent=1, sort_keys=True)
        f.write("\n")
    for scene, n_paths in (("cornell", 800), ("terrain", 1000)):
        gpu_path(scene, n_paths)
        print("path", scene, "done", flush=True)


if __name__ == "__main__":
    main()
