"""Wavefront path tracer (csrc/path.cu, csrc/wavefront.cuh:PathShadeEpilogue) against the reference path tracer's OWN
code: the unmodified examples/path_tracer/main.cc (oracle/_ref/libpt_ref.so behind oracle/pt_ref_shim.cc), i.e. the
reference's MeshLight::sampleDirect, directionCosTheta, revisedONB, fresnel_schlick, reflect, refract, PdfAtoW with the
example's rand() replaced by the device's counter hash.  What it computed is recorded in tests/golden/path_ref_<scene>.npz
(tests/golden/make_reference_golden.py) for a fixed, seeded sample of the camera paths, followed through every bounce.

The check is per BOUNCE on identical inputs (no chaos amplification): the device traces and shades the sampled paths'
rays of bounce b through nrt_path_bounce_device -- the unit nrt_render_path_device repeats --, and every output is
compared with the reference's shading of the same rays: which rays continue, the continuation ray, the path throughput,
the shadow ray and its light contribution, the emitted radiance.  Decisions (lobe choice, Russian roulette, light
visibility set-up) must agree exactly; values agree to 1e-5 (sinf / cosf / sqrtf of CUDA and of glibc differ in the last
bit).  The reference's continuation rays are the next bounce's input."""
import os

import numpy as np
import pytest

from helpers import GOLDEN

pytestmark = pytest.mark.gpu

TILE = (64, 8)


def _rel(a, b, floor=1e-3):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor))) if a.size else 0.0


def _setup(torch, api, S, v, f, mats, ids, emissive, fvn, W, H, spp, bounces, seed, camera="cornell"):
    acc = api.BVHAccel()
    acc.Build(len(f), v, f)
    keep = {"m": torch.as_tensor(np.ascontiguousarray(mats).view(np.float32).reshape(-1), device="cuda"),
            "i": torch.as_tensor(ids.astype(np.int32), device="cuda"),
            "e": torch.as_tensor(emissive.astype(np.int32), device="cuda"),
            "n": torch.as_tensor(fvn.reshape(-1), device="cuda") if fvn is not None else None}
    p = api.PathParams()
    cam = S.scene_camera(camera, W, H)
    for i in range(12):
        p.cam[i] = float(cam[i])
    p.width, p.height, p.spp, p.sample0, p.seed = W, H, spp, 0, seed
    p.tile_w, p.tile_h, p.shard, p.n_shards = TILE[0], TILE[1], 0, 1
    p.max_bounces, p.ray_min_t, p.ray_max_t = bounces, 1e-3, 1e30
    p.n_materials, p.n_emissive = len(mats), len(emissive)
    p.d_materials, p.d_material_ids, p.d_emissive_faces = keep["m"].data_ptr(), keep["i"].data_ptr(), keep["e"].data_ptr()
    p.d_facevarying_normals, p.flags = (keep["n"].data_ptr() if fvn is not None else None), 0
    return acc, p, cam, keep


def scene_setup(scene):
    from nanort_b200 import scenes as S

    if scene == "cornell":
        v, f, mats, ids, emissive = S.cornell_with_materials()
        W, H, spp, bounces, seed = 64, 48, 4, 8, 5
    else:  # BASELINE.json configs[2]: the 1,002,528-triangle terrain under an area light, as bench.py sets it up
        v, f = S.make_scene("terrain")
        v, f, l0, ln = S.with_area_light(v, f, (0.0, 6.0, 0.0), 2.0, 2.0)
        mats = np.concatenate([S.material(diffuse=(0.7, 0.7, 0.7)), S.material(emission=(20, 20, 20))])
        ids = np.zeros(len(f), np.uint32)
        ids[l0:] = 1
        emissive = np.arange(l0, l0 + ln, dtype=np.uint32)
        W, H, spp, bounces, seed = 192, 108, 2, 6, 3
    return v, f, mats, ids, emissive, W, H, spp, bounces, seed


def camera_paths(scene, W, H, spp, seed):
    """Bounce 0 input: the camera ray of every slot (slot = path id); ray index = pixel * spp + sample."""
    from nanort_b200 import dist as nd, scenes as S

    pix_of_slot, smp_of_slot = nd.slot_pixels(W, H, TILE[0], TILE[1], 0, 1, spp)
    valid = np.nonzero(pix_of_slot >= 0)[0]
    order = np.argsort(pix_of_slot[valid] * spp + smp_of_slot[valid], kind="stable")
    rays0 = S.primary_rays(S.scene_camera(scene, W, H), W, H, spp=spp, seed=seed)
    pid = valid[order].astype(np.uint32)
    assert len(rays0) == len(pid)
    return pix_of_slot, smp_of_slot, pid, rays0


def draws(pix, smp, bounce, seed):
    """The six random numbers the device draws for a path at a bounce (dimension 8 + 8 * bounce onwards)."""
    from nanort_b200 import scenes as S

    dim = 8 + 8 * bounce
    return np.stack([S.rand_ps(pix, smp, dim + k, seed) for k in range(6)], axis=1).astype(np.float32)


def _bounce_by_bounce(with_normals, scene="cornell"):
    import torch
    from nanort_b200 import api, scenes as S

    g = np.load(os.path.join(GOLDEN, f"path_ref_{scene}.npz"))
    v, f, mats, ids, emissive, W, H, spp, bounces, seed = scene_setup(scene)
    # face normals as the example's loader makes them (calcNormal), recorded with the reference's results
    fvn = g["fvn"] if with_normals else None
    acc, p, cam, keep = _setup(torch, api, S, v, f, mats, ids, emissive, fvn, W, H, spp, bounces, seed, camera=scene)
    pix_of_slot, smp_of_slot, pid0, rays0 = camera_paths(scene, W, H, spp, seed)
    n_slots = len(pix_of_slot)
    k = g["sample"]
    org, dirs, w = rays0["org"][k].astype(np.float32), rays0["dir"][k].astype(np.float32), np.ones((len(k), 4), np.float32)
    dev = "cuda"

    def f4(xyz, w):
        return torch.as_tensor(np.concatenate([xyz, np.full((len(xyz), 1), w, np.float32)], axis=1).astype(np.float32), device=dev)

    d_weight = torch.ones((n_slots, 4), dtype=torch.float32, device=dev)
    accum = torch.zeros(W * H * 3, dtype=torch.float32, device=dev)
    tied = np.zeros(0, np.uint32)  # paths whose ray hit two primitives at exactly the same t: the pick may differ
    total_checked = total_recorded = emitted = 0
    checked_per_bounce = [0] * bounces
    lobes_seen = set()
    for b in range(bounces):
        if f"b{b}_pid" not in g:
            break
        gp, gmask = g[f"b{b}_pid"], g[f"b{b}_mask"]
        assert (b > 0 or np.array_equal(gp, pid0[k])) and len(gp) == len(org)
        gh = np.nonzero(gmask)[0]
        total_recorded += len(gh)
        want_all = {name: g[f"b{b}_{name}"] for name in ("flags", "next_org", "next_dir", "weight", "shadow_org",
                                                         "shadow_dir", "shadow_max_t", "shadow_contrib", "emission")}
        # the hit records of these rays, from the same traversal kernel: the reference's hits, ties aside
        r = np.zeros(len(gp), S.RAY_DTYPE)
        r["org"], r["dir"], r["min_t"], r["max_t"] = org, dirs, np.float32(1e-3), np.float32(1e30)
        hits, mask = acc.Traverse(r)
        assert np.array_equal(mask, gmask), b
        other = gp[gh][hits["prim_id"][gh] != g[f"b{b}_prim"]]
        assert np.array_equal(hits["t"][gh], g[f"b{b}_t"]), b  # a different primitive only at exactly the same t
        tied = np.union1d(tied, other)
        fed = ~np.isin(gp, tied)
        slot_h = np.cumsum(gmask.astype(np.int64)) - 1  # index of a hit ray among the recorded hits
        sel = np.nonzero(fed)[0]
        h_rec = slot_h[sel][gmask[sel] == 1]  # the recorded hits of the fed rays
        want = {name: a[h_rec] for name, a in want_all.items()}
        pid = gp[sel]
        n = len(pid)
        if n:
            d_o, d_d = f4(org[sel], 1e-3), f4(dirs[sel], 1e30)
            d_pid = torch.as_tensor(pid.astype(np.int32), device=dev)
            d_weight[torch.as_tensor(pid.astype(np.int64), device=dev)] = torch.as_tensor(w[sel], device=dev)
            out_o = torch.zeros((n, 4), dtype=torch.float32, device=dev)
            out_d = torch.zeros((n, 4), dtype=torch.float32, device=dev)
            out_pid = torch.zeros(n, dtype=torch.int32, device=dev)
            sh_o = torch.zeros((n, 4), dtype=torch.float32, device=dev)
            sh_d = torch.zeros((n, 4), dtype=torch.float32, device=dev)
            sh_c = torch.zeros((n, 4), dtype=torch.float32, device=dev)
            accum.zero_()
            n_cont, n_sh = acc.PathBounce(p, b, n, d_o.data_ptr(), d_d.data_ptr(), d_pid.data_ptr(), d_weight.data_ptr(),
                                          out_o.data_ptr(), out_d.data_ptr(), out_pid.data_ptr(), sh_o.data_ptr(),
                                          sh_d.data_ptr(), sh_c.data_ptr(), accum.data_ptr())
            h = np.nonzero(gmask[sel])[0]
            pix = pix_of_slot[pid]
            total_checked += len(h)
            checked_per_bounce[b] = len(h)
            cont = (want["flags"] & 1) != 0
            shad = (want["flags"] & 2) != 0
            emit = (want["flags"] & 4) != 0
            # ---- decisions: which paths continue / sample the light
            assert n_cont == int(cont.sum()) and n_sh == int(shad.sum()), (b, n_cont, int(cont.sum()), n_sh, int(shad.sum()))
            got_pid = out_pid.cpu().numpy()[:n_cont].astype(np.uint32)
            ref_pid = pid[h][cont]
            assert np.array_equal(np.sort(got_pid), np.sort(ref_pid)), f"bounce {b}: different set of continuing paths"
            # ---- continuation rays and throughput, matched by path id
            go, gd = out_o.cpu().numpy()[:n_cont], out_d.cpu().numpy()[:n_cont]
            gsort, rsort = np.argsort(got_pid), np.argsort(ref_pid)
            assert _rel(go[gsort][:, :3], want["next_org"][cont][rsort]) <= 1e-5
            assert float(np.max(np.abs(gd[gsort][:, :3] - want["next_dir"][cont][rsort]))) <= 2e-5 if n_cont else True
            w_out = d_weight.cpu().numpy()
            assert _rel(w_out[ref_pid][:, :3], want["weight"][cont][:, :3], floor=1e-6) <= 1e-5
            assert np.array_equal(w_out[ref_pid][:, 3] != 0, want["weight"][cont][:, 3] != 0), "do_emission flag"
            # ---- shadow rays: matched by (pixel, origin): sort both by the contribution's pixel and the ray origin bits
            gs_o, gs_d, gs_c = sh_o.cpu().numpy()[:n_sh], sh_d.cpu().numpy()[:n_sh], sh_c.cpu().numpy()[:n_sh]
            got_pix = gs_c[:, 3].copy().view(np.uint32)
            ref_pix = pix[h][shad].astype(np.uint32)
            kg = np.lexsort((gs_o[:, 2], gs_o[:, 1], gs_o[:, 0], got_pix))
            ro = want["shadow_org"][shad]
            kr = np.lexsort((ro[:, 2], ro[:, 1], ro[:, 0], ref_pix))
            assert np.array_equal(got_pix[kg], ref_pix[kr])
            assert _rel(gs_o[kg][:, :3], ro[kr]) <= 1e-5
            assert float(np.max(np.abs(gs_d[kg][:, :3] - want["shadow_dir"][shad][kr]))) <= 2e-5 if n_sh else True
            assert _rel(gs_d[kg][:, 3], want["shadow_max_t"][shad][kr]) <= 1e-5
            # the contribution holds both cosines of the light sample: directions that agree to 2e-5 (sinf / cosf of CUDA
            # vs glibc, asserted above) give cosines that agree to 2e-5 ABSOLUTE, i.e. to 2e-5 / cos relative -- grazing
            # samples (cos ~ 0.05) legitimately differ by a few 1e-4; all but a per-mille of the samples sit within 2e-5
            cd = np.abs(gs_c[kg][:, :3] - want["shadow_contrib"][shad][kr]) / np.maximum(np.abs(want["shadow_contrib"][shad][kr]), 1e-6)
            assert (float(cd.max()) <= 1e-3 and float(np.quantile(cd, 0.999)) <= 2e-5) if n_sh else True
            # ---- what reached the frame: emission of this bounce + the light samples the device's shadow pass found visible
            sr = np.zeros(n_sh, S.RAY_DTYPE)
            sr["org"], sr["dir"], sr["min_t"], sr["max_t"] = gs_o[:, :3], gs_d[:, :3], gs_o[:, 3], gs_d[:, 3]
            _, smask = acc.Traverse(sr) if n_sh else (None, np.zeros(0, np.uint8))
            expect_accum = np.zeros((W * H, 3), np.float64)
            np.add.at(expect_accum, pix[h][emit], want["emission"][emit].astype(np.float64))
            vis = smask == 0
            np.add.at(expect_accum, got_pix[vis].astype(np.int64), gs_c[vis][:, :3].astype(np.float64))
            got_accum = accum.cpu().numpy().reshape(-1, 3).astype(np.float64)
            assert np.max(np.abs(got_accum - expect_accum) / np.maximum(np.abs(expect_accum), 1.0)) <= 1e-4, b
            lobes_seen |= {("cont", bool(cont.any())), ("shadow", bool(shad.any())), ("emit", bool(emit.any()))}
            emitted += int(emit.sum())
        # next bounce: the reference's continuation rays of every recorded path
        cont_all = (want_all["flags"] & 1) != 0
        org, dirs, w = want_all["next_org"][cont_all], want_all["next_dir"][cont_all], want_all["weight"][cont_all]
    assert total_checked >= 0.95 * total_recorded and total_recorded > (1300 if scene == "cornell" else 850)
    # the recorded sample reaches every bounce of the Cornell box and the first five of the terrain (no path of the
    # terrain's camera gets further); each of them is checked
    assert all(n > 0 for n in checked_per_bounce[: bounces if scene == "cornell" else 5]), checked_per_bounce
    assert ("shadow", True) in lobes_seen
    assert scene != "cornell" or emitted >= 80, emitted  # the terrain's light is outside the camera's view
    return total_checked


def test_every_bounce_matches_the_reference_functions_with_facevarying_normals():
    _bounce_by_bounce(with_normals=True)


def test_every_bounce_matches_the_reference_functions_with_loader_style_flat_normals():
    """No normals handed to the device: it must fall back to the flat normal the example's loader would have stored
    (calcNormal: cross(v2 - v0, v1 - v0), main.cc:306-312, 566-601) -- orientation included, it decides `inside`,
    refraction and which side of an emitter shines."""
    _bounce_by_bounce(with_normals=False)


def test_every_bounce_matches_the_reference_functions_on_the_1m_triangle_terrain():
    """BASELINE.json configs[2]'s scene (terrain + area light, diffuse): the same per-bounce comparison with the reference's
    own shading code, at 2 spp on 192x108 pixels."""
    _bounce_by_bounce(with_normals=False, scene="terrain")


def test_whole_pass_equals_the_sum_of_its_bounces():
    """nrt_render_path_device (camera generation + the bounce loop on the device) against the same pass driven bounce by
    bounce from the host through nrt_path_bounce_device: identical ray counts, same image up to atomic-add order."""
    import torch
    from nanort_b200 import api, dist as nd, scenes as S

    v, f, mats, ids, emissive = S.cornell_with_materials()
    W, H, spp, bounces, seed = 64, 48, 6, 7, 5
    acc, p, cam, keep = _setup(torch, api, S, v, f, mats, ids, emissive, None, W, H, spp, bounces, seed)
    accum = torch.zeros(W * H * 3, dtype=torch.float32, device="cuda")
    r = acc.RenderPath(p, accum.data_ptr())
    whole = accum.cpu().numpy().astype(np.float64)
    assert r.camera_rays == W * H * spp and r.traverse_launches == 2 * bounces and r.launches == 1 + 4 * bounces

    pix_of_slot, smp_of_slot = nd.slot_pixels(W, H, TILE[0], TILE[1], 0, 1, spp)
    valid = np.nonzero(pix_of_slot >= 0)[0]
    order = np.argsort(pix_of_slot[valid] * spp + smp_of_slot[valid], kind="stable")
    rays0 = S.primary_rays(cam, W, H, spp=spp, seed=seed)
    pid = valid[order].astype(np.int32)
    n = len(pid)
    mk = lambda xyz, w: torch.as_tensor(np.concatenate([xyz, np.full((len(xyz), 1), w, np.float32)], axis=1).astype(np.float32), device="cuda")
    q = [[mk(rays0["org"], 1e-3), mk(rays0["dir"], 1e30), torch.as_tensor(pid, device="cuda")],
         [torch.zeros((n, 4), device="cuda"), torch.zeros((n, 4), device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")]]
    sh = [torch.zeros((n, 4), device="cuda") for _ in range(3)]
    weight = torch.ones((len(pix_of_slot), 4), dtype=torch.float32, device="cuda")
    accum2 = torch.zeros(W * H * 3, dtype=torch.float32, device="cuda")
    radiance, shadow, cur = 0, 0, 0
    for b in range(bounces):
        if n == 0:
            break
        radiance += n
        nc, ns = acc.PathBounce(p, b, n, q[cur][0].data_ptr(), q[cur][1].data_ptr(), q[cur][2].data_ptr(), weight.data_ptr(),
                                q[cur ^ 1][0].data_ptr(), q[cur ^ 1][1].data_ptr(), q[cur ^ 1][2].data_ptr(),
                                sh[0].data_ptr(), sh[1].data_ptr(), sh[2].data_ptr(), accum2.data_ptr())
        shadow += ns
        n, cur = nc, cur ^ 1
    # Identical up to exact-distance ties: where two primitives are hit at the same t (Cornell: shared edges, box bottoms
    # lying in the floor) the fast kernel reports whichever its warp visited last, like the reference (SURVEY.md F3), and
    # the warp's composition depends on the order the queue was compacted in -- such a path may pick the other material.
    assert abs(radiance - r.radiance_rays) <= 4 and abs(shadow - r.shadow_rays) <= 4, (radiance, shadow, r.radiance_rays, r.shadow_rays)
    parts = accum2.cpu().numpy().astype(np.float64).reshape(-1, 3)
    rel = np.max(np.abs(parts - whole.reshape(-1, 3)) / np.maximum(np.abs(whole.reshape(-1, 3)), 1.0), axis=1)
    assert np.count_nonzero(rel > 1e-5) <= 4, np.count_nonzero(rel > 1e-5)


def test_path_tracer_diffuse_only_energy_is_bounded():
    """White furnace-ish sanity: a closed diffuse box with albedo a and an emitter can never return more than
    Le * cos per camera ray; no NaNs; more bounces never darken the image."""
    import torch
    from nanort_b200 import api, scenes as S

    v, f = S.make_scene("cornell")
    v, f, l0, ln = S.with_area_light(v, f, (0.0, 9.99, 0.0), 2.0, 2.0)
    mats = np.concatenate([S.material(diffuse=(0.7, 0.7, 0.7)), S.material(emission=(10, 10, 10))])
    ids = np.zeros(len(f), np.uint32)
    ids[l0:] = 1
    emissive = np.arange(l0, l0 + ln, dtype=np.uint32)
    imgs = []
    for bounces in (1, 2, 6):
        acc, p, cam, keep = _setup(torch, api, S, v, f, mats, ids, emissive, None, 64, 48, 8, bounces, 9)
        accum = torch.zeros(64 * 48 * 3, dtype=torch.float32, device="cuda")
        acc.RenderPath(p, accum.data_ptr())
        got = accum.cpu().numpy().astype(np.float64)
        assert np.isfinite(got).all() and got.min() >= 0
        imgs.append(got.mean())
    assert imgs[0] <= imgs[1] + 1e-6 <= imgs[2] + 2e-6


def test_any_hit_shadow_rays_give_the_same_image():
    """NRT_TRAVERSE_ANY_HIT in nrt_path_params.flags: the shadow launches stop at the first occluder
    (examples/path_tracer/main.cc:675-701 only looks at Traverse's bool) -- same ray counts, same image up to the order of
    the float atomics."""
    import torch
    from nanort_b200 import api, scenes as S

    v, f, mats, ids, emissive = S.cornell_with_materials()
    W, H, spp, bounces, seed = 64, 48, 6, 7, 5
    imgs, counts = [], []
    for flags in (0, api.TRAVERSE_ANY_HIT):
        acc, p, cam, keep = _setup(torch, api, S, v, f, mats, ids, emissive, None, W, H, spp, bounces, seed)
        p.flags = flags
        accum = torch.zeros(W * H * 3, dtype=torch.float32, device="cuda")
        r = acc.RenderPath(p, accum.data_ptr())
        imgs.append(accum.cpu().numpy().astype(np.float64).reshape(-1, 3))
        counts.append((r.camera_rays, r.radiance_rays, r.shadow_rays))
    # same allowance as test_whole_pass_equals_the_sum_of_its_bounces: a radiance ray that hits two primitives at exactly
    # the same t may pick either, run to run (queue compaction order)
    assert counts[0][0] == counts[1][0] and counts[0][2] > 0
    assert abs(counts[0][1] - counts[1][1]) <= 4 and abs(counts[0][2] - counts[1][2]) <= 4, counts
    rel = np.max(np.abs(imgs[0] - imgs[1]) / np.maximum(np.abs(imgs[0]), 1.0), axis=1)
    assert np.count_nonzero(rel > 1e-5) <= 4, np.count_nonzero(rel > 1e-5)
