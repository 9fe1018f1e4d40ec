#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric: Mrays/s, primary + 1-bounce AO rays.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling strong|weak]
                    [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1]): procedural 100,002-triangle sphere grid, 1920x1080, 16 spp of jittered
pinhole primary rays + one cosine-hemisphere AO ray per primary hit (closest-hit queries, as the reference's
CheckForOccluder does).  One "step" = one pass over all samples of the image.

  value     device-resident wavefront pass (nrt_render_ao_device; N > 1: nrt_render_ao_sharded), scene + BVH in HBM.
  e2e       the same rays through the reference-facing batch call nrt_traverse with HOST buffers (pinned):
            H2D of 36-byte rays and D2H of 16-byte hits + 1-byte flags are inside the timed region; the measured
            pinned-copy rates of the box are printed beside it.
  roofline  three roofs for the traversal kernel -- instruction issue, L2 bandwidth, HBM bandwidth -- from counters of a
            committed ncu capture (profiles/r02_traverse_counters.json, per ray) scaled by this run's measured
            rays/s, against roofs measured in this run (nrt_probe_read_gbs) / MEASURED_PEAKS.json; `bound` names the
            largest fraction.  `algorithmic_gbs` is SURVEY.md 8(d)'s bytes-per-ray figure, for reference only.
  parity    gates run BEFORE any timing: fast kernel == conformance kernel on every ray of the step, frame sum ==
            primary misses + unoccluded AO rays; the CPU-baseline leg's reference hits are compared with the GPU's.
  configs   the other BASELINE.json configurations, each with its own gates, clocks and numbers:
            1 M-triangle terrain primary+AO (the north star's >= 1e9 rays/s target), configs[2] path-tracer loop at
            64 spp, configs[3] 10 M-triangle build + 4K primary rays; with --gpus 8 also configs[4] (4Kx4Kx256 spp,
            tile-sharded).
  N > 1     one process per GPU (torchrun).  Default STRONG scaling: the fixed 1920x1080x64 spp frame of the north
            star, tiles dealt round-robin to the ranks, BVH rebuilt identically on every rank, one collective per
            step -- the framebuffer all-gather inside nrt_render_ao_sharded (NCCL, C-ABI; no torch op in the timed
            path).  --scaling weak keeps round 1's 16*N spp.
  --impl reference : the UNMODIFIED reference (oracle/_ref, built from /root/reference/nanort.h) -- or the oracle port
            when that is absent -- traces a bounded sample of the very same ray arrays on the host cores, after a
            thread sweep {1, 2, 4, ..., nproc}; rank 0 only.
  --dump-outputs DIR : after the timed steps, what the last timed step computed, as DIR/<name>.npy (float32 / float64):
            frame.npy, the HEIGHT x WIDTH framebuffer (per pixel, the number of samples whose AO ray was not occluded;
            primary misses count as unoccluded).  The inputs depend on the arguments only, so two builds can be
            compared output for output.  (--impl reference traces a sample sized by a timing calibration: no dump.)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WIDTH, HEIGHT, SPP = 1920, 1080, 16
STRONG_SPP = 64  # the north star's frame: 1920x1080x64 spp, fixed total work
TILE_W, TILE_H = 64, 8
SCENE = "sphere_grid"
METRIC = "Mrays/sec (primary+1-bounce AO)"
UNIT = "Mrays/s"
SM_COUNT, SMSP_PER_SM = 148, 4


# ----------------------------------------------------------------------------------- helpers
def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms for the whole run; window() extracts a timed region."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def window(self, t_begin, t_end):
        """Median SM clock and throttle reasons of the samples taken inside [t_begin, t_end] (time.time())."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        import datetime

        sm, mx, reasons, sm_all = [], [], set(), []
        for ln in list(self.lines):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                clk, cmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            sm_all.append(clk)
            if not (t_begin - 0.05 <= ts <= t_end + 0.05):
                continue
            sm.append(clk)
            mx.append(cmax)
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else (float(np.median(sm_all)) if sm_all else None),
                "sm_max_mhz": max(mx) if mx else None, "samples_in_timed_region": len(sm),
                "samples_total": len(sm_all), "reasons": sorted(reasons)}


def ao_params(api, cam, width, height, spp, diag, n_shards, shard, ao_frac=0.25, flags=0):
    p = api.AoParams()
    for i in range(12):
        p.cam[i] = float(cam[i])
    p.width, p.height, p.spp, p.sample0, p.seed = width, height, spp, 0, 1
    p.tile_w, p.tile_h, p.shard, p.n_shards = TILE_W, TILE_H, shard, n_shards
    p.ray_min_t, p.ray_max_t, p.ao_min_t, p.ao_max_t = 1e-3, 1e30, 1e-3, ao_frac * diag
    p.flags = flags
    return p


def config_dict(n_gpus, scaling, spp_total):
    return {
        "workload": f"sphere_grid 100,002 triangles (BASELINE.json configs[1]), {WIDTH}x{HEIGHT}, {spp_total} spp in total "
                    f"over {n_gpus} GPU(s), primary + 1 cosine AO ray per hit, closest-hit; tiles {TILE_W}x{TILE_H} round-robin "
                    f"over ranks; BVH replicated; framebuffer all-gather (NCCL inside nrt_render_ao_sharded)"
                    + ("" if n_gpus > 1 else "; N=1: the configuration the metric is quoted on (16 spp)"),
        "scaling_mode": scaling,
        "l2_policy": "inputs larger than L2: camera rays are generated inside the traversal kernel (no input stream); the "
                     "only stream between the two launches of a wave is the compacted AO queue, ~9 M rays x 36 B = 330 MB per "
                     "16 Mi-ray wave = 2.6 x the 126 MB L2; scene + BVH (10 MB) stay cache-resident by design",
        "parallelism": f"ray-tile sharding x{n_gpus}",
    }


def dump_outputs(out_dir, **arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, np.float32 if a.dtype.itemsize <= 4 else np.float64))


# ----------------------------------------------------------------------------------- reference arm
def host_cpu_info():
    info = {"nproc": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = info["nproc"]
    try:
        info["cgroup_cpu_max"] = open("/sys/fs/cgroup/cpu.max").read().strip()
    except Exception:
        info["cgroup_cpu_max"] = None
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["model"] = ln.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return info


class CpuReference:
    """The reference's own CPU implementation of the path: oracle/_ref (unmodified nanort.h) when it was built, else the
    oracle port.  This is the one place outside tests/ that executes oracle/ -- as the timed CPU baseline and, with the
    hits it returns, as the checker of the GPU's records (never as a product path)."""

    def __init__(self, verts, faces):
        from oracle import orc

        self.cpu = host_cpu_info()
        self.max_threads = max(1, self.cpu["affinity"])
        self.threads = self.max_threads
        t0 = time.time()
        if orc.Reference.available(True):
            self.kind = "reference"
            self.acc = orc.Reference(True).build(verts, faces)
            self._trav = lambda rays, th: self.acc.traverse(rays, threads=th)
        else:
            self.kind = "port"
            port = orc.Port()
            nodes, idx, _ = port.build(verts, faces, mode=orc.MODE_CPP11)
            self._trav = lambda rays, th: port.traverse(nodes, idx, verts, faces, rays, threads=th)
        self.build_s = time.time() - t0
        self.sweep = None

    def trav(self, rays):
        return self._trav(rays, self.threads)

    def thread_sweep(self, rays, budget_s=12.0):
        """BASELINE.md 3.4: {1, 2, 4, ..., nproc} threads, best of 3 each, on a sample sized for ~1 s single-threaded;
        keeps the best thread count for the timed leg and reports the whole curve (the reference's thread scaling is
        erratic, BASELINE.md section 2 -- all cores is often NOT the fastest)."""
        counts, t = [], 1
        while t < self.max_threads:
            counts.append(t)
            t *= 2
        counts.append(self.max_threads)
        probe = rays[:: max(1, len(rays) // 4000)]
        t0 = time.time()
        self._trav(probe, 1)
        rate1 = len(probe) / max(time.time() - t0, 1e-4)
        n = int(min(len(rays), max(4000, rate1 * 1.0)))
        sample = np.ascontiguousarray(rays[:: max(1, len(rays) // n)])
        curve, t_start = [], time.time()
        for th in counts:
            best = 0.0
            for _ in range(3):
                t0 = time.time()
                self._trav(sample, th)
                best = max(best, len(sample) / max(time.time() - t0, 1e-6))
                if time.time() - t_start > budget_s:
                    break
            curve.append({"threads": th, "mrays_s": best / 1e6})
            if time.time() - t_start > budget_s:
                break
        top = max(curve, key=lambda c: c["mrays_s"])
        self.threads = top["threads"]
        self.sweep = {"sample_rays": len(sample), "curve": curve, "best_threads": top["threads"],
                      "single_thread_mrays_s": curve[0]["mrays_s"], "best_mrays_s": top["mrays_s"]}
        return self.sweep

    def calibrate(self, primary, ao, target_s=10.0):
        """Picks a strided sample of the two exported ray arrays that takes about target_s seconds."""
        probe_n = 20000
        for _ in range(4):  # grow the probe until it runs long enough to give a stable rate
            sp = primary[:: max(1, len(primary) // probe_n)]
            sa = ao[:: max(1, len(ao) // probe_n)]
            t0 = time.time()
            self.trav(sp)
            self.trav(sa)
            dt = max(time.time() - t0, 1e-3)
            if dt > 1.0 or probe_n >= len(primary):
                break
            probe_n *= 6
        rate = (len(sp) + len(sa)) / dt
        want = int(rate * target_s)
        frac = min(1.0, want / float(len(primary) + len(ao)))
        self.stride = max(1, int(round(1.0 / frac)))
        self.sample_primary = np.ascontiguousarray(primary[:: self.stride])
        self.sample_ao = np.ascontiguousarray(ao[:: self.stride])
        self.sample_desc = (f"every {self.stride}-th ray of the step's {len(primary)} primary + {len(ao)} AO rays "
                            f"({len(self.sample_primary)} + {len(self.sample_ao)} rays)")

    def calibrate_standalone(self, S, verts, faces, cam, ao_max_t, target_s=10.0):
        """Reference arm: no GPU code anywhere.  The sample's rays come from the numpy generators (same camera / jitter
        hash as the device pass): every k-th pixel, all SPP samples, AO rays from the reference's own primary hits."""

        def make(stride):
            pixels = np.arange(0, WIDTH * HEIGHT, stride, dtype=np.int64)
            prim = S.primary_rays(cam, WIDTH, HEIGHT, spp=SPP, seed=1, pixels=pixels, min_t=1e-3, max_t=1e30)
            hits, mask = self.trav(prim)
            ao, _ = S.ao_rays(verts, faces, prim, hits, mask, seed=2, min_t=1e-3, max_t=ao_max_t)
            return prim, ao

        stride = max(1, (WIDTH * HEIGHT * SPP) // 20000)
        prim, ao = make(stride)
        self.thread_sweep(np.concatenate([prim, ao]))
        for _ in range(4):  # grow the probe until it runs long enough to give a stable rate
            prim, ao = make(stride)
            t0 = time.time()
            self.trav(prim)
            self.trav(ao)
            dt = max(time.time() - t0, 1e-3)
            if dt > 1.0 or stride == 1:
                break
            stride = max(1, stride // 6)
        rate = (len(prim) + len(ao)) / dt
        want = rate * target_s
        full = WIDTH * HEIGHT * SPP * (1.0 + len(ao) / max(1, len(prim)))
        stride = max(1, int(round(full / want)))
        self.sample_primary, self.sample_ao = make(stride)
        self.sample_desc = (f"every {stride}-th pixel of {WIDTH}x{HEIGHT} at {SPP} spp, numpy-generated: "
                            f"{len(self.sample_primary)} primary + {len(self.sample_ao)} AO rays")

    def step(self):
        t0 = time.time()
        self.hits_primary = self.trav(self.sample_primary)
        self.hits_ao = self.trav(self.sample_ao)
        return time.time() - t0, len(self.sample_primary) + len(self.sample_ao)

    def describe(self, value, extra=None):
        d = {"value": value, "unit": UNIT, "cores": self.threads, "kind": self.kind, "sample": self.sample_desc,
             "build_s": self.build_s, "host": self.cpu, "thread_sweep": self.sweep}
        if extra:
            d.update(extra)
        return d


def reference_arm(args):
    from nanort_b200 import scenes as S

    verts, faces = S.make_scene(SCENE)
    cam = S.scene_camera(SCENE, WIDTH, HEIGHT)
    diag = float(np.linalg.norm(verts.max(axis=0) - verts.min(axis=0)))
    ref = CpuReference(verts, faces)
    # every step traces the same bounded sample; the whole run (W + K steps) is kept to about 2.5 minutes
    per_step = max(2.0, min(10.0, 130.0 / max(1, args.steps + args.warmup)))
    if os.environ.get("NRT_BENCH_REF_STEP_S"):  # tests shrink the sample (tests/test_bench_contract.py)
        per_step = float(os.environ["NRT_BENCH_REF_STEP_S"])
    ref.calibrate_standalone(S, verts, faces, cam, 0.25 * diag, target_s=per_step)
    for _ in range(args.warmup):
        ref.step()
    tot_t, tot_n = 0.0, 0
    for _ in range(args.steps):
        dt, n = ref.step()
        tot_t += dt
        tot_n += n
    val = tot_n / tot_t / 1e6
    spp_total = SPP if args.gpus == 1 or args.scaling == "weak" else STRONG_SPP
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_t / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak" if args.gpus == 1 else args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_dict(args.gpus, args.scaling, spp_total),
        "cpu_baseline": ref.describe(val),
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------- parity gates (GPU side)
def gate_fast_vs_conformance(torch, api, acc, d_rays, n, dev, chunk=1 << 24):
    """Every ray of the step through the production kernel and through the conformance kernel (the reference's visiting
    order over the 40-byte node array); records must be bit-identical, except that at EXACTLY equal distance the two
    visiting orders may report different primitives (the reference itself keeps whichever it met last)."""
    diff_total, tie_total, checked = 0, 0, 0
    m = min(int(n), chunk)
    a = torch.empty(m * 16, dtype=torch.uint8, device=dev)
    b = torch.empty(m * 16, dtype=torch.uint8, device=dev)
    for off in range(0, int(n), chunk):
        m = min(chunk, int(n) - off)
        acc.TraverseDevice(d_rays.data_ptr() + off * 36, m, a.data_ptr(), flags=api.TRAVERSE_FAST)
        acc.TraverseDevice(d_rays.data_ptr() + off * 36, m, b.data_ptr(), flags=api.TRAVERSE_CONFORMANCE)
        ra, rb = a[: m * 16].view(torch.int32).view(-1, 4), b[: m * 16].view(torch.int32).view(-1, 4)
        ne = (ra != rb).any(dim=1)
        nd = int(ne.sum().item())
        if nd:
            same_t = (ra[ne][:, 2] == rb[ne][:, 2])
            tie_total += int(same_t.sum().item())
        diff_total += nd
        checked += m
    return {"rays_checked": checked, "records_different": diff_total, "of_which_exact_t_ties": tie_total,
            "ok": diff_total == tie_total}


def gate_frame_identity(torch, frame, r_primary, r_ao_hits):
    """frame.sum() == primary misses + unoccluded AO rays == primary rays - occluded AO rays (every sample adds 1.0 or
    nothing; float32 sums of <= 2^24 ones per pixel are exact)."""
    got = float(frame.double().sum().item())
    want = float(r_primary - r_ao_hits)
    return {"frame_sum": got, "primary_minus_occluded": want, "ok": got == want}


def compare_with_reference(S, h_rays_sample, gpu_hits, gpu_mask, ref_hits, ref_mask):
    """The CPU leg's hits (unmodified reference, its own tree) against the GPU's for the same sampled rays: hit flags and
    prim_id identical, t/u/v within 1e-5 relative (the north star's tolerance); exact-t ties counted separately."""
    rm, gm = ref_mask.astype(bool), gpu_mask.astype(bool)
    flags_equal = bool(np.array_equal(rm, gm))
    both = rm & gm
    prim_diff = both & (ref_hits["prim_id"] != gpu_hits["prim_id"])
    ties = prim_diff & (ref_hits["t"] == gpu_hits["t"])
    ok_prim = both & ~prim_diff

    def rel(a, b):
        return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-6))) if len(a) else 0.0

    rt = rel(gpu_hits["t"][ok_prim], ref_hits["t"][ok_prim])
    ru = float(np.max(np.abs(gpu_hits["u"][ok_prim] - ref_hits["u"][ok_prim]))) if ok_prim.any() else 0.0
    rv = float(np.max(np.abs(gpu_hits["v"][ok_prim] - ref_hits["v"][ok_prim]))) if ok_prim.any() else 0.0
    bits = bool(np.array_equal(gpu_hits[ok_prim].view(np.uint32), ref_hits[ok_prim].view(np.uint32)))
    n_prim_diff = int(prim_diff.sum())
    return {"rays": int(len(rm)), "hit_flags_equal": flags_equal, "prim_id_different": n_prim_diff,
            "of_which_exact_t_ties": int(ties.sum()), "max_rel_t": rt, "max_abs_u": ru, "max_abs_v": rv,
            "tuv_bit_identical": bits,
            "ok": flags_equal and n_prim_diff == int(ties.sum()) and rt <= 1e-5 and ru <= 1e-5 and rv <= 1e-5}


# ----------------------------------------------------------------------------------- roofline
def traversal_roofline(api, r, n_primary, n_ao, counts, clocks, local_rank):
    """Three roofs for the dominant kernel (traverse_fast3_kernel, both launch kinds of a wave).  Per-ray counters come
    from the committed ncu capture of the same kernels (tools/summarize_ncu.py -> profiles/r02_traverse_counters.json:
    warp instructions, active lanes, L2 bytes, DRAM bytes per ray and launch kind); they are multiplied by THIS run's rays
    per second (in-kernel time from CUDA events inside the pass) and divided by roofs measured in this run."""
    boxes_p, prims_p, boxes_a, prims_a = counts
    n = n_primary + n_ao
    alg_bytes = 52.0 * n + 40.0 * (boxes_p + boxes_a) + 52.0 * (prims_p + prims_a)
    trav_ms = float(r.traverse_ms)
    hbm_peak, hbm_src = measured_peak_gbs()
    roof = {
        "kernel": "traverse_fast3_kernel<CameraRays, ..., PrimaryToAoEpilogue> + traverse_fast3_kernel<SoaRays, ..., AoAccumulateEpilogue>",
        "launches_per_step": int(r.traverse_launches), "avg_launch_ms": trav_ms / max(1, r.traverse_launches),
        "primary_ms": float(r.primary_traverse_ms), "ao_ms": float(r.ao_traverse_ms),
        "traverse_share_of_step": trav_ms / float(r.total_ms),
        "algorithmic_gbs": alg_bytes / (trav_ms * 1e-3) / 1e9,
        "algorithmic_note": "SURVEY.md 8(d): 52 + 40*boxes + 52*prims bytes per ray on the nanort layout; the tree is cache "
                            "resident, so this is NOT DRAM traffic and is not used as `frac`",
        "alg_bytes_per_launch": alg_bytes / max(1, r.traverse_launches), "bytes_per_ray": alg_bytes / n,
        "boxes_per_ray": (boxes_p + boxes_a) / n, "prims_per_ray": (prims_p + prims_a) / n,
    }
    try:
        cj = json.load(open(os.path.join(ROOT, "profiles", "r02_traverse_counters.json")))
    except Exception:
        cj = None
    f_sm = (clocks.get("sm_mhz") or 1965.0) * 1e6
    issue_peak = SM_COUNT * SMSP_PER_SM * f_sm  # one warp instruction per cycle per SM sub-partition
    try:
        l2_peak = api.probe_read_gbs(48 << 20, 8, device=local_rank)
        hbm_probe = api.probe_read_gbs(2 << 30, 4, device=local_rank)
    except Exception as e:  # the probes are reporting aids; the bench line survives without them
        l2_peak, hbm_probe = None, None
        roof["probe_error"] = str(e)
    roof["measured_roofs"] = {"issue_ginst_s": issue_peak / 1e9, "l2_read_gbs": l2_peak, "hbm_read_gbs": hbm_probe,
                              "hbm_copy_gbs": hbm_peak, "hbm_copy_source": hbm_src}
    if cj and trav_ms > 0:
        tp, ta = float(r.primary_traverse_ms) * 1e-3, float(r.ao_traverse_ms) * 1e-3
        kinds = (("primary", n_primary, tp), ("ao", n_ao, ta))
        inst = sum(cj[k]["warp_inst_per_ray"] * cnt for k, cnt, _ in kinds)
        l2b = sum(cj[k]["l2_bytes_per_ray"] * cnt for k, cnt, _ in kinds)
        drb = sum(cj[k]["dram_bytes_per_ray"] * cnt for k, cnt, _ in kinds)
        t = tp + ta
        fr = {"issue": inst / t / issue_peak,
              "l2": (l2b / t / 1e9 / l2_peak) if l2_peak else None,
              "hbm": drb / t / 1e9 / hbm_peak}
        per_kind = {}
        for k, cnt, tk in kinds:
            if tk > 0:
                per_kind[k] = {"mrays_s": cnt / tk / 1e6, "issue_frac": cj[k]["warp_inst_per_ray"] * cnt / tk / issue_peak,
                               "lanes_of_32": cj[k]["lanes"], "warp_inst_per_ray": cj[k]["warp_inst_per_ray"],
                               "l1_wavefront_pct_ncu": cj[k].get("l1_wavefront_pct"),
                               "l2_gbs": cj[k]["l2_bytes_per_ray"] * cnt / tk / 1e9,
                               "dram_gbs": cj[k]["dram_bytes_per_ray"] * cnt / tk / 1e9}
        bound = max((k for k in fr if fr[k] is not None), key=lambda k: fr[k])
        unit = {"issue": "Ginst/s", "l2": "GB/s", "hbm": "GB/s"}[bound]
        ach = {"issue": inst / t / 1e9, "l2": l2b / t / 1e9, "hbm": drb / t / 1e9}[bound]
        peak = {"issue": issue_peak / 1e9, "l2": l2_peak, "hbm": hbm_peak}[bound]
        roof.update({"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": fr[bound], "fractions": fr,
                     "per_launch_kind": per_kind, "traffic": drb / max(1, r.traverse_launches),
                     "counters_source": cj.get("source"),
                     "peak_source": "issue: 148 SMs x 4 sub-partitions x measured SM clock; l2 / hbm read: nrt_probe_read_gbs "
                                    "in this run; hbm copy: " + hbm_src})
    else:
        ach = roof["algorithmic_gbs"]
        roof.update({"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                     "traffic": None, "peak_source": hbm_src,
                     "note": "profiles/r02_traverse_counters.json missing: only the algorithmic figure is available"})
    return roof


# ----------------------------------------------------------------------------------- the other BASELINE configs
def timed_block(torch, dev, fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.time()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1), t_begin, time.time()


def config_terrain_ao(torch, api, S, dev, local_rank, sampler, with_cpu):
    """1 M-triangle terrain, 1920x1080x16 spp primary + AO on one GPU: the north star's ">= 1.0e9 rays/s on a 1 M-triangle
    scene" target."""
    W, H, spp = 1920, 1080, 16
    verts, faces = S.make_scene("terrain")
    acc = api.BVHAccel(device=local_rank)
    acc.Build(len(faces), verts, faces)
    st = acc.GetStatistics()
    bmin, bmax = acc.BoundingBox()
    diag = float(np.linalg.norm(bmax - bmin))
    cam = S.scene_camera("terrain", W, H)
    p = ao_params(api, cam, W, H, spp, diag, 1, 0)
    accum = torch.zeros(W * H, dtype=torch.float32, device=dev)
    # gates on a 2-spp export of the same pass (8.3 M primary + AO rays, every ray fast vs conformance)
    pg = ao_params(api, cam, W, H, 2, diag, 1, 0)
    n = W * H * 2
    d_p = torch.empty(n * 36, dtype=torch.uint8, device=dev)
    d_a = torch.empty(n * 36, dtype=torch.uint8, device=dev)
    n_p, n_a = acc.ExportAOWorkload(pg, accum.data_ptr(), d_p.data_ptr(), d_a.data_ptr())
    gates = {"primary_fast_vs_conformance": gate_fast_vs_conformance(torch, api, acc, d_p, n_p, dev),
             "ao_fast_vs_conformance": gate_fast_vs_conformance(torch, api, acc, d_a, n_a, dev)}
    counts = acc.CountDevice(d_p.data_ptr(), n_p) + acc.CountDevice(d_a.data_ptr(), n_a)
    accum.zero_()
    r = acc.RenderAO(p, accum.data_ptr())
    gates["frame_identity"] = gate_frame_identity(torch, accum, r.primary_rays, r.ao_hits)

    def step():
        accum.zero_()
        acc.RenderAO(p, accum.data_ptr(), want_result=False)

    ms, t0, t1 = timed_block(torch, dev, step, 10, 3)
    rays = int(r.primary_rays + r.ao_rays)
    out = {"name": "terrain_1m_primary_ao", "workload": f"1,002,528-triangle terrain, {W}x{H}x{spp} spp primary + AO, 1 GPU "
                                                         "(north star: >= 1e9 rays/s on a 1 M-triangle scene)",
           "rays_per_step": rays, "steps": 10, "ms_per_step": ms / 10, "value": rays * 10 / (ms * 1e-3) / 1e6, "unit": UNIT,
           "target_mrays_s": 1000.0, "clocks": sampler.window(t0, t1), "parity": gates,
           "build": {"device_ms": st["build_secs"] * 1e3, "nodes": st["num_leaf_nodes"] + st["num_branch_nodes"],
                     "depth": st["max_tree_depth"]},
           "roofline": {"algorithmic_gbs": (52.0 * (n_p + n_a) + 40.0 * (counts[0] + counts[2]) + 52.0 * (counts[1] + counts[3]))
                        / (n_p + n_a) * rays * 10 / (ms * 1e-3) / 1e9,
                        "boxes_per_ray": (counts[0] + counts[2]) / (n_p + n_a), "prims_per_ray": (counts[1] + counts[3]) / (n_p + n_a),
                        "tree_bytes": {"pair_nodes_128B": (st["num_branch_nodes"]) * 128, "triangles_48B": len(faces) * 48},
                        "note": "same kernels as the headline; tree (75 MB wide nodes + 48 MB triangles) is L2-resident"}}
    if with_cpu:
        ref = CpuReference(verts, faces)
        hp = d_p[: n_p * 36].cpu().numpy().view(S.RAY_DTYPE)
        ha = d_a[: n_a * 36].cpu().numpy().view(S.RAY_DTYPE)
        ref.thread_sweep(np.concatenate([hp[::13], ha[::13]]), budget_s=6.0)
        ref.calibrate(hp, ha, target_s=4.0)
        dt, cnt = ref.step()
        gh, gm = acc.Traverse(np.concatenate([ref.sample_primary, ref.sample_ao]))
        rh = np.concatenate([ref.hits_primary[0], ref.hits_ao[0]])
        rm = np.concatenate([ref.hits_primary[1], ref.hits_ao[1]])
        out["parity"]["vs_reference_cpu"] = compare_with_reference(S, None, gh, gm, rh, rm)
        out["cpu_baseline"] = ref.describe(cnt / dt / 1e6)
    out["parity_ok"] = all(g.get("ok", False) for g in out["parity"].values())
    acc.free()
    return out


def config_path_tracer(torch, api, S, dev, local_rank, sampler):
    """BASELINE.json configs[2]: 1 M-triangle terrain + area light, 1920x1080, 64 spp, the reference path tracer's loop
    (<= 10 bounces, Russian roulette, next-event estimation with shadow rays); rays/s counts EVERY Traverse."""
    W, H, spp = 1920, 1080, 64
    v, f = S.make_scene("terrain")
    v, f, l0, ln = S.with_area_light(v, f, (0.0, 6.0, 0.0), 2.0, 2.0)
    mats = np.concatenate([S.material(diffuse=(0.7, 0.7, 0.7)), S.material(emission=(20, 20, 20))])
    ids = np.zeros(len(f), np.uint32)
    ids[l0:] = 1
    emissive = np.arange(l0, l0 + ln, dtype=np.uint32)
    acc = api.BVHAccel(device=local_rank)
    acc.Build(len(f), v, f)
    cam = S.scene_camera("terrain", W, H)
    d_m = torch.as_tensor(mats.view(np.float32).reshape(-1), device=dev)
    d_i = torch.as_tensor(ids.astype(np.int32), device=dev)
    d_e = torch.as_tensor(emissive.astype(np.int32), device=dev)
    p = api.PathParams()
    for i in range(12):
        p.cam[i] = float(cam[i])
    p.width, p.height, p.spp, p.sample0, p.seed = W, H, spp, 0, 3
    p.tile_w, p.tile_h, p.shard, p.n_shards = TILE_W, TILE_H, 0, 1
    p.max_bounces, p.ray_min_t, p.ray_max_t = 10, 1e-3, 1e30
    p.n_materials, p.n_emissive = len(mats), len(emissive)
    p.d_materials, p.d_material_ids, p.d_emissive_faces = d_m.data_ptr(), d_i.data_ptr(), d_e.data_ptr()
    p.d_facevarying_normals, p.flags = None, 0
    accum = torch.zeros(W * H * 3, dtype=torch.float32, device=dev)
    res = {}

    def step():
        accum.zero_()
        res["r"] = acc.RenderPath(p, accum.data_ptr())

    step()
    torch.cuda.synchronize(dev)
    t0 = time.time()
    ms_total, steps = 0.0, 3
    for _ in range(steps):
        step()
        ms_total += float(res["r"].total_ms)
    t1 = time.time()
    r = res["r"]
    rays = int(r.radiance_rays + r.shadow_rays)
    img = accum.view(H, W, 3) / spp
    finite = bool(torch.isfinite(img).all().item())
    out = {"name": "configs[2]_path_tracer_loop", "workload": f"1,002,528-triangle terrain + area light, {W}x{H}x{spp} spp, "
                                                               "<= 10 bounces, RR, NEE shadow rays (examples/path_tracer loop)",
           "camera_paths": int(r.camera_rays), "radiance_traverse_calls": int(r.radiance_rays), "shadow_traverse_calls": int(r.shadow_rays),
           "rays_per_step": rays, "steps": steps, "ms_per_step": ms_total / steps, "value": rays * steps / (ms_total * 1e-3) / 1e6,
           "unit": UNIT, "launches_per_step": int(r.launches), "traverse_share_of_step": float(r.traverse_ms) / float(r.total_ms),
           "clocks": sampler.window(t0, t1),
           "parity": {"counts": {"camera_paths": int(r.camera_rays), "expected": W * H * spp, "ok": int(r.camera_rays) == W * H * spp},
                      "image": {"finite": finite, "mean_radiance": [float(x) for x in img.mean(dim=(0, 1)).tolist()], "ok": finite},
                      "note": "shading parity against the reference's own code is the job of tests/test_gpu_path.py"},
           "timing": "device time of the whole pass (CUDA events inside nrt_render_path_device)"}
    out["parity_ok"] = all(g.get("ok", True) for g in out["parity"].values() if isinstance(g, dict))
    acc.free()
    return out


def config_build_10m(torch, api, S, dev, local_rank, sampler):
    """BASELINE.json configs[3]: 10 M-triangle (flattened instanced) scene: BVH build time + 3840x2160 primary rays."""
    W, H = 3840, 2160
    v, f = S.make_scene("instanced")
    builds = []
    acc = None
    for _ in range(3):
        if acc is not None:
            acc.free()
        acc = api.BVHAccel(device=local_rank)
        t0 = time.time()
        acc.Build(len(f), v, f)
        builds.append((acc.GetStatistics()["build_secs"] * 1e3, (time.time() - t0) * 1e3))
    st = acc.GetStatistics()
    bmin, bmax = acc.BoundingBox()
    diag = float(np.linalg.norm(bmax - bmin))
    cam = S.scene_camera("instanced", W, H)
    p = ao_params(api, cam, W, H, 1, diag, 1, 0, ao_frac=0.02)
    n = W * H
    accum = torch.zeros(n, dtype=torch.float32, device=dev)
    d_p = torch.empty(n * 36, dtype=torch.uint8, device=dev)
    d_a = torch.empty(n * 36, dtype=torch.uint8, device=dev)
    n_p, n_a = acc.ExportAOWorkload(p, accum.data_ptr(), d_p.data_ptr(), d_a.data_ptr())
    gates = {"primary_fast_vs_conformance": gate_fast_vs_conformance(torch, api, acc, d_p, n_p, dev)}
    hits = torch.empty(n * 16, dtype=torch.uint8, device=dev)

    def step():
        acc.TraverseDevice(d_p.data_ptr(), n_p, hits.data_ptr())

    ms, t0, t1 = timed_block(torch, dev, step, 10, 3)
    boxes, prims = acc.CountDevice(d_p.data_ptr(), n_p)
    nodes = st["num_leaf_nodes"] + st["num_branch_nodes"]
    best = min(b[0] for b in builds)
    out = {"name": "configs[3]_build_10m_4k_primary", "workload": f"{len(f):,}-triangle flattened instanced scene: Build + {W}x{H} primary rays",
           "build_ms": {"device_best_of_3": best, "device_all": [b[0] for b in builds], "wall_incl_upload_best": min(b[1] for b in builds),
                        "nodes": nodes, "depth": st["max_tree_depth"],
                        "algorithmic_bytes_per_pass": len(f) * (12 + 36) + len(f) * 4 + nodes * 40,
                        "note": "SURVEY.md 8(d): N*(12+36) read + N*4 indices + nodes*40 written per pass"},
           "rays_per_step": int(n_p), "steps": 10, "ms_per_step": ms / 10, "value": n_p * 10 / (ms * 1e-3) / 1e6, "unit": UNIT,
           "clocks": sampler.window(t0, t1), "parity": gates,
           "roofline": {"boxes_per_ray": boxes / n_p, "prims_per_ray": prims / n_p,
                        "algorithmic_gbs": (52.0 * n_p + 40.0 * boxes + 52.0 * prims) * 10 / (ms * 1e-3) / 1e9,
                        "tree_bytes": {"pair_nodes_128B": st["num_branch_nodes"] * 128, "triangles_48B": len(f) * 48},
                        "note": "the one scene whose tree (0.4 GB + 0.5 GB) exceeds the 126 MB L2"}}
    out["parity_ok"] = all(g.get("ok", False) for g in out["parity"].values())
    acc.free()
    return out


# ----------------------------------------------------------------------------------- main
def bind_to_gpu_numa_node(torch, local_rank):
    """Multi-rank runs: keep this rank's threads -- and with them its pinned host buffers (first touch) -- on the CPUs
    NVML reports as local to the rank's GPU, so that the host-buffer arm of 8 ranks does not cross the socket
    interconnect.  Best effort; any failure leaves the default affinity."""
    try:
        import pynvml

        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1 only: strong = the fixed 1920x1080x64 spp frame (default), weak = 16*N spp")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the additional BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 0)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world

    if args.impl == "reference":
        if rank != 0:
            return 0  # rank 0 alone runs and prints the reference arm
        return reference_arm(args)

    import torch

    from nanort_b200 import api, dist as nd, scenes as S

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        bind_to_gpu_numa_node(torch, local_rank)
    distributed = world > 1
    comm = None
    if distributed:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        # the library's own communicator (C-ABI): rank 0 makes the NCCL id, torch.distributed only ships the 128 bytes
        ids = [api.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = api.Comm(ids[0], rank, world, device=local_rank)

    sampler = ClockSampler(local_rank)
    sampler.start()

    verts, faces = S.make_scene(SCENE)
    cam = S.scene_camera(SCENE, WIDTH, HEIGHT)
    n_shards, shard = world, rank
    scaling = "weak" if (not distributed or args.scaling == "weak") else "strong"
    spp_total = SPP * world if (distributed and args.scaling == "weak") else (STRONG_SPP if distributed else SPP)

    acc = api.BVHAccel(device=local_rank)
    t0 = time.time()
    acc.Build(len(faces), verts, faces)
    build_wall_ms = (time.time() - t0) * 1e3
    stats = acc.GetStatistics()
    bmin, bmax = acc.BoundingBox()
    diag = float(np.linalg.norm(bmax - bmin))
    p = ao_params(api, cam, WIDTH, HEIGHT, spp_total, diag, n_shards, shard)
    accum = torch.zeros(WIDTH * HEIGHT, dtype=torch.float32, device=dev)

    # ---- the step's ray arrays, exported once (untimed) for the gates, the host-buffer arm, the CPU baseline, the counters
    slots = nd.shard_ray_count(WIDTH, HEIGHT, TILE_W, TILE_H, shard, n_shards, p.spp)
    d_primary = torch.empty(slots * 36, dtype=torch.uint8, device=dev)
    d_ao = torch.empty(slots * 36, dtype=torch.uint8, device=dev)
    n_primary, n_ao = acc.ExportAOWorkload(p, accum.data_ptr(), d_primary.data_ptr(), d_ao.data_ptr())
    assert n_primary == slots, (n_primary, slots)
    accum.zero_()

    # ---- parity gates, before any timing
    parity = {"primary_fast_vs_conformance": gate_fast_vs_conformance(torch, api, acc, d_primary, n_primary, dev),
              "ao_fast_vs_conformance": gate_fast_vs_conformance(torch, api, acc, d_ao, n_ao, dev)}
    frame = torch.zeros(WIDTH * HEIGHT, dtype=torch.float32, device=dev)
    if distributed:
        r0 = comm.RenderAO(acc, p, frame.data_ptr())
        tot = torch.tensor([float(r0.primary_rays), float(r0.ao_hits)], dtype=torch.float64, device=dev)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        parity["gathered_frame_identity"] = gate_frame_identity(torch, frame, tot[0].item(), tot[1].item())
        # every rank must hold the same frame after the all-gather
        chk = torch.tensor([float(frame.double().sum().item())], dtype=torch.float64, device=dev)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        parity["frame_equal_on_all_ranks"] = {"ok": bool(lo.item() == hi.item())}
    else:
        r0 = acc.RenderAO(p, frame.data_ptr())
        parity["frame_identity"] = gate_frame_identity(torch, frame, r0.primary_rays, r0.ao_hits)

    def device_step():
        if distributed:
            comm.RenderAO(acc, p, frame.data_ptr(), want_result=False)  # render own tiles + all-gather + unpack, all C-ABI
        else:
            accum.zero_()
            acc.RenderAO(p, accum.data_ptr(), want_result=False)

    def sync_all():
        torch.cuda.synchronize(dev)
        if distributed:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- value: device-resident pass, EXACTLY --steps steps between the two events
    for _ in range(args.warmup):
        device_step()
    sync_all()
    time.sleep(0.3)  # let nvidia-smi reach its streaming state before the timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    t_begin = time.time()
    e0.record()
    for _ in range(args.steps):
        device_step()
    e1.record()
    sync_all()
    t_end = time.time()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, frame=(frame if distributed else accum).view(HEIGHT, WIDTH).cpu().numpy())
    # the same steps again for >= 2 s (not part of `value`): clocks and thermals are sampled over a region long enough
    # for nvidia-smi's 50 ms period to see them; its rate is reported as `sustained`
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_sus0 = time.time()
    e2.record()
    sus_steps = 0
    while time.time() - t_sus0 < 2.0:
        for _ in range(args.steps):
            device_step()
        sus_steps += args.steps
        torch.cuda.synchronize(dev)
    e3.record()
    sync_all()
    t_sus1 = time.time()
    ms_sus = e2.elapsed_time(e3)
    clocks = sampler.window(t_begin, t_sus1)
    clocks["window"] = "timed region + the >= 2 s sustained block that follows it"
    clocks["timed_region_only"] = sampler.window(t_begin, t_end)
    # one more instrumented pass (outside the timed region) for counts, launch counts and the in-kernel time
    accum.zero_()
    r = acc.RenderAO(p, accum.data_ptr(), want_result=True)
    rays_step = int(r.primary_rays + r.ao_rays)
    t = torch.tensor([ms, ms_sus], dtype=torch.float64, device=dev)
    tot = torch.tensor([rays_step], dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_max, ms_sus_max, rays_all = float(t[0].item()), float(t[1].item()), float(tot.item())
    value = rays_all * args.steps / (ms_max * 1e-3) / 1e6
    sustained = {"value": rays_all * sus_steps / (ms_sus_max * 1e-3) / 1e6, "unit": UNIT, "steps": sus_steps,
                 "seconds": ms_sus_max * 1e-3}

    # ---- opt-in extra, NOT part of `value`: the same pass with NRT_TRAVERSE_ANY_HIT on the AO launch (the occlusion
    # rays stop at their first hit; nanort itself has no any-hit).  Same framebuffer bit for bit, fewer node visits.
    extras = {}
    if not distributed:
        try:
            p_any = ao_params(api, cam, WIDTH, HEIGHT, spp_total, diag, n_shards, shard, flags=api.TRAVERSE_ANY_HIT)
            ref_frame = accum.clone()
            any_frame = torch.zeros_like(accum)
            for _ in range(2):
                any_frame.zero_()
                ra = acc.RenderAO(p_any, any_frame.data_ptr(), want_result=True)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(args.steps):
                any_frame.zero_()
                acc.RenderAO(p_any, any_frame.data_ptr(), want_result=False)
            a1.record()
            torch.cuda.synchronize(dev)
            ms_any = a0.elapsed_time(a1)
            extras["occlusion_any_hit"] = {
                "value": rays_step * args.steps / (ms_any * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_any / args.steps,
                "ao_launch_ms": float(ra.ao_traverse_ms), "closest_hit_ao_launch_ms": float(r.ao_traverse_ms),
                "frame_identical_to_closest_hit": bool(torch.equal(any_frame, ref_frame)),
                "occluded_identical": int(ra.ao_hits) == int(r.ao_hits),
                "note": "opt-in (nrt_ao_params.flags |= NRT_TRAVERSE_ANY_HIT); the headline `value` is closest-hit on "
                        "every ray, like the reference's Traverse"}
            del ref_frame, any_frame
        except Exception as e:
            extras["occlusion_any_hit"] = {"error": str(e)}

    # ---- roofline of the dominant kernel
    counts = acc.CountDevice(d_primary.data_ptr(), n_primary) + acc.CountDevice(d_ao.data_ptr(), n_ao)
    roofline = traversal_roofline(api, r, n_primary, n_ao, counts, clocks, local_rank)

    # ---- e2e: host buffers through nrt_traverse (H2D rays, D2H hits + flags inside the timed region)
    e2e = None
    if not args.no_e2e:
        hp = api.PinnedArray(n_primary, S.RAY_DTYPE)
        ha = api.PinnedArray(max(n_ao, 1), S.RAY_DTYPE)
        hp.array[:] = d_primary.cpu().numpy().view(S.RAY_DTYPE)
        ha.array[:n_ao] = d_ao[: n_ao * 36].cpu().numpy().view(S.RAY_DTYPE)
        hits_p, mask_p = api.PinnedArray(n_primary, S.HIT_DTYPE), api.PinnedArray(n_primary, np.uint8)
        hits_a, mask_a = api.PinnedArray(max(n_ao, 1), S.HIT_DTYPE), api.PinnedArray(max(n_ao, 1), np.uint8)

        def host_step():
            acc.Traverse(hp.array, hits=hits_p.array, mask=mask_p.array)
            acc.Traverse(ha.array[:n_ao], hits=hits_a.array[:n_ao], mask=mask_a.array[:n_ao])

        for _ in range(2):
            host_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            host_step()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        # the host-buffer arm must report what the device pass found
        assert int(mask_p.array.sum()) == n_ao, "primary hits of the host-buffer arm != AO ray count"
        try:
            h2d, d2h = api.probe_copy_gbs(1 << 30, 0, device=local_rank), api.probe_copy_gbs(1 << 30, 1, device=local_rank)
        except Exception:
            h2d = d2h = None
        # N > 1: the same copy probe on ALL ranks at once -- what each GPU's link gets while its neighbours' are busy
        # (the ranks of one socket share its memory controllers and PCIe root: this, not a kernel, is why `e2e` stops
        # scaling with N)
        concurrent = None
        if distributed:
            # every rank reaches every collective below whatever its own probe does (a failed probe reports NaN)
            def probe(direction):
                try:
                    return float(api.probe_copy_gbs(1 << 30, direction, device=local_rank))
                except Exception:
                    return float("nan")
            dist.barrier()
            ch2d = probe(0)
            dist.barrier()
            cd2h = probe(1)
            both = torch.tensor([ch2d, cd2h], dtype=torch.float64, device=dev)
            lo, sm = both.clone(), both.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            concurrent = {"h2d_min_per_gpu": float(lo[0].item()), "h2d_sum": float(sm[0].item()),
                          "d2h_min_per_gpu": float(lo[1].item()), "d2h_sum": float(sm[1].item()),
                          "note": "nrt_probe_copy_gbs, 1 GiB per rank, all ranks at the same time"}
        e2e_rate = rays_all * args.steps / float(tt.item()) / 1e6
        per_gpu = e2e_rate / world * 1e6
        e2e = {"value": e2e_rate, "unit": UNIT,
               "h2d_bytes_per_step": int(36 * (n_primary + n_ao)), "d2h_bytes_per_step": int(17 * (n_primary + n_ao)),
               "api": "nrt_traverse (host rays -> host hits), pinned buffers, 2 calls per step",
               "measured_pinned_copy_gbs": {"h2d": h2d, "d2h": d2h, "note": "nrt_probe_copy_gbs, 1 GiB, this rank alone"},
               "concurrent_pinned_copy_gbs": concurrent,
               "achieved_copy_gbs_per_gpu": {"h2d": 36 * per_gpu / 1e9, "d2h": 17 * per_gpu / 1e9},
               "bound": "PCIe / host memory: 36 B up + 17 B down per ray"}
        # opt-in compact records (NRT_TRAVERSE_RAY32: the 32-byte ray without nanort::Ray::type, no hit flags: a miss is
        # prim_id == 0xFFFFFFFF): same hits, 32 B up + 16 B down per ray.  NOT the headline: the reference's Ray is 36 B.
        # (every rank reaches the collectives below whatever happens to its own leg)
        c_dt, c_same, c_err = float("nan"), False, None
        try:
            r32 = np.dtype((np.void, 32))
            hp32, ha32 = api.PinnedArray(n_primary, r32), api.PinnedArray(max(n_ao, 1), r32)
            hp32.array.view(np.uint8).reshape(-1, 32)[:] = hp.array.view(np.uint8).reshape(-1, 36)[:, :32]
            ha32.array.view(np.uint8).reshape(-1, 32)[:n_ao] = ha.array.view(np.uint8).reshape(-1, 36)[:n_ao, :32]
            hits_p2 = api.PinnedArray(n_primary, S.HIT_DTYPE)

            def compact_step():
                acc.Traverse(hp32.array, hits=hits_p2.array, mask=False, flags=api.TRAVERSE_RAY32)
                acc.Traverse(ha32.array[:n_ao], hits=hits_a.array[:n_ao], mask=False, flags=api.TRAVERSE_RAY32)

            for _ in range(2):
                compact_step()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                compact_step()
            torch.cuda.synchronize(dev)
            c_dt = time.perf_counter() - t0
            c_same = bool(np.array_equal(hits_p2.array.view(np.uint32), hits_p.array.view(np.uint32)))
            del hp32, ha32, hits_p2
        except Exception as e:  # a reporting extra: the bench line survives without it
            c_err = str(e)
        c_ok = c_err is None and c_dt == c_dt
        tc = torch.tensor([c_dt if c_ok else 0.0], dtype=torch.float64, device=dev)
        tok = torch.tensor([1.0 if c_ok else 0.0], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
            dist.all_reduce(tok, op=dist.ReduceOp.MIN)
        if tok.item() == 1.0:
            e2e["compact_records"] = {"value": rays_all * args.steps / float(tc.item()) / 1e6, "unit": UNIT,
                                      "api": "nrt_traverse(..., hit_mask = NULL, NRT_TRAVERSE_RAY32)",
                                      "h2d_bytes_per_step": int(32 * (n_primary + n_ao)),
                                      "d2h_bytes_per_step": int(16 * (n_primary + n_ao)),
                                      "hits_identical_to_the_36_byte_call": c_same}
        else:
            e2e["compact_records"] = {"error": c_err or "failed on another rank"}
        # for comparison, the wavefront entry point end to end: camera parameters in (host struct), framebuffer out to
        # pinned host memory every step -- what a renderer pays when it hands the whole pass to the library
        fb_host = torch.empty(WIDTH * HEIGHT, dtype=torch.float32).pin_memory()

        def render_step():
            device_step()
            fb_host.copy_(frame if distributed else accum, non_blocking=True)
            torch.cuda.synchronize(dev)

        for _ in range(2):
            render_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            render_step()
        dt = time.perf_counter() - t0
        tr = torch.tensor([dt], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(tr, op=dist.ReduceOp.MAX)
        e2e["render_api"] = {"value": rays_all * args.steps / float(tr.item()) / 1e6, "unit": UNIT,
                             "api": ("nrt_render_ao_sharded" if distributed else "nrt_render_ao_device") + " + framebuffer D2H per step",
                             "h2d_bytes_per_step": C.sizeof(api.AoParams), "d2h_bytes_per_step": WIDTH * HEIGHT * 4}

    # ---- CPU baseline beside it (rank 0, N = 1 only): thread sweep, then a bounded sample of the same rays; its hits
    # double as the reference check of the GPU's records for those rays
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        h_primary = d_primary.cpu().numpy().view(S.RAY_DTYPE)
        h_ao = d_ao[: n_ao * 36].cpu().numpy().view(S.RAY_DTYPE)
        ref = CpuReference(verts, faces)
        ref.thread_sweep(np.concatenate([h_primary[::61], h_ao[::61]]))
        ref.calibrate(h_primary, h_ao, target_s=10.0)
        dt, n = ref.step()
        gh, gm = acc.Traverse(np.concatenate([ref.sample_primary, ref.sample_ao]))
        parity["vs_reference_cpu"] = compare_with_reference(
            S, None, gh, gm, np.concatenate([ref.hits_primary[0], ref.hits_ao[0]]),
            np.concatenate([ref.hits_primary[1], ref.hits_ao[1]]))
        cpu_baseline = ref.describe(n / dt / 1e6)
    parity["ok"] = all(g.get("ok", False) for g in parity.values() if isinstance(g, dict))

    # ---- the other BASELINE configurations
    configs = []
    if not args.no_configs:
        if not distributed:
            for fn in (lambda: config_terrain_ao(torch, api, S, dev, local_rank, sampler, with_cpu=not args.no_cpu_baseline),
                       lambda: config_path_tracer(torch, api, S, dev, local_rank, sampler),
                       lambda: config_build_10m(torch, api, S, dev, local_rank, sampler)):
                try:
                    configs.append(fn())
                except Exception as e:  # a failing extra config is reported, it does not take the headline line with it
                    configs.append({"error": repr(e)})
        elif world >= int(os.environ.get("NRT_BENCH_C5_MIN_WORLD", "8")):  # configs[4] names 8 GPUs; lower it to rehearse the path
            try:
                configs.append(config_c5_sharded(torch, dist, api, S, dev, local_rank, rank, world, comm, sampler))
            except Exception as e:
                configs.append({"error": repr(e)})
    sampler.stop()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args.gpus, scaling, spp_total),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(r.launches + (2 if distributed else 0)) * args.steps,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity, "sustained": sustained,
            "build": {"device_ms": stats["build_secs"] * 1e3, "wall_ms_incl_upload": build_wall_ms,
                      "nodes": stats["num_leaf_nodes"] + stats["num_branch_nodes"], "depth": stats["max_tree_depth"]},
            "rays_per_step": rays_all, "ao_occluded_fraction": float(r.ao_hits) / max(1, r.ao_rays),
            "extras": extras, "configs": configs,
        }
        print(json.dumps(line), flush=True)
    if comm is not None:
        comm.free()
    if distributed:
        dist.destroy_process_group()
    return 0


def config_c5_sharded(torch, dist, api, S, dev, local_rank, rank, world, comm, sampler):
    """BASELINE.json configs[4]: 1 M-triangle terrain, 4096x4096, 256 spp primary + AO, tiles of 64x64 pixels round-robin
    over the ranks, framebuffer all-gather (201 MB in RGB32F terms; one float per pixel here = 67 MB)."""
    W, H, spp = 4096, 4096, 256
    verts, faces = S.make_scene("terrain")
    acc = api.BVHAccel(device=local_rank)
    acc.Build(len(faces), verts, faces)
    bmin, bmax = acc.BoundingBox()
    diag = float(np.linalg.norm(bmax - bmin))
    cam = S.scene_camera("terrain", W, H)
    p = ao_params(api, cam, W, H, spp, diag, world, rank)
    p.tile_w, p.tile_h = 64, 64
    frame = torch.zeros(W * H, dtype=torch.float32, device=dev)
    r = comm.RenderAO(acc, p, frame.data_ptr())  # warm-up + counts
    tot = torch.tensor([float(r.primary_rays), float(r.ao_rays), float(r.ao_hits)], dtype=torch.float64, device=dev)
    dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    gate = gate_frame_identity(torch, frame, tot[0].item(), tot[2].item())
    torch.cuda.synchronize(dev)
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    steps = 2
    for _ in range(steps):
        comm.RenderAO(acc, p, frame.data_ptr(), want_result=False)
    e1.record()
    torch.cuda.synchronize(dev)
    dist.barrier()
    t1 = time.time()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    rays = float(tot[0].item() + tot[1].item())
    parity = {"gathered_frame_identity": gate}
    if rank == 0:
        # a strided sample of this frame's camera rays and of the AO rays they spawn (host generators, same arithmetic as
        # the device): production kernel == conformance kernel on every sampled ray, and == the unmodified reference
        pix = np.arange(0, W * H, 193, dtype=np.int64)
        prim = S.primary_rays(cam, W, H, spp=1, seed=1, pixels=pix, min_t=1e-3, max_t=1e30)
        h, m = acc.Traverse(prim)
        ao, _ = S.ao_rays(verts, faces, prim, h, m, seed=2, min_t=1e-3, max_t=0.25 * diag)
        sample = np.concatenate([prim, ao])
        d_s = torch.as_tensor(sample.view(np.uint8).reshape(-1), device=dev)
        parity["sample_fast_vs_conformance"] = gate_fast_vs_conformance(torch, api, acc, d_s, len(sample), dev)
        try:
            ref = CpuReference(verts, faces)
            gh, gm = acc.Traverse(sample)
            rh, rm = ref.trav(sample)
            parity["sample_vs_reference_cpu"] = compare_with_reference(S, None, gh, gm, rh, rm)
        except Exception as e:  # the reference library is test infrastructure; its absence does not fail the config
            parity["sample_vs_reference_cpu"] = {"skipped": repr(e)}
    acc.free()
    return {"name": "configs[4]_4k4k_256spp_sharded", "workload": f"1,002,528-triangle terrain, {W}x{H}x{spp} spp primary + AO, "
                                                                   f"64x64-pixel tiles round-robin over {world} GPUs, framebuffer all-gather",
            "rays_per_step": rays, "steps": steps, "ms_per_step": float(t.item()) / steps,
            "value": rays * steps / (float(t.item()) * 1e-3) / 1e6, "unit": UNIT, "clocks": sampler.window(t0, t1),
            "parity": parity, "parity_ok": all(g.get("ok", True) for g in parity.values())}


if __name__ == "__main__":
    sys.exit(main())
