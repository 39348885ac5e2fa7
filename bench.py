#!/usr/bin/env python
"""bench.py -- the measurement contract of this repo.

    python bench.py --gpus N --steps K --warmup W                      # our arm (CUDA backend)
    python bench.py --impl reference --gpus N --steps K --warmup W     # the reference's own CPU renderer (oracle/_ref)

Metric (BASELINE.json): Mrays/s (primary+secondary) at 1080p, 8 bounces, on the "hall-250k" synthetic scene
(config #2: diffuse; `--workload hall-principled` = config #3).  A STEP is one sample per pixel of the frame through the
whole wavefront: raygen -> trace -> shade -> shadow -> [sort -> trace(+lights) -> shade -> shadow] x 8 -> resolve.
rays = rays handed to the closest-hit trace (primary + every bounce), from device counters (SURVEY.md section 8(d)).

value   : whole-job Mrays/s with the scene resident in HBM, K steps enqueued back to back, timed with CUDA events on the
          launching stream (max over ranks), one framebuffer gather per sample batch inside the timed region when N > 1.
e2e     : the same metric through the public API one blocking call at a time -- RendererBase::RenderScene (pass
          descriptor host->device) and a device->host read of the whole frame into page-locked memory per step (N = 1:
          the renderer's mirror, as get_raw_pixels_ref; N > 1: every rank copies its strip into ONE shared page-locked
          host frame over its own PCIe link, then a barrier).  The unchanged scene is not re-uploaded per step (a real
          caller does not either); one upload + one step is timed separately (scene_upload_plus_one_step_ms).
N > 1   : weak scaling -- the frame grows to 1920 x (1080 N) and rank r renders rows [1080 r, 1080 (r+1)) of it; no
          inter-bounce communication; the device-timed arm keeps one NCCL gather of the strips per sample batch, the e2e
          arm delivers to the host as above.  `strong_scaling`: ONE 1920x1080 frame split over the N ranks.
configs : at N = 1 the other BASELINE.json configs (#1 Cornell 256^2, #3 hall-principled, #5 instanced 4096^2) are measured
          in the same run and reported as sub-objects; `cpu_baseline` = the reference's AVX-512 renderer on the host cores
          this process may really use (affinity and cgroup quota), on a bounded sample of the same workload.
--dump-outputs DIR : after the timed steps, the frame the timed path delivered after its last step is written as
          DIR/raw.npy (linear radiance, (H, W, 4) float32) and, at N = 1, DIR/final.npy (the tonemapped plane).  Together
          they stay within 64 * 10^6 bytes: an array that does not fit the rest of that budget is replaced by a fixed,
          seeded sample of its pixels, (k, 4) (at 1080p: raw.npy whole, final.npy 93% of its pixels).  The scenes are
          generated deterministically and the built-in sampler table is used, so the same arguments give the same inputs
          on every run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# NCCL writes its banner / debug lines to stdout by default: stdout carries the ONE JSON line of the contract and nothing else
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mrays/s (primary+secondary) at 1080p, 8 bounces"
UNIT = "Mrays/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="hall-diffuse", choices=["hall-diffuse", "hall-principled", "cornell", "c5-instanced"])
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the extra BASELINE.json configs (#1, #3, #5) at N=1")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--gather-every", type=int, default=0, help="steps per framebuffer gather (0 = once per timed batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", default="auto", help="WxHxSPP of the bounded CPU sample (auto: by host core count)")
    ap.add_argument("--no-sort", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the planes of the last timed step to DIR/*.npy")
    return ap.parse_args()


DUMP_BUDGET = 64 * 10 ** 6  # bytes, .npy headers included
NPY_HEADER = 128


def dump_outputs(out_dir, arrays):
    """Save each (H, W, C) array as out_dir/<name>.npy in float32, in order; an array that does not fit what is left of
    DUMP_BUDGET is saved as a fixed, seeded sample of its pixels instead."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BUDGET
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes + NPY_HEADER > left:
            px = a.reshape(-1, a.shape[-1])
            k = max(left - NPY_HEADER, 0) // px[0].nbytes
            a = px[np.sort(np.random.default_rng(0).choice(len(px), k, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes + NPY_HEADER


def make_desc(workload, w, h):
    from ray_b200 import scenes
    if workload == "hall-diffuse":
        return scenes.hall("diffuse", w, h)
    if workload == "hall-principled":
        return scenes.hall("principled", w, h)
    if workload == "c5-instanced":
        return scenes.c5_instanced(w, h)
    return scenes.cornell_box(w, h)


def host_cores():
    """Host threads this process can really use: affinity mask capped by the cgroup cpu quota (a 1-GPU lease of a big
    node reports 128 logical CPUs but may be throttled to a fraction of them)."""
    info = {"cpu_count": os.cpu_count() or 1}
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else info["cpu_count"]
    info["affinity"] = n
    info["cgroup_quota"] = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                txt = f.read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    info["cgroup_quota"] = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                        info["cgroup_quota"] = q / float(f2.read().split()[0])
            break
        except Exception:
            continue
    if info["cgroup_quota"]:
        n = max(1, min(n, int(info["cgroup_quota"] + 0.5)))
    info["threads"] = n
    return info


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def roofline(counters, kms, samples):
    """Per kernel family: ALGORITHMIC stream bytes (SURVEY.md section 8(d)) / device time of the family.
    The dominant family (largest device time) is the one reported as `roofline`."""
    prim, sec, sh = counters["primary_rays"], counters["secondary_rays"], counters["shadow_rays"]
    rays = prim + sec
    fam = {
        # read o,d,xy,depth (40 B incl. both uint2) + t_max 4 B (primary only keeps a hit record: 20 B), write hit 20 B
        "trace_closest": 56 * rays,
        # read ray 72 + hit 20; write 72/secondary ray + 48/shadow ray; radiance 16 W (primary) | 32 RMW (secondary);
        # primary AOVs 64 RMW
        "shade": 92 * rays + 76 * sec + 48 * sh + 80 * prim + 32 * sec,  # 72 B ray + 4 B sort key per secondary ray
        # read 48 B shadow ray, RMW 32 B radiance
        "trace_shadow": 80 * sh,
        # scatter: key 4 R + ray 72 R + ray 72 W (keys and the histogram are produced by the shade kernel)
        "sort": 148 * sec,
        # temp 16 R, full 32 RMW, half 32 RMW (every other iteration), raw 16 W, final 16 W, variance 16 W, req 4
        "resolve": 124 * (prim // max(samples, 1)) * samples,
        "raygen": 92 * prim,
    }
    peak, peak_src = measured_peak_gbs()
    out = {}
    for k, b in fam.items():
        ms, n = kms[k]
        if ms > 0 and n > 0:
            out[k] = {"ms_total": ms, "launches": int(n), "avg_launch_ms": ms / n, "algorithmic_bytes": int(b),
                      "achieved_gbs": b / (ms * 1e-3) / 1e9}
    dom = max(out, key=lambda k: out[k]["ms_total"])
    d = out[dom]
    traffic = None
    prof = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get(dom)
        except Exception:
            traffic = None
    scene_term = 224 * counters["nodes_visited"] + 384 * counters["leaves_tested"]
    return {"bound": "hbm", "kernel": dom, "achieved": d["achieved_gbs"], "peak": peak, "unit": "GB/s",
            "frac": d["achieved_gbs"] / peak, "traffic": traffic, "peak_source": peak_src,
            "bytes_per_launch": d["algorithmic_bytes"] / d["launches"], "avg_launch_ms": d["avg_launch_ms"],
            "note": "branchy scalar FP over an L2-resident scene: latency/divergence-bound, not bandwidth-bound; "
                    "scene_term_bytes = 224 B x nodes visited + 384 B x leaf blocks tested (cold-cache upper bound)",
            "scene_term_bytes": int(scene_term), "families": out}


def rays_per_sample_ref(osc, w, h):
    """Ray count of ONE sample through the reference's own stage functions (the API has no ray counters)."""
    import numpy as np
    from ray_b200.cuda import HIT_DTYPE
    cam = osc.camera()
    rays, hits = osc.generate_primary_rays(w, h, (0, 0, w, h), 1)
    rays, hits = osc.trace_rays(1, rays, hits, False)
    total = len(rays)
    temp = np.zeros((h, w, 4), np.float32)
    sec, sh, _, _ = osc.shade(w, h, 1, True, 0, rays, hits, temp)
    for bounce in range(1, cam.max_total_depth + 1):
        if len(sec) == 0:
            break
        hits0 = np.zeros(len(sec), dtype=HIT_DTYPE)
        hits0["obj_index"] = -1
        hits0["prim_index"] = -1
        hits0["t"] = np.float32(3.402823466e+30)
        hits0["v"] = -1.0
        total += len(sec)
        r2, h2 = osc.trace_rays(1, sec, hits0, True)
        sec, sh, _, _ = osc.shade(w, h, 1, False, bounce, r2, h2, temp)
    return total


def cpu_reference_run(workload, sample, steps, warmup):
    """Time the reference's widest CPU renderer (oracle/_ref, all host threads) on a bounded sample of the workload."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle
    from ray_b200 import capi, scenes
    cores = host_cores()
    threads = int(os.environ.get("BENCH_CPU_THREADS", "0")) or cores["threads"]
    if sample == "auto":
        # ~10-30 s of CPU work: a 16th of the frame per 16 hardware threads (at least 480x270), 2 spp per step
        sample = "1920x1080x2" if threads >= 128 else ("960x540x2" if threads >= 24 else "480x270x2")
    w, h, spp = [int(x) for x in sample.lower().split("x")]
    tile = 64 if (w // 64) * (h // 64) >= 4 * threads else 32
    desc = make_desc(workload, w, h)
    feats = oracle.load().ro_cpu_features()
    rtype, rname = capi.RT_REFERENCE, "REF"
    for bit, t, n in ((8, capi.RT_AVX512, "AVX512"), (4, capi.RT_AVX2, "AVX2"), (2, capi.RT_AVX, "AVX"), (1, capi.RT_SSE41, "SSE41")):
        if feats & bit:
            rtype, rname = t, n
            break
    osc = scenes.build(desc, oracle.Scene(wide=(rtype != capi.RT_REFERENCE)))
    rps = rays_per_sample_ref(osc, w, h)
    r = oracle.Renderer(rtype, w, h)
    for _ in range(warmup):
        r.render_mt(osc, 1, threads, tile)
    secs = 0.0
    for _ in range(steps):
        secs += r.render_mt(osc, spp, threads, tile)
    value = rps * spp * steps / secs / 1e6
    return {"value": value, "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": f"{workload} at {w}x{h}, {spp} spp per step x {steps} steps, Ray::{rname} renderer "
                      f"(unmodified reference, oracle/_ref), {threads} threads over {tile}x{tile} tiles "
                      f"(os.cpu_count {cores['cpu_count']}, affinity {cores['affinity']}, cgroup quota {cores['cgroup_quota']}); "
                      f"rays/sample counted once with the reference's Ref:: stage functions ({rps})",
            "seconds": secs, "ms_per_step": secs / steps * 1e3, "spp_per_step": spp, "frame": f"{w}x{h}",
            "host": cores}


def cpu_single_thread_ref(workload, w, h, spp):
    """config #1 is quoted on RendererRef, single thread: time it on a bounded number of samples."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle
    from ray_b200 import capi, scenes
    desc = make_desc(workload, w, h)
    osc = scenes.build(desc, oracle.Scene(wide=False))
    rps = rays_per_sample_ref(osc, w, h)
    r = oracle.Renderer(capi.RT_REFERENCE, w, h)
    r.render_mt(osc, 1, 1, 64)
    secs = r.render_mt(osc, spp, 1, 64)
    return {"value": rps * spp / secs / 1e6, "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": f"{workload} {w}x{h}, {spp} spp, Ray::Reference renderer (RendererRef, BVH2), 1 thread"}


def measure_config(workload, w, h, steps, warmup, device=0):
    """One more BASELINE.json config on one GPU: device-timed K steps (scene resident) + the blocking public-API path."""
    import ctypes as C
    from ray_b200 import cuda, host, scenes
    t0 = time.perf_counter()
    desc = make_desc(workload, w, h)
    r = host.Renderer(w, h, device=device)
    s = scenes.build(desc, r.create_scene())
    build_s = time.perf_counter() - t0
    lib = cuda.load_library()
    ctx = r.native_context()
    rect = (0, 0, w, h)
    it = 0
    for _ in range(warmup):
        it = r.render(s, rect, it, 1)
    r.reset_stats()
    lib.rc_event_record(ctx, 0)
    it = r.render(s, rect, it, steps)
    lib.rc_event_record(ctx, 1)
    f = C.c_float(0)
    lib.rc_event_elapsed_ms(ctx, 0, 1, C.byref(f))
    ms = float(f.value)
    c = r.counters()
    rays = c["primary_rays"] + c["secondary_rays"]
    kms = r.kernel_ms()
    # e2e: one blocking RenderScene + frame read-back per step (scene already resident: it did not change)
    r.pixels(host.RAW, copy=False)
    r.reset_stats()
    e2e_steps = max(min(steps, 4), 1)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        it = r.render(s, rect, it, 1)
        r.pixels(host.RAW, copy=False)
    e2e_s = time.perf_counter() - t0
    c2 = r.counters()
    out = {"workload": f"{workload} {w}x{h}", "value": rays / (ms * 1e-3) / 1e6, "unit": UNIT, "steps": steps,
           "ms_per_step": ms / steps, "rays_per_step": rays / steps, "shadow_rays_per_step": c["shadow_rays"] / steps,
           "e2e": {"value": (c2["primary_rays"] + c2["secondary_rays"]) / e2e_s / 1e6, "unit": UNIT,
                   "d2h_bytes_per_step": w * h * 16, "h2d_bytes_per_step": 256, "steps": e2e_steps},
           "triangles": desc.triangle_count(), "instances": len(desc.instances), "bvh8_nodes": s.node_count(),
           "scene_build_s": build_s, "family_ms": {k: round(v[0], 3) for k, v in kms.items()},
           "nodes_per_ray": c["nodes_visited"] / max(rays + c["shadow_rays"], 1)}
    s.close()
    r.close()
    return out


def main():
    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    w, h = a.width, a.height
    config = {"workload": f"{a.workload} ({'hall-250k' if a.workload.startswith('hall') else 'cornell'}, {w}x{h} per GPU, "
                          f"max 8 bounces, Box filter)", "spp_per_step": 1, "frame": f"{w}x{h * max(a.gpus, 1)}",
              "parallelism": f"image strips x{a.gpus}", "l2": "per-step streams (>= 400 MB of rays/hits/frame planes) "
                                                              "exceed the 126 MB L2: no explicit flush"}

    if a.impl == "reference":
        if rank != 0:
            return 0
        base = cpu_reference_run(a.workload, a.cpu_sample, a.steps, a.warmup)
        config = dict(config, spp_per_step=base["spp_per_step"], frame=base["frame"], parallelism=f"{base['cores']} host threads")
        line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": a.gpus,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": base["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import numpy as np
    from ray_b200 import capi, cuda, dist as rdist, host, scenes

    use_dist = world > 1
    if use_dist:
        import torch
        import torch.distributed as tdist
        torch.cuda.set_device(local_rank)
        tdist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n = max(world, 1)
    H = h * n
    desc = make_desc(a.workload, w, H)
    r = host.Renderer(w, H, device=local_rank)
    if a.no_sort:
        r.set_render_flags(capi.RC_RENDER_NO_SORT)
    s = scenes.build(desc, r.create_scene())
    rect = rdist.strip_rect(rank, n, w, H)
    lib = cuda.load_library()
    ctx = r.native_context()
    frame_t = rdist.device_frame_tensor(r, capi.RC_BUF_RAW, local_rank) if use_dist else None
    gather_every = a.gather_every if a.gather_every > 0 else a.steps

    def gather():
        if use_dist:
            x, y, ww, hh = rect
            return rdist.gather_strips(frame_t[y:y + hh], w, H, dst=0)

    it = 0
    for _ in range(max(a.warmup, 0)):
        it = r.render(s, rect, it, 1)
    gather()
    if use_dist:
        torch.cuda.synchronize()
        tdist.barrier()
        torch.cuda.synchronize()
    r.reset_stats()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    # ---- timed region: K steps, device-timed ----
    if use_dist:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    lib.rc_event_record(ctx, 0)
    done = 0
    frame = None
    while done < a.steps:
        k = min(gather_every, a.steps - done)
        it = r.render(s, rect, it, k)  # k samples enqueued back to back, one sync
        done += k
        frame = gather()
    lib.rc_event_record(ctx, 1)
    if use_dist:
        e1.record()
        torch.cuda.synchronize()
        tdist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        tdist.all_reduce(ms, op=tdist.ReduceOp.MAX)
        ms = float(ms.item())
    else:
        import ctypes as C
        f = C.c_float(0)
        lib.rc_event_elapsed_ms(ctx, 0, 1, C.byref(f))
        ms = float(f.value)
    clk = clocks.stop() if rank == 0 else None
    c = r.counters()
    kms = r.kernel_ms()
    rays_local = c["primary_rays"] + c["secondary_rays"]
    launches_local = int(sum(v[1] for v in kms.values()))
    if use_dist:
        t = torch.tensor([rays_local, c["shadow_rays"], launches_local], dtype=torch.float64, device="cuda")
        tdist.all_reduce(t, op=tdist.ReduceOp.SUM)
        rays_total, shadow_total, launches_total = float(t[0]), float(t[1]), int(t[2])
    else:
        rays_total, shadow_total, launches_total = float(rays_local), float(c["shadow_rays"]), launches_local
    value = rays_total / (ms * 1e-3) / 1e6
    if a.dump_outputs and rank == 0:
        if use_dist:
            dump_outputs(a.dump_outputs, {"raw": frame.cpu().numpy()})
        else:
            dump_outputs(a.dump_outputs, {"raw": r.pixels(host.RAW), "final": r.pixels(host.FINAL)})

    # ---- e2e: one blocking public-API call per step + delivery of the frame to the host ----
    # The scene does not change between the samples of a progressive render, so it is uploaded once (timed separately
    # below); a step's host->device input is its pass descriptor.  N > 1: every rank copies ITS strip device->host
    # straight into one shared page-locked host frame (N PCIe links in parallel), then a barrier.
    v = s.view()
    scene_bytes = sum(getattr(v, f).count * getattr(v, f).stride for f in (
        "wnodes", "mtris", "tri_indices", "tri_materials", "materials", "mesh_instances", "vertices", "vtx_indices",
        "lights", "light_cwnodes"))
    ta = time.perf_counter()
    r.invalidate_scene()
    it = r.render(s, rect, it, 1)
    upload_plus_step_ms = 1e3 * (time.perf_counter() - ta)
    e2e_steps = max(min(a.steps, 8), 1)
    shared = rdist.SharedHostFrame(w, H) if use_dist else None
    if not use_dist:
        r.pixels(host.RAW, copy=False)  # warm-up: the first read-back sets up the renderer's page-locked mirror
    else:
        rdist.deliver_strip(r, capi.RC_BUF_RAW, rect, shared)
    r.reset_stats()
    if use_dist:
        torch.cuda.synchronize()
        tdist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        it = r.render(s, rect, it, 1)
        if use_dist:
            rdist.deliver_strip(r, capi.RC_BUF_RAW, rect, shared)
            tdist.barrier()  # the frame is complete on the host once every rank has delivered
        else:
            img = r.pixels(host.RAW, copy=False)  # borrowed view of the pinned mirror, as get_raw_pixels_ref()
    if use_dist:
        torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    c2 = r.counters()
    e2e_rays = c2["primary_rays"] + c2["secondary_rays"]
    if use_dist:
        t = torch.tensor([e2e_rays, e2e_s], dtype=torch.float64, device="cuda")
        tsum = t.clone()
        tdist.all_reduce(tsum, op=tdist.ReduceOp.SUM)
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        e2e_rays, e2e_s = float(tsum[0]), float(t[1])
    e2e_value = e2e_rays / e2e_s / 1e6
    d2h = w * H * 16  # the whole frame reaches the host every step (N strips over N links)

    bvh_nodes = s.node_count()
    strong = None
    if use_dist:
        # strong scaling: the SAME 1920x1080 frame split into N strips (config #4 read literally), device-timed
        shared.close()
        s.close()
        r.close()
        desc2 = make_desc(a.workload, w, h)
        r2 = host.Renderer(w, h, device=local_rank)
        s2 = scenes.build(desc2, r2.create_scene())
        rect2 = rdist.strip_rect(rank, n, w, h)
        it2 = 0
        for _ in range(3):
            it2 = r2.render(s2, rect2, it2, 1)
        torch.cuda.synchronize()
        tdist.barrier()
        r2.reset_stats()
        k = max(min(a.steps, 8), 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        it2 = r2.render(s2, rect2, it2, k)
        wall = time.perf_counter() - t0
        e1.record()
        torch.cuda.synchronize()
        c3 = r2.counters()
        t = torch.tensor([c3["primary_rays"] + c3["secondary_rays"], wall], dtype=torch.float64, device="cuda")
        tsum = t.clone()
        tdist.all_reduce(tsum, op=tdist.ReduceOp.SUM)
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        strong = {"frame": f"{w}x{h}", "steps": k, "value": float(tsum[0]) / float(t[1]) / 1e6, "unit": UNIT,
                  "ms_per_step": float(t[1]) / k * 1e3,
                  "note": "fixed frame split into N row strips, k samples enqueued back to back per rank, max over ranks "
                          "of the blocking call's wall time"}
        s2.close()
        r2.close()
    if rank != 0:
        if use_dist:
            tdist.destroy_process_group()
        return 0

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 256,
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "scene_bytes_uploaded_once": int(scene_bytes),
                    "scene_upload_plus_one_step_ms": upload_plus_step_ms,
                    "pinned_shared_frame": (shared.pinned if shared else True),
                    "one_shared_host_frame": (bool(getattr(shared, "shared", True)) if shared else True),
                    "note": "per step: one blocking RenderScene (pass descriptor host->device) + the whole frame "
                            "device->host into page-locked memory (1 GPU: the renderer's mirror, as get_raw_pixels_ref; "
                            "N GPUs: every rank copies its strip into one shared host frame, then a barrier); the "
                            "unchanged scene is not re-uploaded (one upload + step timed separately)"},
            "gpu_launches": launches_total, "clocks": clk,
            "rays": {"per_step": rays_total / a.steps, "shadow_per_step": shadow_total / a.steps,
                     "Mshadow_per_s": shadow_total / (ms * 1e-3) / 1e6},
            "scene": {"triangles": desc.triangle_count(), "bvh8_nodes": bvh_nodes, "scene_bytes": int(scene_bytes)},
            "roofline": roofline(c, kms, a.steps)}
    if strong:
        line["strong_scaling"] = strong
    if a.gpus == 1 and not a.no_extra_configs and a.workload == "hall-diffuse":
        # the other single-GPU configurations of BASELINE.json, measured in the same run (bounded steps each)
        extra = {}
        for key, wl, ww, hh, st, wu in (("config1_cornell_256x256_64spp", "cornell", 256, 256, 64, 3),
                                        ("config3_hall_principled_1080p", "hall-principled", 1920, 1080, 8, 3),
                                        ("config5_instanced_10M_4096x4096", "c5-instanced", 4096, 4096, 4, 3)):
            try:
                extra[key] = measure_config(wl, ww, hh, st, wu, local_rank)
            except Exception as e:
                extra[key] = {"error": str(e)}
        if not a.no_cpu_baseline:
            try:
                extra["config1_cornell_256x256_64spp"]["cpu_baseline"] = cpu_single_thread_ref("cornell", 256, 256, 8)
            except Exception as e:
                extra["config1_cornell_256x256_64spp"]["cpu_baseline"] = {"error": str(e)}
        line["configs"] = extra
    if not a.no_cpu_baseline and a.gpus == 1:
        try:
            base = cpu_reference_run(a.workload, a.cpu_sample, 2, 1)
            line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "host")}
        except Exception as e:  # the oracle is test infrastructure: its absence must not hide the GPU number
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": host_cores()["threads"], "kind": "reference",
                                    "sample": f"unavailable: {e}"}
    print(json.dumps(line))
    if use_dist:
        tdist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
