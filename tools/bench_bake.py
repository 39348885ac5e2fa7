"""Lightmap-baking benchmark: the floor of hall-250k (131,072 triangles, uv = its [0,1]^2 grid) as its own mesh and
instance, baked at 2048^2 with the Geo camera of include/ray_cuda.h.  Prints one JSON line:

  card / power_limit_w        what the numbers were measured on
  bake                        ms per sample and Mrays/s (primary + secondary + shadow rays), all flags off
  bake_indirect               the same with SKIP_DIRECT | LIGHTING_ONLY (the usual indirect-lighting bake)
  sh_overhead_ms              ms per sample with OUTPUT_SH on minus off
  list_build_ms               building the per-texel candidate lists: a blocking Geo pass right after the lists were
                              dropped (scene re-upload) minus a blocking pass that reuses them, both with warm kernels
  raygen_geo_ms / replaced_ms k_raygen_geo per sample next to k_raygen + the primary closest-hit trace of a
                              perspective render of the same scene with the same pixel count, the work it replaces

    python tools/bench_bake.py [--size 2048] [--steps 16] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from ray_b200 import capi, cuda, host, scenes  # noqa: E402


def split_floor(desc):
    """hall(): one mesh whose first material group is the floor grid -> floor as mesh 0 / instance 0, the rest as
    mesh 1 / instance 1 (same vertices, same materials)."""
    m = desc.meshes[0]
    front, back, first, n_idx = m.groups[0]
    assert first == 0
    floor = scenes.MeshDesc(m.attrs, m.indices[:n_idx].copy(), [(front, back, 0, n_idx)])
    rest = scenes.MeshDesc(m.attrs, m.indices[n_idx:].copy(), [(f, b, s - n_idx, c) for f, b, s, c in m.groups[1:]])
    desc.meshes = [floor, rest]
    desc.instances = [(0, scenes.IDENTITY.T.reshape(16), {}), (1, scenes.IDENTITY.T.reshape(16), {})]
    return n_idx // 3


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits",
                                       "-i", "0"], text=True).strip().split(", ")
        return out[0], float(out[1])
    except Exception:
        return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    n = a.size
    desc = scenes.hall("diffuse", n, n)
    floor_tris = split_floor(desc)
    hs = scenes.build(desc, host.Scene(None))
    ctx = cuda.Context(0)
    ctx.resize(n, n)
    ctx.upload_tables(host.builtin_sampler_table())
    view = hs.view()
    ctx.upload_scene(view)
    persp = hs.camera()
    geo_cam = capi.rc_camera.from_buffer_copy(persp)
    geo_cam.type = capi.CAM_GEO
    geo_cam.filter = capi.FILTER_BOX
    persp.filter = capi.FILTER_BOX
    geo = (0, 0, floor_tris)

    def run(cam, flags, steps, warmup):
        ctx.clear()
        it = 0
        for _ in range(warmup):
            it += 1
            ctx.render(ctx.make_pass(cam, (0, 0, n, n), it, flags, geo))
        ctx.reset_stats()
        t0 = time.perf_counter()
        for _ in range(steps):
            it += 1
            ctx.render(ctx.make_pass(cam, (0, 0, n, n), it, flags | capi.RC_RENDER_ASYNC, geo))
        ctx.sync()
        ms = (time.perf_counter() - t0) * 1e3 / steps
        c = ctx.counters()
        rays = c["primary_rays"] + c["secondary_rays"] + c["shadow_rays"]
        return {"ms_per_sample": ms, "Mrays_per_s": rays / (ms * steps * 1e-3) / 1e6,
                "primary_rays_per_sample": c["primary_rays"] / steps}, ctx.stats_us(), ctx.kernel_ms()

    bake, us_geo, _ = run(geo_cam, 0, a.steps, a.warmup)

    def blocking_pass_ms(reupload):
        if reupload:  # a scene upload drops the candidate lists: the next Geo pass rebuilds them
            ctx.upload_scene(view)
        ctx.clear()
        t0 = time.perf_counter()
        ctx.render(ctx.make_pass(geo_cam, (0, 0, n, n), 1, 0, geo))
        return (time.perf_counter() - t0) * 1e3

    rebuild = float(np.median([blocking_pass_ms(True) for _ in range(5)]))
    reuse = float(np.median([blocking_pass_ms(False) for _ in range(5)]))
    bake_ind, _, _ = run(geo_cam, capi.RC_RENDER_SKIP_DIRECT | capi.RC_RENDER_LIGHTING_ONLY, a.steps, a.warmup)
    bake_sh, _, _ = run(geo_cam, capi.RC_RENDER_OUTPUT_SH, a.steps, a.warmup)
    _, us_persp, _ = run(persp, 0, a.steps, a.warmup)
    name, power = card()
    line = {"workload": f"hall-250k floor bake {n}x{n}", "floor_triangles": floor_tris, "card": name,
            "power_limit_w": power, "steps": a.steps, "warmup": a.warmup,
            "bake": bake, "bake_indirect": bake_ind,
            "sh_overhead_ms": bake_sh["ms_per_sample"] - bake["ms_per_sample"],
            "list_build_ms": rebuild - reuse,
            # stats_t: [0] primary ray generation, [1] primary trace (device events, us over the timed steps)
            "raygen_geo_ms": us_geo[0] / 1e3 / a.steps,
            "replaced_ms": (us_persp[0] + us_persp[1]) / 1e3 / a.steps,
            "persp_raygen_ms": us_persp[0] / 1e3 / a.steps, "persp_primary_trace_ms": us_persp[1] / 1e3 / a.steps}
    print(json.dumps(line))
    ctx.close()
    hs.close()


if __name__ == "__main__":
    main()
