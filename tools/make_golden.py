"""Generate tests/golden/*.npz from the oracle (the unmodified reference, oracle/_ref).  Run here, commit the output.

Each fixture holds (a) the byte-exact scene arrays of the reference's own Cpu::Scene (wide BVH) for a small scene, in the
layouts rc_upload_scene takes, (b) inputs and the reference's outputs of the hot-path stages:
  primary rays (Ref::GeneratePrimaryRays)           -> hits (Ref::TraceRays, closest hit)
  secondary rays of bounce 1 (Ref::ShadePrimary)    -> hits (Ref::TraceRays with IntersectAreaLights)
  shadow rays of the primary shade                  -> radiance buffer after Ref::TraceShadowRays
  a 4-spp linear image of Ref's whole RenderScene   (needs the reference's PMJ02 table, so the GPU test that uses it is
                                                     skipped when the oracle library is absent)
tests/test_golden.py checks the oracle against these (CPU, pins the oracle build) and the CUDA path against them (GPU).

    python tools/make_golden.py --cuda-images OUT.npz   (on a B200; no oracle needed)
stores what the CUDA path renders (tests/golden/cuda_images.npz): the fixture scenes over their stored arrays and the
host-layer cases of tests/test_golden.py, so that every later change to the device or host code is checked against them.
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from ray_b200 import capi, scenes  # noqa: E402
import oracle  # noqa: E402

ARRAYS = ["wnodes", "mtris", "tri_indices", "tri_materials", "materials", "mesh_instances", "vertices", "vtx_indices",
          "lights", "li_indices", "light_cwnodes"]
SCALARS = ["tlas_root", "visible_lights_count", "blocker_lights_count", "env_map", "back_map", "env_light_index",
           "sky_map_spread_angle"]


def view_to_dict(v):
    out = {}
    for name in ARRAYS:
        a = getattr(v, name)
        nbytes = a.count * a.stride
        buf = np.ctypeslib.as_array(C.cast(a.ptr, C.POINTER(C.c_uint8)), shape=(nbytes,)).copy() if nbytes else \
            np.zeros(0, np.uint8)
        out["arr_" + name] = buf
        out["stride_" + name] = np.uint32(a.stride)
    for name in SCALARS:
        out["s_" + name] = np.asarray(getattr(v, name))
    for name in ("env_col", "back_col", "bounds_min", "bounds_max"):
        out["s_" + name] = np.asarray(list(getattr(v, name)), np.float32)
    return out


def make(name, desc, iteration=2, spp=4):
    w, h = desc.width, desc.height
    sc = scenes.build(desc, oracle.Scene(wide=True))
    cam = sc.camera()
    d = view_to_dict(sc.view())
    d["cam"] = np.frombuffer(bytes(cam), np.uint8).copy()
    d["wh"] = np.asarray([w, h], np.int32)
    d["filter_table"] = sc.filter_table()  # reference UpdateFilterTable output for cam.filter / cam.fwidth
    d["iteration"] = np.int32(iteration)
    rays, hits = sc.generate_primary_rays(w, h, (0, 0, w, h), iteration)
    d["primary_rays"], d["primary_hits_in"] = rays, hits
    rays1, hits1 = sc.trace_rays(iteration, rays, hits, False)
    d["primary_hits_out"] = hits1
    temp = np.zeros((h, w, 4), np.float32)
    sec, sh, base, dn = sc.shade(w, h, iteration, True, 0, rays1, hits1, temp)
    d["secondary_rays"], d["shadow_rays"] = sec, sh
    d["temp_after_primary_shade"] = temp.copy()
    sc.trace_shadow_rays(w, iteration, sh, cam.clamp_direct, temp)
    d["temp_after_primary_shadow"] = temp.copy()
    hits0 = np.zeros(len(sec), dtype=hits.dtype)
    hits0["obj_index"] = -1
    hits0["prim_index"] = -1
    hits0["t"] = np.float32(3.402823466e+30)
    hits0["v"] = -1.0
    _, hits2 = sc.trace_rays(iteration, sec, hits0, True)
    d["secondary_hits_out"] = hits2
    ref = oracle.Renderer(capi.RT_REFERENCE, w, h)
    it = 0
    for _ in range(spp):
        it = ref.render(sc, (0, 0, w, h), it)
    d["image_raw_4spp"] = ref.pixels(1)
    out = os.path.join(ROOT, "tests", "golden", name + ".npz")
    np.savez_compressed(out, **d)
    print(name, os.path.getsize(out) // 1024, "KiB", "rays", len(rays), "sec", len(sec), "shadow", len(sh))


def cuda_images(out):
    from common import render_golden
    from test_golden import GOLDEN, GOLDEN_SPP, HOST_CASES, render_host_case
    d = {}
    for path in GOLDEN:
        name = os.path.splitext(os.path.basename(path))[0]
        planes, _ = render_golden(np.load(path), GOLDEN_SPP)
        d.update({f"{name}_{k}": v for k, v in planes.items()})
    for name in HOST_CASES:
        planes, _, _ = render_host_case(name)
        d.update({f"{name}_{k}": v for k, v in planes.items()})
    np.savez_compressed(out, **d)
    print(out, os.path.getsize(out) // 1024, "KiB", sorted(d))


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--cuda-images":
        cuda_images(sys.argv[2])
    else:
        make("cornell_48", scenes.cornell_box(48, 48))
        make("zoo_64x48", scenes.material_zoo(64, 48))
