"""Shared helpers of the parity tests: build one scene description into both the oracle and the CUDA context, or, where
the oracle library is not built, into the CUDA context alone with results checked against stored digests."""
import atexit
import hashlib
import json
import os

import numpy as np

from ray_b200 import capi, cuda, scenes

DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cuda_digests.json")


def maybe_oracle():
    """The oracle module when its library (built from the reference's sources) is present, else None."""
    import oracle
    return oracle if oracle.available() else None


class Stored:
    """What the CUDA path computed for the parity cases when the oracle library is absent, stored as SHA-256 digests of
    the output bytes (tests/golden/cuda_digests.json): the check is bitwise, and the whole set of cases fits in a few KB.
    They pin what the CUDA path computed when they were recorded; where the oracle library is present the same tests
    compare with the reference instead.  `RAY_B200_STORE_DIGESTS=<file> python -m pytest -m gpu tests` on a B200
    records them into <file> instead of checking (a key met twice in one run must give the same digest)."""

    def __init__(self):
        self.data = json.load(open(DIGESTS)) if os.path.exists(DIGESTS) else {}
        self.out = os.environ.get("RAY_B200_STORE_DIGESTS")
        if self.out:
            self.data = {}
            atexit.register(lambda: json.dump(self.data, open(self.out, "w"), indent=0, sort_keys=True))

    def check(self, key, *arrays):
        h = hashlib.sha256()
        for a in arrays:
            h.update(np.ascontiguousarray(a).tobytes())
        d = h.hexdigest()
        if self.out and key not in self.data:
            self.data[key] = d
        assert key in self.data, f"no stored result for {key}"
        assert self.data[key] == d, f"{key}: the CUDA path no longer computes the stored result"


STORED = Stored()


class HostPair:
    """The scene built by the product's host layer (no reference library) in a CUDA context with the built-in sampler
    and filter tables; the stand-in for Pair where the oracle is absent (`osc` is None)."""

    def __init__(self, desc, device=0):
        from ray_b200 import host
        self.desc = desc
        self.w, self.h = desc.width, desc.height
        self.osc = None
        self.hs = scenes.build(desc, host.Scene(None))
        self.cam = self.hs.camera()
        self.ctx = cuda.Context(device)
        self.ctx.resize(self.w, self.h)
        ft = host.builtin_filter_table(self.cam.filter, desc.camera.filter_width) \
            if self.cam.filter != capi.FILTER_BOX else None
        self.ctx.upload_tables(host.builtin_sampler_table(), ft)
        self.view = self.hs.view()
        self.ctx.upload_scene(self.view)

    def make_pass(self, iteration, rect=None, flags=0):
        return self.ctx.make_pass(self.cam, rect or (0, 0, self.w, self.h), iteration, flags)

    def close(self):
        self.ctx.close()
        self.hs.close()


def make_pair(desc, device=0, tex_compression=False):
    """Pair when the oracle library is present, HostPair otherwise."""
    o = maybe_oracle()
    return Pair(o, desc, device, tex_compression) if o else HostPair(desc, device)


class Pair:
    """Oracle scene (reference Cpu::Scene, wide BVH) + CUDA context holding byte-identical arrays (oracle mode 1b)."""

    def __init__(self, oracle, desc, device=0, tex_compression=False):
        self.oracle = oracle
        self.desc = desc
        self.w, self.h = desc.width, desc.height
        self.osc = scenes.build(desc, oracle.Scene(wide=True, tex_compression=tex_compression))
        self.cam = self.osc.camera()
        self.ctx = cuda.Context(device)
        self.ctx.resize(self.w, self.h)
        ft = self.osc.filter_table() if self.cam.filter != capi.FILTER_BOX else None
        self.ctx.upload_tables(oracle.pmj_table(), ft)
        self.view = self.osc.view()
        self.ctx.upload_scene(self.view)

    def make_pass(self, iteration, rect=None, flags=0):
        return self.ctx.make_pass(self.cam, rect or (0, 0, self.w, self.h), iteration, flags)

    def close(self):
        self.ctx.close()
        self.osc.close()


GOLDEN_ARRAYS = ["wnodes", "mtris", "tri_indices", "tri_materials", "materials", "mesh_instances", "vertices",
                 "vtx_indices", "lights", "li_indices", "light_cwnodes"]


def view_from_golden(g, keep):
    """rc_scene_view over the reference-built scene arrays stored in a tests/golden/*.npz fixture; `keep` holds the
    buffers alive for as long as the view is used."""
    v = capi.rc_scene_view()
    for name in GOLDEN_ARRAYS:
        buf = np.ascontiguousarray(g["arr_" + name])
        keep.append(buf)
        stride = int(g["stride_" + name])
        a = capi.rc_array(buf.ctypes.data if buf.size else None, buf.size // stride if stride else 0, stride)
        setattr(v, name, a)
    for name in ("tlas_root", "visible_lights_count", "blocker_lights_count", "env_map", "back_map", "env_light_index"):
        setattr(v, name, int(g["s_" + name]))
    v.sky_map_spread_angle = float(g["s_sky_map_spread_angle"])
    for name in ("env_col", "back_col", "bounds_min", "bounds_max"):
        arr = getattr(v, name)
        for i, x in enumerate(g["s_" + name]):
            arr[i] = float(x)
    return v


def golden_context(g, keep, device=0):
    """A CUDA context holding a fixture's scene, its reference filter table and the host layer's built-in sampler
    table (the reference's PMJ02 table is not part of the fixtures); returns (context, camera)."""
    from ray_b200 import host
    w, h = [int(x) for x in g["wh"]]
    ctx = cuda.Context(device)
    ctx.resize(w, h)
    ctx.upload_tables(host.builtin_sampler_table(), g["filter_table"])
    ctx.upload_scene(view_from_golden(g, keep))
    return ctx, capi.rc_camera.from_buffer_copy(g["cam"].tobytes())


def render_golden(g, spp):
    """`spp` samples of rc_render over a fixture's scene; returns the linear and the tonemapped planes and the counters."""
    keep = []
    ctx, cam = golden_context(g, keep)
    ctx.clear((0, 0, 0, 0))
    for i in range(1, spp + 1):
        ctx.render(ctx.make_pass(cam, (0, 0, ctx.w, ctx.h), i))
    out = {"raw": ctx.readback(capi.RC_BUF_RAW), "final": ctx.readback(capi.RC_BUF_FINAL)}
    counters = ctx.counters()
    ctx.close()
    return out, counters


def by_xy(a):
    """Sort a ray / shadow-ray record array by its pixel key (one record per pixel per stage)."""
    order = np.argsort(a["xy"], kind="stable")
    return a[order]


def bits_equal(a, b):
    """Exact (bitwise) equality of two structured / float arrays, NaNs included."""
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def field_mismatch(a, b):
    """Per-field count of records that differ bitwise (diagnostics)."""
    out = {}
    for name in a.dtype.names:
        x = np.ascontiguousarray(a[name]).view(np.uint8).reshape(len(a), -1)
        y = np.ascontiguousarray(b[name]).view(np.uint8).reshape(len(b), -1)
        n = int((x != y).any(axis=1).sum())
        if n:
            out[name] = n
    return out
