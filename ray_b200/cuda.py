"""ctypes binding of libray_cuda.so (include/ray_cuda.h) -- the product's device path.

There is no fallback: if the shared library is missing, or no sm_100 device is present, constructing a Context raises.
"""
import ctypes as C
import os

import numpy as np

from . import capi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libray_cuda.so")

RAY_DTYPE = np.dtype([("o", "<f4", 3), ("d", "<f4", 3), ("pdf", "<f4"), ("c", "<f4", 3), ("ior", "<f4", 4),
                      ("cone_width", "<f4"), ("cone_spread", "<f4"), ("xy", "<u4"), ("depth", "<u4")])
HIT_DTYPE = np.dtype([("obj_index", "<i4"), ("prim_index", "<i4"), ("t", "<f4"), ("u", "<f4"), ("v", "<f4")])
SHADOW_DTYPE = np.dtype([("o", "<f4", 3), ("depth", "<u4"), ("d", "<f4", 3), ("dist", "<f4"), ("c", "<f4", 3),
                         ("xy", "<u4")])
assert RAY_DTYPE.itemsize == 72 and HIT_DTYPE.itemsize == 20 and SHADOW_DTYPE.itemsize == 48

_lib = None


def load_library():
    """Load libray_cuda.so (built by __graft_entry__.build()). Raises if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for the CUDA backend)")
    lib = C.CDLL(LIB_PATH)
    P = C.POINTER
    vp = C.c_void_p
    sig = {
        "rc_device_count": (C.c_int, []),
        "rc_create": (C.c_int, [C.c_int, P(vp)]),
        "rc_destroy": (None, [vp]),
        "rc_last_error": (C.c_char_p, [vp]),
        "rc_device_name": (C.c_char_p, [vp]),
        "rc_resize": (C.c_int, [vp, C.c_int, C.c_int]),
        "rc_clear": (C.c_int, [vp, P(C.c_float)]),
        "rc_upload_tables": (C.c_int, [vp, vp, C.c_int, C.c_int, vp, C.c_int]),
        "rc_upload_scene": (C.c_int, [vp, P(capi.rc_scene_view)]),
        "rc_render": (C.c_int, [vp, P(capi.rc_pass_desc)]),
        "rc_denoise_nlm": (C.c_int, [vp, P(capi.rc_rect), C.c_int]),
        "rc_sync": (C.c_int, [vp]),
        "rc_readback": (C.c_int, [vp, C.c_int, P(capi.rc_rect), vp, C.c_int]),
        "rc_readback_required_samples": (C.c_int, [vp, vp]),
        "rc_enable_stats": (C.c_int, [vp, C.c_int]),
        "rc_get_stats": (C.c_int, [vp, P(C.c_uint64)]),
        "rc_get_counters": (C.c_int, [vp, P(capi.rc_counters)]),
        "rc_reset_stats": (C.c_int, [vp]),
        "rc_get_kernel_ms": (C.c_int, [vp, P(C.c_double), P(C.c_uint64)]),
        "rc_stage_generate_primary_rays": (C.c_int, [vp, P(capi.rc_pass_desc), vp, vp, P(C.c_int)]),
        "rc_stage_generate_geo_rays": (C.c_int, [vp, P(capi.rc_pass_desc), vp, vp, P(C.c_int)]),
        "rc_stage_trace_rays": (C.c_int, [vp, P(capi.rc_pass_desc), vp, vp, C.c_int, C.c_int]),
        "rc_stage_shade": (C.c_int, [vp, P(capi.rc_pass_desc), C.c_int, C.c_int, vp, vp, C.c_int, vp, P(C.c_int), vp,
                                     P(C.c_int)]),
        "rc_stage_trace_shadow_rays": (C.c_int, [vp, P(capi.rc_pass_desc), vp, C.c_int, C.c_float]),
        "rc_stage_sort_rays": (C.c_int, [vp, vp, C.c_int, vp]),
        "rc_debug_fill_temp": (C.c_int, [vp, P(C.c_float)]),
        "rc_debug_write_plane": (C.c_int, [vp, C.c_int, vp]),
        "rc_debug_unet_tensor": (C.c_int, [vp, C.c_uint32, C.c_int, C.c_int, C.c_int, vp, P(C.c_int32)]),
        "rc_abi_sizeof": (C.c_int, [C.c_int]),
        "rc_host_alloc": (vp, [C.c_size_t]),
        "rc_host_free": (None, [vp]),
        "rc_device_ptr": (vp, [vp, C.c_int]),
        "rc_event_record": (C.c_int, [vp, C.c_int]),
        "rc_event_elapsed_ms": (C.c_int, [vp, C.c_int, C.c_int, P(C.c_float)]),
        "rc_readback_async": (C.c_int, [vp, C.c_int, P(capi.rc_rect), vp, C.c_int]),
        "rc_unet_set_weights": (C.c_int, [vp, vp]),
        "rc_build_lbvh": (C.c_int, [vp, vp, C.c_uint32, vp, vp]),
        "rc_update_instances": (C.c_int, [vp, vp, C.c_uint32]),
        "rc_scene_upload_bytes": (C.c_uint64, [vp]),
        "rc_set_view_lut": (C.c_int, [vp, C.c_uint32, vp, C.c_int]),
        "rc_denoise_unet": (C.c_int, [vp, C.c_int, P(capi.rc_rect), C.c_uint32]),
        "rc_comm_init": (C.c_int, [P(vp), C.c_int, P(vp)]),
        "rc_comm_destroy": (None, [vp]),
        "rc_comm_last_error": (C.c_char_p, [vp]),
        "rc_comm_strip": (C.c_int, [P(capi.rc_rect), C.c_int, C.c_int, P(capi.rc_rect)]),
        "rc_comm_upload_scene": (C.c_int, [vp, P(capi.rc_scene_view)]),
        "rc_comm_upload_tables": (C.c_int, [vp, vp, C.c_int, C.c_int, vp, C.c_int]),
        "rc_comm_render": (C.c_int, [vp, P(capi.rc_pass_desc)]),
        "rc_comm_sync": (C.c_int, [vp]),
        "rc_gather": (C.c_int, [vp, C.c_int, P(capi.rc_rect), vp, C.c_int]),
        "rc_gather_device": (C.c_int, [vp, C.c_int, P(capi.rc_rect)]),
        "rc_comm_get_counters": (C.c_int, [vp, P(capi.rc_counters)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError here = the library does not export what include/ray_cuda.h declares
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


EXPORTED_SYMBOLS = [
    "rc_device_count", "rc_create", "rc_destroy", "rc_last_error", "rc_device_name", "rc_resize", "rc_clear",
    "rc_upload_tables", "rc_upload_scene", "rc_render", "rc_denoise_nlm", "rc_sync", "rc_readback", "rc_readback_required_samples",
    "rc_enable_stats", "rc_get_stats", "rc_get_counters", "rc_reset_stats", "rc_get_kernel_ms",
    "rc_stage_generate_primary_rays", "rc_stage_generate_geo_rays", "rc_stage_trace_rays", "rc_stage_shade", "rc_stage_trace_shadow_rays",
    "rc_stage_sort_rays", "rc_debug_fill_temp", "rc_debug_write_plane", "rc_debug_unet_tensor", "rc_abi_sizeof", "rc_host_alloc", "rc_host_free", "rc_device_ptr",
    "rc_event_record", "rc_event_elapsed_ms", "rc_readback_async", "rc_comm_init", "rc_comm_destroy", "rc_comm_last_error",
    "rc_comm_strip", "rc_comm_upload_scene", "rc_comm_upload_tables", "rc_comm_render", "rc_comm_sync", "rc_gather",
    "rc_gather_device", "rc_comm_get_counters", "rc_unet_set_weights", "rc_denoise_unet", "rc_build_lbvh", "rc_update_instances", "rc_scene_upload_bytes", "rc_set_view_lut",
]


class CudaError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """Thin object wrapper over rc_ctx. One per device."""

    def __init__(self, device=0):
        self.lib = load_library()
        self._ctx = C.c_void_p()
        rc = self.lib.rc_create(device, C.byref(self._ctx))
        if rc != 0:
            self._ctx = None
            raise CudaError(f"rc_create(device={device}) failed with code {rc} (no sm_100 CUDA device?)")
        self.w = self.h = 0

    def close(self):
        if getattr(self, "_ctx", None):
            self.lib.rc_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise CudaError(f"{what}: {self.lib.rc_last_error(self._ctx).decode()}")

    @property
    def device_name(self):
        return self.lib.rc_device_name(self._ctx).decode()

    def resize(self, w, h):
        self._check(self.lib.rc_resize(self._ctx, w, h), "rc_resize")
        self.w, self.h = w, h

    def clear(self, rgba=(0, 0, 0, 0)):
        arr = (C.c_float * 4)(*rgba)
        self._check(self.lib.rc_clear(self._ctx, arr), "rc_clear")

    def upload_tables(self, pmj, filter_table=None):
        pmj = np.ascontiguousarray(pmj, dtype=np.uint32)
        ft = None if filter_table is None else np.ascontiguousarray(filter_table, dtype=np.float32)
        self._check(self.lib.rc_upload_tables(self._ctx, _ptr(pmj), 32, 4096, None if ft is None else _ptr(ft),
                                              0 if ft is None else len(ft)), "rc_upload_tables")

    def upload_scene(self, view: capi.rc_scene_view):
        self._check(self.lib.rc_upload_scene(self._ctx, C.byref(view)), "rc_upload_scene")

    def update_instances(self, view: capi.rc_scene_view, first_tlas_node):
        self._check(self.lib.rc_update_instances(self._ctx, C.byref(view), first_tlas_node), "rc_update_instances")

    def set_view_lut(self, view_transform, lut):
        """lut: 48^3 uint32 (packed 10-10-10-2) or None"""
        if lut is None:
            self._check(self.lib.rc_set_view_lut(self._ctx, view_transform, None, 48), "rc_set_view_lut")
            return
        lut = np.ascontiguousarray(lut, dtype=np.uint32)
        assert lut.size == 48 ** 3
        self._check(self.lib.rc_set_view_lut(self._ctx, view_transform, lut.ctypes.data, 48), "rc_set_view_lut")

    def scene_upload_bytes(self):
        return int(self.lib.rc_scene_upload_bytes(self._ctx))

    def make_pass(self, cam: capi.rc_camera, rect, iteration, flags=0, geo=None):
        """geo = (instance, tri_first, tri_count): the mesh instance a Geo camera (cam.type == CAM_GEO) bakes."""
        p = capi.rc_pass_desc()
        p.cam = cam
        p.rect = capi.rc_rect(*rect)
        p.iteration = iteration
        p.flags = flags
        if geo is not None:
            p.geo_instance, p.geo_tri_first, p.geo_tri_count = (int(x) for x in geo)
        return p

    def render(self, p: capi.rc_pass_desc):
        self._check(self.lib.rc_render(self._ctx, C.byref(p)), "rc_render")

    def unet_set_weights(self, layers):
        """layers: 16 x (weights fp16 ndarray [cout, cin, 3, 3], bias fp16 ndarray [cout]) in pass order"""
        class L(C.Structure):
            _fields_ = [("weights", C.c_void_p), ("bias", C.c_void_p), ("cin", C.c_int32), ("cout", C.c_int32)]
        arr = (L * 16)()
        keep = []
        for i, (w, b) in enumerate(layers):
            w = np.ascontiguousarray(w, dtype=np.float16)
            b = np.ascontiguousarray(b, dtype=np.float16)
            keep += [w, b]
            arr[i] = L(w.ctypes.data, b.ctypes.data, w.shape[1], w.shape[0])
        self._check(self.lib.rc_unet_set_weights(self._ctx, C.byref(arr)), "rc_unet_set_weights")

    def denoise_unet(self, rect, flags=0, pass_index=-1):
        r = capi.rc_rect(*rect)
        self._check(self.lib.rc_denoise_unet(self._ctx, pass_index, C.byref(r), flags), "rc_denoise_unet")

    LBVH_NODE = np.dtype([("mn", "<f4", 3), ("mx", "<f4", 3), ("left", "<u4"), ("right", "<u4"), ("first", "<u4"),
                          ("count", "<u4")])

    def build_lbvh(self, boxes):
        """boxes: (n, 6) float32 {min xyz, max xyz}.  Returns (nodes[2n-1] of LBVH_NODE, order[n])."""
        boxes = np.ascontiguousarray(boxes, dtype=np.float32)
        n = boxes.shape[0]
        nodes = np.zeros(2 * n - 1, dtype=self.LBVH_NODE)
        order = np.zeros(n, dtype=np.uint32)
        self._check(self.lib.rc_build_lbvh(self._ctx, boxes.ctypes.data, n, nodes.ctypes.data, order.ctypes.data),
                    "rc_build_lbvh")
        return nodes, order

    def denoise_nlm(self, rect, iteration):
        r = capi.rc_rect(*rect)
        self._check(self.lib.rc_denoise_nlm(self._ctx, C.byref(r), int(iteration)), "rc_denoise_nlm")

    def sync(self):
        self._check(self.lib.rc_sync(self._ctx), "rc_sync")

    def readback(self, which, rect=None):
        rect = rect or (0, 0, self.w, self.h)
        r = capi.rc_rect(*rect)
        out = np.empty((r.h, r.w, 4), dtype=np.float32)
        self._check(self.lib.rc_readback(self._ctx, which, C.byref(r), _ptr(out), r.w), "rc_readback")
        return out

    def required_samples(self):
        out = np.empty((self.h, self.w), dtype=np.uint16)
        self._check(self.lib.rc_readback_required_samples(self._ctx, _ptr(out)), "rc_readback_required_samples")
        return out

    def enable_stats(self, on=True):
        self._check(self.lib.rc_enable_stats(self._ctx, 1 if on else 0), "rc_enable_stats")

    def stats_us(self):
        a = (C.c_uint64 * 11)()
        self._check(self.lib.rc_get_stats(self._ctx, a), "rc_get_stats")
        return list(a)

    def counters(self):
        c = capi.rc_counters()
        self._check(self.lib.rc_get_counters(self._ctx, C.byref(c)), "rc_get_counters")
        return {k: getattr(c, k) for k, _ in capi.rc_counters._fields_}

    def reset_stats(self):
        self._check(self.lib.rc_reset_stats(self._ctx), "rc_reset_stats")

    def kernel_ms(self):
        ms = (C.c_double * 6)()
        n = (C.c_uint64 * 6)()
        self._check(self.lib.rc_get_kernel_ms(self._ctx, ms, n), "rc_get_kernel_ms")
        names = ["raygen", "trace_closest", "shade", "trace_shadow", "sort", "resolve"]
        return {k: (ms[i], n[i]) for i, k in enumerate(names)}

    # ---- stage entry points ----
    def stage_generate_primary_rays(self, p):
        n = p.rect.w * p.rect.h
        rays = np.zeros(n, dtype=RAY_DTYPE)
        hits = np.zeros(n, dtype=HIT_DTYPE)
        cnt = C.c_int(0)
        self._check(self.lib.rc_stage_generate_primary_rays(self._ctx, C.byref(p), _ptr(rays), _ptr(hits),
                                                            C.byref(cnt)), "rc_stage_generate_primary_rays")
        return rays[:cnt.value], hits[:cnt.value]

    def stage_generate_geo_rays(self, p):
        n = p.rect.w * p.rect.h
        rays = np.zeros(n, dtype=RAY_DTYPE)
        hits = np.zeros(n, dtype=HIT_DTYPE)
        cnt = C.c_int(0)
        self._check(self.lib.rc_stage_generate_geo_rays(self._ctx, C.byref(p), _ptr(rays), _ptr(hits), C.byref(cnt)),
                    "rc_stage_generate_geo_rays")
        return rays[:cnt.value], hits[:cnt.value]

    def stage_trace_rays(self, p, rays, hits, trace_lights):
        rays = np.ascontiguousarray(rays.copy())
        hits = np.ascontiguousarray(hits.copy())
        self._check(self.lib.rc_stage_trace_rays(self._ctx, C.byref(p), _ptr(rays), _ptr(hits), len(rays),
                                                 1 if trace_lights else 0), "rc_stage_trace_rays")
        return rays, hits

    def stage_shade(self, p, primary, bounce, rays, hits):
        rays = np.ascontiguousarray(rays)
        hits = np.ascontiguousarray(hits)
        n = len(rays)
        sec = np.zeros(max(n, 1), dtype=RAY_DTYPE)
        sh = np.zeros(max(n, 1), dtype=SHADOW_DTYPE)
        ns, nh = C.c_int(0), C.c_int(0)
        self._check(self.lib.rc_stage_shade(self._ctx, C.byref(p), 1 if primary else 0, bounce, _ptr(rays), _ptr(hits),
                                            n, _ptr(sec), C.byref(ns), _ptr(sh), C.byref(nh)), "rc_stage_shade")
        return sec[:ns.value], sh[:nh.value]

    def stage_trace_shadow_rays(self, p, shadow_rays, clamp_val):
        shadow_rays = np.ascontiguousarray(shadow_rays)
        self._check(self.lib.rc_stage_trace_shadow_rays(self._ctx, C.byref(p), _ptr(shadow_rays), len(shadow_rays),
                                                        float(clamp_val)), "rc_stage_trace_shadow_rays")

    def stage_sort_rays(self, rays):
        rays = np.ascontiguousarray(rays.copy())
        keys = np.zeros(len(rays), dtype=np.uint32)
        self._check(self.lib.rc_stage_sort_rays(self._ctx, _ptr(rays), len(rays), _ptr(keys)), "rc_stage_sort_rays")
        return rays, keys

    def fill_temp(self, rgba=(0, 0, 0, 0)):
        arr = (C.c_float * 4)(*rgba)
        self._check(self.lib.rc_debug_fill_temp(self._ctx, arr), "rc_debug_fill_temp")

    def debug_write_plane(self, which, array):
        """Overwrite frame plane `which` (RC_BUF_FINAL .. RC_BUF_TEMP) with an (h, w, 4) float32 array."""
        a = np.ascontiguousarray(array, dtype=np.float32)
        if a.shape != (self.h, self.w, 4):
            raise ValueError(f"debug_write_plane: expected shape {(self.h, self.w, 4)}, got {a.shape}")
        self._check(self.lib.rc_debug_write_plane(self._ctx, which, _ptr(a)), "rc_debug_write_plane")

    def debug_unet_dims(self, tensor, flags):
        """(rows, cols, channel stride) of UNet tensor `tensor` of the path `flags` selects, as stored."""
        dims = (C.c_int32 * 3)()
        self._check(self.lib.rc_debug_unet_tensor(self._ctx, flags, tensor, 0, 0, None, dims), "rc_debug_unet_tensor")
        return tuple(dims)

    def debug_unet_tensor(self, tensor, flags, rows=None):
        """UNet tensor `tensor` (0..14: output of that pass, 15: the tensor-core path's network input) of the path
        `flags` selects, exactly as stored, as float32 (rows, cols, channel stride); rows = (row0, nrows) reads only
        those rows of the stored layout."""
        n, cols, cs = self.debug_unet_dims(tensor, flags)
        row0, nrows = (0, n) if rows is None else (int(rows[0]), int(rows[1]))
        out = np.empty((max(nrows, 0), cols, cs), dtype=np.float32)
        dims = (C.c_int32 * 3)()
        self._check(self.lib.rc_debug_unet_tensor(self._ctx, flags, tensor, row0, nrows, _ptr(out), dims),
                    "rc_debug_unet_tensor")
        return out
