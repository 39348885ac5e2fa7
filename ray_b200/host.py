"""ctypes binding of libray_host.so (include/ray_host.h): the product's public API as seen from Python.

    r = host.Renderer(w, h, device=0)          # Ray::CreateRenderer(settings, log, ..., eRendererType::CUDA)
    s = r.create_scene()                       # RendererBase::CreateScene
    scenes.build(desc, s)                      # SceneBase::AddMaterial / AddMesh / ... / Finalize
    it = r.render(s, (0, 0, w, h), it, count)  # RendererBase::RenderScene (count > 1: one sync for `count` samples)
    img = r.pixels(host.RAW)                   # get_raw_pixels_ref

No fallback: the constructor raises if the library or an sm_100 device is missing.
"""
import ctypes as C
import os

import numpy as np

from . import capi
from . import cuda as _cuda

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libray_host.so")
FINAL, RAW, BASE_COLOR, DEPTH_NORMALS = 0, 1, 2, 3

EXPORTED_SYMBOLS = [
    "rh_create_renderer", "rh_create_renderer_multi", "rh_device_count", "rh_set_unet_weights", "rh_set_view_lut", "rh_denoise_unet", "rh_destroy_renderer", "rh_device_name", "rh_error_count", "rh_last_error", "rh_resize",
    "rh_clear", "rh_create_scene", "rh_destroy_scene", "rh_set_environment", "rh_denoise", "rh_add_texture", "rh_add_material_node",
    "rh_add_material_principled", "rh_add_mesh", "rh_add_mesh_instance", "rh_set_mesh_instance_transform",
    "rh_remove_mesh_instance", "rh_add_light_directional",
    "rh_add_light_sphere", "rh_add_light_spot", "rh_add_light_rect", "rh_add_light_disk", "rh_add_light_line",
    "rh_add_camera", "rh_finalize", "rh_triangle_count", "rh_node_count", "rh_scene_view", "rh_get_camera", "rh_render",
    "rh_get_pixels", "rh_get_sh_data", "rh_get_stats", "rh_reset_stats", "rh_get_counters", "rh_get_kernel_ms", "rh_set_sampler_table",
    "rh_set_render_flags", "rh_invalidate_scene", "rh_native_context", "rh_builtin_sampler_table", "rh_builtin_filter_table", "rh_abi_sizeof",
]

_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    _cuda.load_library()  # libray_host.so links against libray_cuda.so (rpath $ORIGIN)
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(LIB_PATH)
    vp, P = C.c_void_p, C.POINTER
    u32 = C.c_uint32
    sig = {
        "rh_create_renderer": (vp, [C.c_int, C.c_int, C.c_int]),
        "rh_create_renderer_multi": (vp, [C.c_int, C.c_int, C.c_char_p]),
        "rh_device_count": (C.c_int, [vp]),
        "rh_set_unet_weights": (C.c_int, [vp, vp, C.c_uint32]),
        "rh_set_view_lut": (C.c_int, [vp, C.c_uint32, vp]),
        "rh_denoise_unet": (C.c_int, [vp, P(capi.rc_rect), C.c_int]),
        "rh_destroy_renderer": (None, [vp]),
        "rh_device_name": (C.c_char_p, [vp]),
        "rh_error_count": (C.c_int, [vp]),
        "rh_last_error": (C.c_char_p, [vp]),
        "rh_resize": (None, [vp, C.c_int, C.c_int]),
        "rh_clear": (None, [vp, P(C.c_float)]),
        "rh_create_scene": (vp, [vp]),
        "rh_destroy_scene": (None, [vp]),
        "rh_set_environment": (None, [vp, P(capi.rs_environment_desc)]),
        "rh_add_texture": (u32, [vp, P(capi.rs_tex_desc)]),
        "rh_denoise": (None, [vp, P(capi.rc_rect), C.c_int]),
        "rh_add_material_node": (u32, [vp, P(capi.rs_shading_node_desc)]),
        "rh_add_material_principled": (u32, [vp, P(capi.rs_principled_mat_desc)]),
        "rh_add_mesh": (u32, [vp, P(capi.rs_mesh_desc)]),
        "rh_add_mesh_instance": (u32, [vp, P(capi.rs_mesh_instance_desc)]),
        "rh_set_mesh_instance_transform": (None, [vp, u32, vp]),
        "rh_remove_mesh_instance": (None, [vp, u32]),
        "rh_add_light_directional": (u32, [vp, P(capi.rs_directional_light_desc)]),
        "rh_add_light_sphere": (u32, [vp, P(capi.rs_sphere_light_desc)]),
        "rh_add_light_spot": (u32, [vp, P(capi.rs_spot_light_desc)]),
        "rh_add_light_rect": (u32, [vp, P(capi.rs_rect_light_desc)]),
        "rh_add_light_disk": (u32, [vp, P(capi.rs_disk_light_desc)]),
        "rh_add_light_line": (u32, [vp, P(capi.rs_line_light_desc)]),
        "rh_add_camera": (u32, [vp, P(capi.rs_camera_desc)]),
        "rh_finalize": (None, [vp]),
        "rh_triangle_count": (u32, [vp]),
        "rh_node_count": (u32, [vp]),
        "rh_scene_view": (None, [vp, P(capi.rc_scene_view)]),
        "rh_get_camera": (None, [vp, P(capi.rc_camera)]),
        "rh_render": (None, [vp, vp, P(capi.rc_rect), P(C.c_int), C.c_int]),
        "rh_get_pixels": (P(C.c_float), [vp, C.c_int, P(C.c_int)]),
        "rh_get_sh_data": (P(C.c_float), [vp, P(C.c_int)]),
        "rh_get_stats": (None, [vp, P(C.c_uint64)]),
        "rh_reset_stats": (None, [vp]),
        "rh_get_counters": (None, [vp, P(capi.rc_counters)]),
        "rh_get_kernel_ms": (None, [vp, P(C.c_double), P(C.c_uint64)]),
        "rh_set_sampler_table": (None, [vp, vp]),
        "rh_set_render_flags": (None, [vp, u32]),
        "rh_invalidate_scene": (None, [vp]),
        "rh_native_context": (vp, [vp]),
        "rh_builtin_sampler_table": (None, [vp]),
        "rh_builtin_filter_table": (None, [u32, C.c_float, vp]),
        "rh_abi_sizeof": (C.c_int, [C.c_int]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class HostError(RuntimeError):
    pass


def builtin_sampler_table():
    t = np.zeros(32 * 4096 * 2, dtype=np.uint32)
    load_library().rh_builtin_sampler_table(t.ctypes.data_as(C.c_void_p))
    return t


def builtin_filter_table(filter, width):
    t = np.zeros(1024, dtype=np.float32)
    load_library().rh_builtin_filter_table(filter, float(width), t.ctypes.data_as(C.c_void_p))
    return t


class Scene:
    """Cuda::Scene behind the scene-building verbs used by ray_b200.scenes.build()."""

    def __init__(self, renderer=None):
        """`renderer=None` gives a free-standing scene (no GPU needed): scene building is pure host work."""
        self.lib = renderer.lib if renderer is not None else load_library()
        self.renderer = renderer
        self.h = self.lib.rh_create_scene(renderer.h if renderer is not None else None)

    def close(self):
        if getattr(self, "h", None):
            self.lib.rh_destroy_scene(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_environment(self, env_col, back_col, importance_sample=True, env_map=capi.RS_INVALID,
                        back_map=capi.RS_INVALID, env_map_rotation=0.0, back_map_rotation=0.0):
        d = capi.rs_environment_desc(env_col=tuple(env_col), back_col=tuple(back_col),
                                     importance_sample=1 if importance_sample else 0, env_map=env_map,
                                     back_map=back_map, env_map_rotation=env_map_rotation,
                                     back_map_rotation=back_map_rotation)
        self.lib.rh_set_environment(self.h, C.byref(d))

    def add_texture(self, pixels, is_srgb=True, is_normalmap=False, generate_mipmaps=False, reconstruct_z=False,
                    convention=0):
        """SceneBase::AddTexture for a (h, w, c) uint8 array, c in 1..4; returns the texture handle."""
        d, keep = capi.make_tex_desc(pixels, is_srgb, is_normalmap, generate_mipmaps, reconstruct_z, convention)
        return self.lib.rh_add_texture(self.h, C.byref(d))

    def add_material_node(self, d):
        return self.lib.rh_add_material_node(self.h, C.byref(d))

    def add_material_principled(self, d):
        return self.lib.rh_add_material_principled(self.h, C.byref(d))

    def add_mesh(self, attrs, indices, groups, allow_spatial_splits=False, use_fast_bvh_build=False):
        attrs = np.ascontiguousarray(attrs, dtype=np.float32)
        indices = np.ascontiguousarray(indices, dtype=np.uint32)
        fp = attrs.ctypes.data_as(C.POINTER(C.c_float))
        m = capi.rs_mesh_desc()
        m.vtx_positions = capi.rs_vtx_attribute(fp, attrs.size, 0, 8)
        m.vtx_normals = capi.rs_vtx_attribute(fp, attrs.size, 3, 8)
        m.vtx_binormals = capi.rs_vtx_attribute(None, 0, 0, 0)
        m.vtx_uvs = capi.rs_vtx_attribute(fp, attrs.size, 6, 8)
        m.vtx_indices = indices.ctypes.data_as(C.POINTER(C.c_uint32))
        m.vtx_indices_count = len(indices)
        m.base_vertex = 0
        garr = (capi.rs_mat_group_desc * len(groups))(*[capi.rs_mat_group_desc(*g) for g in groups])
        m.groups = garr
        m.groups_count = len(groups)
        m.allow_spatial_splits = 1 if allow_spatial_splits else 0
        m.use_fast_bvh_build = 1 if use_fast_bvh_build else 0
        return self.lib.rh_add_mesh(self.h, C.byref(m))

    def add_mesh_instance(self, mesh, xform, camera_visibility=True, diffuse_visibility=True, specular_visibility=True,
                          refraction_visibility=True, shadow_visibility=True):
        d = capi.rs_mesh_instance_desc(xform=tuple(float(x) for x in xform), mesh=mesh,
                                       camera_visibility=int(camera_visibility),
                                       diffuse_visibility=int(diffuse_visibility),
                                       specular_visibility=int(specular_visibility),
                                       refraction_visibility=int(refraction_visibility),
                                       shadow_visibility=int(shadow_visibility))
        return self.lib.rh_add_mesh_instance(self.h, C.byref(d))

    def set_mesh_instance_transform(self, instance, xform):
        m = np.ascontiguousarray(xform, dtype=np.float32).reshape(16)
        self.lib.rh_set_mesh_instance_transform(self.h, instance, m.ctypes.data)

    def remove_mesh_instance(self, instance):
        self.lib.rh_remove_mesh_instance(self.h, instance)

    def add_light(self, kind, d):
        return getattr(self.lib, f"rh_add_light_{kind}")(self.h, C.byref(d))

    def add_camera(self, d):
        return self.lib.rh_add_camera(self.h, C.byref(d))

    def finalize(self):
        self.lib.rh_finalize(self.h)
        if self.renderer is not None:
            self.renderer.check()

    def triangle_count(self):
        return self.lib.rh_triangle_count(self.h)

    def node_count(self):
        return self.lib.rh_node_count(self.h)

    def view(self):
        v = capi.rc_scene_view()
        self.lib.rh_scene_view(self.h, C.byref(v))
        return v

    def camera(self):
        c = capi.rc_camera()
        self.lib.rh_get_camera(self.h, C.byref(c))
        return c


class Renderer:
    """Cuda::Renderer (RendererBase) through the C wrapper."""

    def __init__(self, w, h, device=0, devices=None):
        """`devices` (e.g. "0,1,2,3", "0-7", "all") shards the frame over several GPUs of this node in one process."""
        self.lib = load_library()
        if devices is not None:
            self.h = self.lib.rh_create_renderer_multi(w, h, str(devices).encode())
        else:
            self.h = self.lib.rh_create_renderer(w, h, device)
        if not self.h:
            raise HostError("Ray::CreateRenderer(CUDA) failed: no usable sm_100 CUDA device (there is no CPU fallback)")
        self.w, self.hh = w, h

    def close(self):
        if getattr(self, "h", None):
            self.lib.rh_destroy_renderer(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self):
        """Raise if the backend logged an error (the reference's tests fail on any ILog::Error)."""
        if self.lib.rh_error_count(self.h):
            raise HostError(self.lib.rh_last_error(self.h).decode())

    @property
    def device_name(self):
        return self.lib.rh_device_name(self.h).decode()

    def create_scene(self):
        return Scene(self)

    def resize(self, w, h):
        self.lib.rh_resize(self.h, w, h)
        self.w, self.hh = w, h
        self.check()

    def clear(self, rgba=(0, 0, 0, 0)):
        self.lib.rh_clear(self.h, (C.c_float * 4)(*rgba))
        self.check()

    def render(self, scene, rect, iteration, count=1):
        r = capi.rc_rect(*rect)
        it = C.c_int(iteration)
        self.lib.rh_render(self.h, scene.h, C.byref(r), C.byref(it), count)
        self.check()
        return it.value

    def set_unet_weights(self, layers, flags=0):
        """layers: 16 x (weights fp16 [cout, cin, 3, 3], bias fp16 [cout]) in pass order (include/ray_cuda.h)"""
        class L(C.Structure):
            _fields_ = [("weights", C.c_void_p), ("bias", C.c_void_p), ("cin", C.c_int32), ("cout", C.c_int32)]
        arr = (L * 16)()
        keep = []
        for i, (w, b) in enumerate(layers):
            w = np.ascontiguousarray(w, dtype=np.float16)
            b = np.ascontiguousarray(b, dtype=np.float16)
            keep += [w, b]
            arr[i] = L(w.ctypes.data, b.ctypes.data, w.shape[1], w.shape[0])
        if self.lib.rh_set_unet_weights(self.h, C.byref(arr), flags) != 0:
            self.check()

    def set_view_lut(self, view_transform, lut):
        lut = np.ascontiguousarray(lut, dtype=np.uint32)
        assert lut.size == 48 ** 3
        if self.lib.rh_set_view_lut(self.h, view_transform, lut.ctypes.data) != 0:
            raise HostError(self.lib.rh_last_error(self.h).decode())

    def denoise_unet(self, rect, iteration):
        r = capi.rc_rect(*rect)
        n = self.lib.rh_denoise_unet(self.h, C.byref(r), int(iteration))
        self.check()
        return n

    def denoise(self, rect, iteration):
        """RendererBase::DenoiseImage(region): joint NLM filter; results through pixels(FINAL) / pixels(RAW)."""
        r = capi.rc_rect(*rect)
        self.lib.rh_denoise(self.h, C.byref(r), int(iteration))
        self.check()

    def pixels(self, which=RAW, copy=True):
        """RendererBase::get_pixels_ref / get_raw_pixels_ref / get_aux_pixels_ref: reads the plane back into the
        renderer's page-locked mirror.  copy=False returns a view of that mirror, BORROWED exactly like the reference's
        color_data_rgba_t (valid until the next RenderScene / Resize); copy=True detaches it."""
        pitch = C.c_int(0)
        p = self.lib.rh_get_pixels(self.h, which, C.byref(pitch))
        self.check()
        a = np.ctypeslib.as_array(p, shape=(self.hh, pitch.value, 4))[:, :self.w, :]
        return a.copy() if copy else a

    def sh_data(self):
        """RendererBase::get_sh_data_ref as an (h, w, 3, 4) array (channel r/g/b, 4 L1 coefficients), or None when no
        pass with camera output_sh has run."""
        pitch = C.c_int(0)
        p = self.lib.rh_get_sh_data(self.h, C.byref(pitch))
        self.check()
        if not p:
            return None
        return np.ctypeslib.as_array(p, shape=(self.hh, pitch.value, 3, 4))[:, :self.w].copy()

    def stats_us(self):
        a = (C.c_uint64 * 11)()
        self.lib.rh_get_stats(self.h, a)
        return list(a)

    def reset_stats(self):
        self.lib.rh_reset_stats(self.h)

    def counters(self):
        c = capi.rc_counters()
        self.lib.rh_get_counters(self.h, C.byref(c))
        return {k: getattr(c, k) for k, _ in capi.rc_counters._fields_}

    def kernel_ms(self):
        ms = (C.c_double * 6)()
        n = (C.c_uint64 * 6)()
        self.lib.rh_get_kernel_ms(self.h, ms, n)
        names = ["raygen", "trace_closest", "shade", "trace_shadow", "sort", "resolve"]
        return {k: (ms[i], n[i]) for i, k in enumerate(names)}

    def set_sampler_table(self, table):
        t = np.ascontiguousarray(table, dtype=np.uint32)
        assert t.size == 32 * 4096 * 2
        self.lib.rh_set_sampler_table(self.h, t.ctypes.data_as(C.c_void_p))

    def set_render_flags(self, flags):
        self.lib.rh_set_render_flags(self.h, flags)

    def invalidate_scene(self):
        self.lib.rh_invalidate_scene(self.h)

    def native_context(self):
        """The rc_ctx* under this renderer (for rc_event_* / rc_device_ptr through ray_b200.cuda)."""
        return C.c_void_p(self.lib.rh_native_context(self.h))
