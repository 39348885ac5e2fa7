"""ctypes mirrors of the C structs in include/ray_scene_desc.h and include/ray_cuda.h.

Field order and types must match the headers exactly; tests/test_abi.py checks sizeof() of every struct against the
values the C compiler reports (through rc_abi_sizeof / rh_abi_sizeof).
"""
import ctypes as C

RS_INVALID = 0xFFFFFFFF

# eShadingNode (reference SceneBase.h:41)
NODE_DIFFUSE, NODE_GLOSSY, NODE_REFRACTIVE, NODE_EMISSIVE, NODE_MIX, NODE_TRANSPARENT, NODE_PRINCIPLED = range(7)
# ePixelFilter
FILTER_BOX, FILTER_GAUSSIAN, FILTER_BLACKMAN_HARRIS = range(3)
# eRendererType (reference RendererBase.h:22-34) + the new backend
RT_REFERENCE, RT_SSE41, RT_AVX, RT_AVX2, RT_AVX512, RT_NEON, RT_VULKAN, RT_DX12, RT_CUDA = range(9)

f32, u32, i32, u64 = C.c_float, C.c_uint32, C.c_int32, C.c_uint64


class rs_shading_node_desc(C.Structure):
    _fields_ = [("type", u32), ("base_color", f32 * 3), ("base_texture", u32), ("normal_map", u32),
                ("normal_map_intensity", f32), ("mix_materials", u32 * 2), ("roughness", f32),
                ("roughness_texture", u32), ("anisotropic", f32), ("anisotropic_rotation", f32), ("sheen", f32),
                ("specular", f32), ("strength", f32), ("fresnel", f32), ("ior", f32), ("tint", f32),
                ("metallic_texture", u32), ("importance_sample", u32), ("mix_add", u32)]

    @classmethod
    def default(cls, **kw):
        d = cls(type=NODE_DIFFUSE, base_color=(1, 1, 1), base_texture=RS_INVALID, normal_map=RS_INVALID,
                normal_map_intensity=1.0, mix_materials=(RS_INVALID, RS_INVALID), roughness=0.0,
                roughness_texture=RS_INVALID, anisotropic=0.0, anisotropic_rotation=0.0, sheen=0.0, specular=0.0,
                strength=1.0, fresnel=1.0, ior=1.0, tint=0.0, metallic_texture=RS_INVALID, importance_sample=0,
                mix_add=0)
        _apply(d, kw)
        return d


class rs_principled_mat_desc(C.Structure):
    _fields_ = [("base_color", f32 * 3), ("base_texture", u32), ("metallic", f32), ("metallic_texture", u32),
                ("specular", f32), ("specular_texture", u32), ("specular_tint", f32), ("roughness", f32),
                ("roughness_texture", u32), ("anisotropic", f32), ("anisotropic_rotation", f32), ("sheen", f32),
                ("sheen_tint", f32), ("clearcoat", f32), ("clearcoat_roughness", f32), ("ior", f32),
                ("transmission", f32), ("transmission_roughness", f32), ("emission_color", f32 * 3),
                ("emission_texture", u32), ("emission_strength", f32), ("alpha", f32), ("alpha_texture", u32),
                ("normal_map", u32), ("normal_map_intensity", f32), ("importance_sample", u32)]

    @classmethod
    def default(cls, **kw):
        d = cls(base_color=(1, 1, 1), base_texture=RS_INVALID, metallic=0.0, metallic_texture=RS_INVALID,
                specular=0.5, specular_texture=RS_INVALID, specular_tint=0.0, roughness=0.5,
                roughness_texture=RS_INVALID, anisotropic=0.0, anisotropic_rotation=0.0, sheen=0.0, sheen_tint=0.5,
                clearcoat=0.0, clearcoat_roughness=0.0, ior=1.45, transmission=0.0, transmission_roughness=0.0,
                emission_color=(0, 0, 0), emission_texture=RS_INVALID, emission_strength=1.0, alpha=1.0,
                alpha_texture=RS_INVALID, normal_map=RS_INVALID, normal_map_intensity=1.0, importance_sample=0)
        _apply(d, kw)
        return d


RS_TEX_RGBA8888, RS_TEX_RGB888, RS_TEX_RG88, RS_TEX_R8 = 1, 2, 3, 4


class rs_tex_desc(C.Structure):
    _fields_ = [("format", u32), ("convention", u32), ("data", C.c_void_p), ("w", i32), ("h", i32), ("is_srgb", u32),
                ("is_normalmap", u32), ("generate_mipmaps", u32), ("reconstruct_z", u32)]


class rs_mat_group_desc(C.Structure):
    _fields_ = [("front_mat", u32), ("back_mat", u32), ("vtx_start", u64), ("vtx_count", u64)]


class rs_vtx_attribute(C.Structure):
    _fields_ = [("data", C.POINTER(f32)), ("count", u64), ("offset", i32), ("stride", i32)]


class rs_mesh_desc(C.Structure):
    _fields_ = [("vtx_positions", rs_vtx_attribute), ("vtx_normals", rs_vtx_attribute),
                ("vtx_binormals", rs_vtx_attribute), ("vtx_uvs", rs_vtx_attribute),
                ("vtx_indices", C.POINTER(u32)), ("vtx_indices_count", u64), ("base_vertex", i32),
                ("groups", C.POINTER(rs_mat_group_desc)), ("groups_count", u32), ("allow_spatial_splits", u32),
                ("use_fast_bvh_build", u32)]


class rs_mesh_instance_desc(C.Structure):
    _fields_ = [("xform", f32 * 16), ("mesh", u32), ("camera_visibility", u32), ("diffuse_visibility", u32),
                ("specular_visibility", u32), ("refraction_visibility", u32), ("shadow_visibility", u32)]


class rs_light_common(C.Structure):
    _fields_ = [("color", f32 * 3), ("multiple_importance", u32), ("cast_shadow", u32), ("diffuse_visibility", u32),
                ("specular_visibility", u32), ("refraction_visibility", u32)]

    @classmethod
    def default(cls, **kw):
        d = cls(color=(1, 1, 1), multiple_importance=1, cast_shadow=1, diffuse_visibility=1, specular_visibility=1,
                refraction_visibility=1)
        _apply(d, kw)
        return d


class rs_directional_light_desc(C.Structure):
    _fields_ = [("c", rs_light_common), ("direction", f32 * 3), ("angle", f32)]


class rs_sphere_light_desc(C.Structure):
    _fields_ = [("c", rs_light_common), ("position", f32 * 3), ("radius", f32)]


class rs_spot_light_desc(C.Structure):
    _fields_ = [("c", rs_light_common), ("position", f32 * 3), ("direction", f32 * 3), ("spot_size", f32),
                ("spot_blend", f32), ("radius", f32)]


class rs_rect_light_desc(C.Structure):
    _fields_ = [("c", rs_light_common), ("width", f32), ("height", f32), ("doublesided", u32), ("sky_portal", u32),
                ("xform", f32 * 16)]


class rs_disk_light_desc(C.Structure):
    _fields_ = [("c", rs_light_common), ("size_x", f32), ("size_y", f32), ("doublesided", u32), ("sky_portal", u32),
                ("xform", f32 * 16)]


class rs_line_light_desc(C.Structure):
    _fields_ = [("c", rs_light_common), ("radius", f32), ("height", f32), ("sky_portal", u32), ("xform", f32 * 16)]


class rs_camera_desc(C.Structure):
    _fields_ = [("type", u32), ("filter", u32), ("view_transform", u32), ("ltype", u32), ("filter_width", f32),
                ("origin", f32 * 3), ("fwd", f32 * 3), ("up", f32 * 3), ("shift", f32 * 2), ("exposure", f32),
                ("fov", f32), ("gamma", f32), ("sensor_height", f32), ("focus_distance", f32), ("focal_length", f32),
                ("fstop", f32), ("lens_rotation", f32), ("lens_ratio", f32), ("lens_blades", i32),
                ("clip_start", f32), ("clip_end", f32), ("mi_index", u32), ("uv_index", u32), ("lighting_only", u32),
                ("skip_direct_lighting", u32), ("skip_indirect_lighting", u32), ("no_background", u32),
                ("output_sh", u32), ("max_diff_depth", u32), ("max_spec_depth", u32), ("max_refr_depth", u32),
                ("max_transp_depth", u32), ("max_total_depth", u32), ("min_total_depth", u32),
                ("min_transp_depth", u32), ("clamp_direct", f32), ("clamp_indirect", f32), ("min_samples", i32),
                ("variance_threshold", f32), ("regularize_alpha", f32)]

    @classmethod
    def default(cls, **kw):
        d = cls(type=0, filter=FILTER_BLACKMAN_HARRIS, view_transform=0, ltype=0, filter_width=1.5, origin=(0, 0, 0),
                fwd=(0, 0, 0), up=(0, 0, 0), shift=(0, 0), exposure=0.0, fov=45.0, gamma=1.0, sensor_height=0.036,
                focus_distance=1.0, focal_length=0.0, fstop=0.0, lens_rotation=0.0, lens_ratio=1.0, lens_blades=0,
                clip_start=0.0, clip_end=3.402823466e+30, mi_index=0xFFFFFFFF, uv_index=0, lighting_only=0,
                skip_direct_lighting=0, skip_indirect_lighting=0, no_background=0, output_sh=0, max_diff_depth=4,
                max_spec_depth=8, max_refr_depth=8, max_transp_depth=8, max_total_depth=8, min_total_depth=2,
                min_transp_depth=2, clamp_direct=0.0, clamp_indirect=0.0, min_samples=128, variance_threshold=0.0,
                regularize_alpha=0.03)
        _apply(d, kw)
        return d


class rs_environment_desc(C.Structure):
    _fields_ = [("env_col", f32 * 3), ("back_col", f32 * 3), ("importance_sample", u32), ("env_map", u32),
                ("back_map", u32), ("env_map_rotation", f32), ("back_map_rotation", f32)]


# ---- include/ray_cuda.h -------------------------------------------------------------------------------------------
class rc_array(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("count", u32), ("stride", u32)]


RC_TEX_MIP_LEVELS = 12


class rc_texture(C.Structure):
    _fields_ = [("handle", u32), ("channels", u32), ("res", (C.c_uint16 * 2) * RC_TEX_MIP_LEVELS),
                ("pixels", C.c_void_p * RC_TEX_MIP_LEVELS)]


class rc_scene_view(C.Structure):
    _fields_ = [("wnodes", rc_array), ("mtris", rc_array), ("tri_indices", rc_array), ("tri_materials", rc_array),
                ("materials", rc_array), ("mesh_instances", rc_array), ("vertices", rc_array),
                ("vtx_indices", rc_array), ("lights", rc_array), ("li_indices", rc_array), ("light_cwnodes", rc_array),
                ("tlas_root", u32), ("visible_lights_count", u32), ("blocker_lights_count", u32),
                ("env_col", f32 * 3), ("env_map", u32), ("back_col", f32 * 3), ("back_map", u32),
                ("env_light_index", u32), ("sky_map_spread_angle", f32), ("bounds_min", f32 * 3),
                ("bounds_max", f32 * 3), ("textures", C.POINTER(rc_texture)), ("texture_count", u32), ("qtree_levels", i32),
                ("env_map_rotation", f32), ("back_map_rotation", f32), ("qtree_mips", C.c_void_p * 16)]


class rc_camera(C.Structure):
    _fields_ = [("type", u32), ("filter", u32), ("view_transform", u32), ("fov", f32), ("exposure", f32),
                ("gamma", f32), ("sensor_height", f32), ("focus_distance", f32), ("focal_length", f32),
                ("fstop", f32), ("lens_rotation", f32), ("lens_ratio", f32), ("lens_blades", i32),
                ("clip_start", f32), ("clip_end", f32), ("origin", f32 * 3), ("fwd", f32 * 3), ("side", f32 * 3),
                ("up", f32 * 3), ("shift", f32 * 2), ("max_diff_depth", u32), ("max_spec_depth", u32),
                ("max_refr_depth", u32), ("max_transp_depth", u32), ("max_total_depth", u32),
                ("min_total_depth", u32), ("min_transp_depth", u32), ("clamp_direct", f32), ("clamp_indirect", f32),
                ("min_samples", i32), ("variance_threshold", f32), ("regularize_alpha", f32)]


class rc_rect(C.Structure):
    _fields_ = [("x", i32), ("y", i32), ("w", i32), ("h", i32)]


class rc_pass_desc(C.Structure):
    _fields_ = [("cam", rc_camera), ("rect", rc_rect), ("iteration", i32), ("flags", u32), ("geo_instance", u32),
                ("geo_tri_first", u32), ("geo_tri_count", u32)]


class rc_counters(C.Structure):
    _fields_ = [("primary_rays", u64), ("secondary_rays", u64), ("shadow_rays", u64), ("nodes_visited", u64),
                ("leaves_tested", u64), ("samples", u64)]


RC_RENDER_ASYNC, RC_RENDER_NO_SORT = 1, 2
RC_RENDER_SKIP_DIRECT, RC_RENDER_SKIP_INDIRECT, RC_RENDER_LIGHTING_ONLY, RC_RENDER_NO_BACKGROUND, RC_RENDER_OUTPUT_SH = \
    4, 8, 16, 32, 64
CAM_PERSP, CAM_ORTHO, CAM_GEO = 0, 1, 2
RC_UNET_TENSOR_CORES, RC_UNET_FP32 = 0, 1
RC_BUF_FINAL, RC_BUF_RAW, RC_BUF_BASE_COLOR, RC_BUF_DEPTH_NORMALS, RC_BUF_FULL, RC_BUF_HALF, RC_BUF_TEMP = range(7)
RC_BUF_SH_R, RC_BUF_SH_G, RC_BUF_SH_B = 7, 8, 9


def _apply(struct, kw):
    for k, v in kw.items():
        if not hasattr(struct, k):
            raise AttributeError(f"{type(struct).__name__} has no field {k}")
        cur = getattr(struct, k)
        if isinstance(cur, C.Array):
            for i, x in enumerate(v):
                cur[i] = x
        else:
            setattr(struct, k, v)


def make_tex_desc(pixels, is_srgb=True, is_normalmap=False, generate_mipmaps=False, reconstruct_z=False, convention=0):
    """rs_tex_desc over a (h, w, c) or (h, w) uint8 array; returns (desc, keep-alive array)."""
    import numpy as np
    a = np.ascontiguousarray(pixels, dtype=np.uint8)
    if a.ndim == 2:
        a = a[:, :, None]
    h, w, c = a.shape
    fmt = {4: RS_TEX_RGBA8888, 3: RS_TEX_RGB888, 2: RS_TEX_RG88, 1: RS_TEX_R8}[c]
    d = rs_tex_desc(fmt, convention, a.ctypes.data, w, h, 1 if is_srgb else 0, 1 if is_normalmap else 0,
                    1 if generate_mipmaps else 0, 1 if reconstruct_z else 0)
    d._keep = a
    return d, a
