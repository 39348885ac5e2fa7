/* ray_host.h -- flat C view of the C++ host layer (libray_host.so, namespace RayB200), for bindings (ctypes).
 *
 * One function per RendererBase / SceneBase call that the hot path uses (reference RendererBase.h:133-253,
 * SceneBase.h:371-516).  The C++ classes are the product API; this header only flattens them.  Errors are reported
 * the way the reference reports them -- through the ILog: rh_error_count() returns how many ILog::Error calls happened
 * since the renderer was created and rh_last_error() the last message (tests treat any Error as a failure, like the
 * reference's tests/test_scene.h:63-73).
 */
#ifndef RAY_HOST_H
#define RAY_HOST_H

#include <stdint.h>

#include "ray_cuda.h"
#include "ray_scene_desc.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rh_renderer rh_renderer;
typedef struct rh_scene rh_scene;

/* Ray::CreateRenderer(settings_t{w,h,preferred_device}, log, parallel_for, CUDA).  NULL when no sm_100 device exists. */
rh_renderer *rh_create_renderer(int w, int h, int device);
/* several devices of this node: `devices` is settings_t::preferred_device of the CUDA backend ("0,1,2,3", "0-7", "all");
 * the frame is sharded over them in row bands (rc_comm_* of ray_cuda.h) */
rh_renderer *rh_create_renderer_multi(int w, int h, const char *devices);
int rh_device_count(rh_renderer *r);
/* UNet denoiser (RendererBase::InitUNetFilter + DenoiseImage(pass, region) x pass_count): weights as rc_unet_layer[16] */
int rh_set_unet_weights(rh_renderer *r, const rc_unet_layer layers[16], uint32_t unet_flags);
/* AgX / Filmic view transform table (48^3 packed 10-10-10-2) for camera_desc_t::view_transform = view_transform */
int rh_set_view_lut(rh_renderer *r, uint32_t view_transform, const uint32_t *lut);
int rh_denoise_unet(rh_renderer *r, const rc_rect *rect, int iteration);
void rh_destroy_renderer(rh_renderer *r);
const char *rh_device_name(rh_renderer *r);
int rh_error_count(rh_renderer *r);
const char *rh_last_error(rh_renderer *r);
void rh_resize(rh_renderer *r, int w, int h);
void rh_clear(rh_renderer *r, const float rgba[4]);

rh_scene *rh_create_scene(rh_renderer *r);
void rh_destroy_scene(rh_scene *s);
void rh_set_environment(rh_scene *s, const rs_environment_desc *d);
/* SceneBase::AddTexture (SceneBase.h:392): returns TextureHandle::_index for the texture fields of the material descs */
uint32_t rh_add_texture(rh_scene *s, const rs_tex_desc *d);
uint32_t rh_add_material_node(rh_scene *s, const rs_shading_node_desc *d);
uint32_t rh_add_material_principled(rh_scene *s, const rs_principled_mat_desc *d);
uint32_t rh_add_mesh(rh_scene *s, const rs_mesh_desc *d);
uint32_t rh_add_mesh_instance(rh_scene *s, const rs_mesh_instance_desc *d);
/* SceneBase::SetMeshInstanceTransform / RemoveMeshInstance (take effect at the next rh_finalize; a Finalize that follows
 * only transform / analytic-light edits makes the renderer refresh the top level alone: rc_update_instances) */
void rh_set_mesh_instance_transform(rh_scene *s, uint32_t instance, const float *xform /* 16, column-major as in the desc */);
void rh_remove_mesh_instance(rh_scene *s, uint32_t instance);
uint32_t rh_add_light_directional(rh_scene *s, const rs_directional_light_desc *d);
uint32_t rh_add_light_sphere(rh_scene *s, const rs_sphere_light_desc *d);
uint32_t rh_add_light_spot(rh_scene *s, const rs_spot_light_desc *d);
uint32_t rh_add_light_rect(rh_scene *s, const rs_rect_light_desc *d);
uint32_t rh_add_light_disk(rh_scene *s, const rs_disk_light_desc *d);
uint32_t rh_add_light_line(rh_scene *s, const rs_line_light_desc *d);
uint32_t rh_add_camera(rh_scene *s, const rs_camera_desc *d);
void rh_finalize(rh_scene *s);
uint32_t rh_triangle_count(rh_scene *s);
uint32_t rh_node_count(rh_scene *s);
void rh_scene_view(rh_scene *s, rc_scene_view *out); /* pointers into the scene's arrays, valid until it changes */
void rh_get_camera(rh_scene *s, rc_camera *out);

/* RendererBase::RenderScene(scene, RegionContext{rect, *iteration}); *iteration is updated like region.iteration.
 * count > 1 = that many consecutive calls with one synchronisation at the end (Cuda::Renderer::RenderSceneBatch). */
void rh_render(rh_renderer *r, rh_scene *s, const rc_rect *rect, int *iteration, int count);
/* RendererBase::DenoiseImage(const RegionContext &): NLM filter of the region at RegionContext::iteration = iteration */
void rh_denoise(rh_renderer *r, const rc_rect *rect, int iteration);
/* which: 0 get_pixels_ref, 1 get_raw_pixels_ref, 2 aux BaseColor, 3 aux DepthNormals; borrowed pointer */
const float *rh_get_pixels(rh_renderer *r, int which, int *pitch);
/* RendererBase::get_sh_data_ref: w*h shl1_data_t {coeff_r[4], coeff_g[4], coeff_b[4]} (row pitch *pitch = w) of the
 * passes with camera_desc_t::output_sh; NULL when no such pass ran since the renderer was created or resized */
const float *rh_get_sh_data(rh_renderer *r, int *pitch);
void rh_get_stats(rh_renderer *r, uint64_t us[11]);
void rh_reset_stats(rh_renderer *r);
/* CUDA-backend extras */
void rh_get_counters(rh_renderer *r, rc_counters *out);
void rh_get_kernel_ms(rh_renderer *r, double ms[6], uint64_t launches[6]);
void rh_set_sampler_table(rh_renderer *r, const uint32_t *table);
void rh_set_render_flags(rh_renderer *r, uint32_t rc_render_flags);
void rh_invalidate_scene(rh_renderer *r); /* next render re-uploads the scene arrays */
void *rh_native_context(rh_renderer *r);   /* the rc_ctx* (include/ray_cuda.h) under the renderer */
/* the host layer's own tables (tests compare them with the reference's) */
void rh_builtin_sampler_table(uint32_t *out /* 32*4096*2 */);
void rh_builtin_filter_table(uint32_t filter, float filter_width, float *out /* 1024 */);
int rh_abi_sizeof(int which); /* 0..11: the rs_* structs in declaration order of ray_scene_desc.h */

#ifdef __cplusplus
}
#endif
#endif /* RAY_HOST_H */
