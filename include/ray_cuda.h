/* ray_cuda.h -- C-ABI of libray_cuda.so: the sm_100a driver layer under Ray::Cuda::Renderer.
 *
 * This is the boundary SURVEY.md section 8(b) specifies: `extern "C"`, opaque context, plain pointers and sizes,
 * caller-owned host memory, int return codes (0 = ok; rc_last_error() explains a failure), no C++ types and no
 * exceptions across the boundary, one context per device, not thread-safe.  The only intended caller is the C++
 * Cuda::Renderer (ray_b200/csrc/host, or the binding shown in INTEGRATION.md for the reference tree); tests drive it
 * through ctypes.
 *
 * What each entry point replaces in the reference (file:line relative to the reference tree):
 *   rc_create/rc_destroy      backend construction in Ray::CreateRenderer (Ray.cpp:53-133; a failing rc_create is
 *                             what makes Cuda::Renderer's ctor throw so the factory falls through)
 *   rc_resize / rc_clear      Cpu::Renderer::Resize / Clear (internal/RendererCPU.h:266-301)
 *   rc_upload_tables          the `rand_seq = __pmj02_samples` argument (internal/RendererCPU.h:445) and
 *                             filter_table_ (internal/RendererCPU.h:1234-1258)
 *   rc_upload_scene           construction of scene_data_t from Cpu::Scene's arrays (internal/RendererCPU.h:390-413)
 *   rc_render                 the body of Cpu::Renderer<P>::RenderScene (internal/RendererCPU.h:374-659):
 *                             GeneratePrimaryRays, TraceRays, ShadePrimary, TraceShadowRays, the bounce loop with
 *                             SortRays/TraceRays/ShadeSecondary/TraceShadowRays, accumulate + tonemap + variance
 *   rc_readback               get_pixels_ref / get_raw_pixels_ref / get_aux_pixels_ref (RendererCPU.h:255-265)
 *   rc_get_stats              RendererBase::GetStats (RendererBase.h:230-245)
 *   rc_stage_*                the SIMDPolicy stage functions (internal/RendererCPU.h:39-189) on caller-provided AoS
 *                             buffers in the reference's own ray_data_t / hit_data_t / shadow_ray_t layouts --
 *                             test/debug entry points used for per-stage parity against Ref::*
 */
#ifndef RAY_CUDA_H
#define RAY_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rc_ctx rc_ctx;

/* One scene array: pointer to the first element, element count (capacity of the SparseStorage), element size. */
typedef struct rc_array {
    const void *ptr;
    uint32_t count;
    uint32_t stride;
} rc_array;

/* One texture of the scene's texture storages (reference internal/TextureStorageCPU.h, SceneCPU.h:65-76), handed over
 * DECODED: row-major 8-bit texels, `channels` per texel, one pointer per mip level.  `handle` is what material_t::textures[]
 * and light_t::tri.tex_index carry without the flag bits 24..27: (storage << 28) | index (Core.h:159-161,
 * SceneCPU.cpp:191-204).  The texel a lookup returns is the one TexStorageBase::Fetch(index, x, y, lod) returns
 * (x %= w, y %= h; channels missing in the storage repeat the last stored one; value = byte / 255.0f), so the binding on
 * the reference side either walks Fetch() or hands over its pixel arrays.  Levels the storage does not have alias the
 * last real one exactly as TexStorage*::Allocate fills res[]/lod_offsets[] (TextureStorageCPU.cpp:234-250). */
#define RC_TEX_MIP_LEVELS 12 /* NUM_MIP_LEVELS, Constants.inl:91 */
typedef struct rc_texture {
    uint32_t handle;
    uint32_t channels; /* 1..4 */
    uint16_t res[RC_TEX_MIP_LEVELS][2];
    const uint8_t *pixels[RC_TEX_MIP_LEVELS];
} rc_texture;

/* View of a finalized wide-BVH Cpu::Scene (reference internal/SceneCPU.h:50-98).  Layouts are the reference's
 * (internal/Core.h); strides are checked against them. */
typedef struct rc_scene_view {
    rc_array wnodes;         /* wbvh_node_t          224 B */
    rc_array mtris;          /* mtri_accel_t         384 B */
    rc_array tri_indices;    /* uint32_t               4 B */
    rc_array tri_materials;  /* tri_mat_data_t         4 B */
    rc_array materials;      /* material_t            76 B */
    rc_array mesh_instances; /* mesh_instance_t      144 B */
    rc_array vertices;       /* vertex_t              44 B */
    rc_array vtx_indices;    /* uint32_t               4 B */
    rc_array lights;         /* light_t               64 B */
    rc_array li_indices;     /* uint32_t               4 B */
    rc_array light_cwnodes;  /* light_cwbvh_node_t   208 B */
    uint32_t tlas_root;      /* 0xffffffff = empty scene */
    uint32_t visible_lights_count, blocker_lights_count;
    /* environment_t subset (Core.h:393-410) */
    float env_col[3];
    uint32_t env_map;        /* 0xffffffff or the handle of an RGBE lat-long texture of the RGBA storage (in `textures`) */
    float back_col[3];
    uint32_t back_map;       /* likewise, for camera rays */
    uint32_t env_light_index;
    float sky_map_spread_angle; /* must be 0: the procedural sky is out of scope */
    /* Cpu::Scene::GetBounds (ray-sort grid) */
    float bounds_min[3], bounds_max[3];
    /* textures referenced by materials / triangle lights (NULL / 0 for an untextured scene).  Texels arrive decoded
     * (BCn through TexStorage::Fetch); YCoCg-coded colour textures (TEX_YCOCG_BIT in the handle, produced when texture
     * compression is on) are converted on the device after the fetch. */
    const rc_texture *textures;
    uint32_t texture_count;
    /* environment map sampling (environment_t, Core.h:393-410): rotations in radians and the importance-sampling
     * quad-tree built by Cpu::Scene::PrepareEnvMapQTree_nolock (SceneCPU.cpp:1058-1211): level i is an array of
     * 4^(qtree_levels-1-i) fvec4 (four quadrant luminances each), exactly environment_t::qtree_mips[i] */
    int32_t qtree_levels;
    float env_map_rotation, back_map_rotation;
    const float *qtree_mips[16];
} rc_scene_view;

/* camera_t (reference Types.h:102-115) + pass_settings_t (Types.h:92-100), flattened to 32-bit fields. */
typedef struct rc_camera {
    uint32_t type;   /* eCamType: Persp (0) or Geo (2, see rc_pass_desc); Ortho (1) is not supported */
    uint32_t filter; /* ePixelFilter */
    uint32_t view_transform; /* eViewTransform: Standard (0), or 1..9 (AgX / Filmic) after rc_set_view_lut */
    float fov, exposure, gamma, sensor_height;
    float focus_distance, focal_length, fstop, lens_rotation, lens_ratio;
    int32_t lens_blades;
    float clip_start, clip_end;
    float origin[3], fwd[3], side[3], up[3], shift[2];
    uint32_t max_diff_depth, max_spec_depth, max_refr_depth, max_transp_depth, max_total_depth;
    uint32_t min_total_depth, min_transp_depth;
    float clamp_direct, clamp_indirect;
    int32_t min_samples;
    float variance_threshold;
    float regularize_alpha;
} rc_camera;

typedef struct rc_rect {
    int32_t x, y, w, h;
} rc_rect;

/* Pass flags (rc_pass_desc::flags).  The reference-side binding maps ePassFlags onto the last five by name.
 *
 * Call the first surface a camera (or Geo) ray hits S.  The flags apply to every camera type; the rc_stage_* entry
 * points ignore them.
 *   RC_RENDER_SKIP_DIRECT     drops light reaching S in one segment: the bounce-0 shadow rays are not traced and the
 *                             shading of bounce 1 adds no colour (emission, light hit, miss term).  Bounce-1 rays
 *                             still continue.
 *   RC_RENDER_SKIP_INDIRECT   keeps S's shadow-ray light and the bounce-1 colour, drops everything after: the bounce
 *                             loop ends after the bounce-1 shading and the bounce-1 shadow rays are not traced.
 *   RC_RENDER_LIGHTING_ONLY   at S the material's base colour (value x base texture) is white for shading; the
 *                             base-colour AOV still records the real colour.
 *   RC_RENDER_NO_BACKGROUND   camera rays that miss contribute (0,0,0) (their alpha is 0 already).
 *   S's own emission (E0) is never dropped.  So, with the same seeds, per pixel and sample: full + E0_only ==
 *   SKIP_INDIRECT + SKIP_DIRECT up to fp32 summation order, where E0_only sets both SKIP flags.
 *   A light that casts no shadow adds its light at the surface it lights straight into that surface's colour, with no
 *   shadow ray, so it cannot be told from emission there: rc_render refuses SKIP_DIRECT, SKIP_INDIRECT and OUTPUT_SH
 *   (with rc_last_error) on a scene whose sampled lights include one with cast_shadow = 0.
 *   RC_RENDER_OUTPUT_SH       also accumulates L1 spherical harmonics of the light arriving at S (RC_BUF_SH_*): per
 *                             sample, the shadow-ray light of S (D) along the bounce-0 shadow-ray direction and
 *                             everything that came back through the bounce-1 ray (I) along that ray's direction,
 *                             sum of L * Y_k(w) with real SH in world space Y = {0.282095, 0.488603 w.y,
 *                             0.488603 w.z, 0.488603 w.x}, times 2^exposure, kept as the same running mean as
 *                             RC_BUF_FULL.  E0 is excluded, so where E0 = 0 coefficient 0 = 0.282095 * RAW rgb. */
enum { RC_RENDER_ASYNC = 1 /* do not synchronise before returning; call rc_sync */,
       RC_RENDER_NO_SORT = 2 /* skip the results-neutral inter-bounce ray sort */,
       RC_RENDER_SKIP_DIRECT = 4, RC_RENDER_SKIP_INDIRECT = 8, RC_RENDER_LIGHTING_ONLY = 16,
       RC_RENDER_NO_BACKGROUND = 32, RC_RENDER_OUTPUT_SH = 64 };

/* Geo camera (cam.type == 2): lightmap baking of one mesh instance.  geo_instance names the instance, and
 * [geo_tri_first, geo_tri_first + geo_tri_count) the global triangle range of its mesh; they are read only for a Geo
 * camera and must lie inside the uploaded mesh_instances / tri_materials.  Ortho (1) is not supported.
 *
 * Texel (x, y) of the w x h frame covers texture coordinates [x, x+1) x [y, y+1) in texel units s = u*w, t = v*h,
 * with NO v flip (the convention of the texture fetch, so a baked map binds as a texture of the same mesh as it is).
 * For each active pixel of the rect the sample point is (x + jx, y + jy), (jx, jy) the pixel-filter draw of the
 * perspective ray generator (the filter itself is ignored: box within the texel).  The winner is the LOWEST-indexed
 * triangle of the range whose uv triangle contains the point: all three edge functions >= 0 after orienting by the sign
 * of the uv area, in fp32 texel units, both windings, uvs not wrapped; triangles with |uv area| < 1e-12 texel^2 never
 * win.  A winner emits one ray and its hit with no primary trace: P = xform * interpolated position, N = normalised
 * world-space interpolated vertex normal, ray o = P, d = -N, c = 1, pdf = 1e6, camera depth, empty IOR stack,
 * cone_width = world size of one texel on that triangle, cone_spread = 0; hit obj = geo_instance, prim = the global
 * triangle id (front face), t = 0, u/v = weights of the triangle's 2nd/3rd vertex.  No winner: no ray, and the
 * pixel's sample is 0.  So RAW alpha is the covered fraction of the samples (RGB premultiplied by it), uncovered texels
 * stay 0, AOVs are written for covered samples only (normal N, depth 0), and the rays count as primary_rays.
 * The per-texel candidate lists are built on the device at the first Geo pass and kept until the scene, the range or
 * the frame size changes; a range whose texel-clamped uv boxes add up to more than 2^28 texel entries (1 GiB) is
 * refused. */
typedef struct rc_pass_desc {
    rc_camera cam;
    rc_rect rect;
    int32_t iteration; /* value of RegionContext::iteration AFTER the increment RenderScene does (>= 1) */
    uint32_t flags;
    uint32_t geo_instance, geo_tri_first, geo_tri_count; /* Geo camera only */
} rc_pass_desc;

/* RC_BUF_SH_R/G/B: w x h RGBA32F planes holding the 4 L1 SH coefficients of one colour channel (RC_RENDER_OUTPUT_SH).
 * They exist from the first pass with RC_RENDER_OUTPUT_SH on; rc_clear / rc_resize zero them. */
enum { RC_BUF_FINAL = 0, RC_BUF_RAW = 1, RC_BUF_BASE_COLOR = 2, RC_BUF_DEPTH_NORMALS = 3, RC_BUF_FULL = 4,
       RC_BUF_HALF = 5, RC_BUF_TEMP = 6, RC_BUF_SH_R = 7, RC_BUF_SH_G = 8, RC_BUF_SH_B = 9 };

/* Ray bookkeeping of the last rc_render calls since rc_reset_stats: what Mrays/s is computed from. */
typedef struct rc_counters {
    uint64_t primary_rays;
    uint64_t secondary_rays; /* sum over bounces of the rays handed to the closest-hit trace */
    uint64_t shadow_rays;
    uint64_t nodes_visited;  /* BVH8 inner nodes box-tested (closest + shadow) */
    uint64_t leaves_tested;  /* 8-triangle blocks tested */
    uint64_t samples;        /* rc_render calls */
} rc_counters;

int rc_device_count(void);
int rc_create(int device, rc_ctx **out_ctx);
void rc_destroy(rc_ctx *ctx);
const char *rc_last_error(const rc_ctx *ctx);
const char *rc_device_name(const rc_ctx *ctx);

int rc_resize(rc_ctx *ctx, int w, int h);
int rc_clear(rc_ctx *ctx, const float rgba[4]);

/* pmj: dims*samples*2 uint32 (dims must be 32, samples 4096).  filter_table may be NULL (Box filter). */
int rc_upload_tables(rc_ctx *ctx, const uint32_t *pmj, int dims, int samples, const float *filter_table,
                     int filter_table_size);
int rc_upload_scene(rc_ctx *ctx, const rc_scene_view *scene);

int rc_render(rc_ctx *ctx, const rc_pass_desc *pass);
int rc_sync(rc_ctx *ctx);
/* RendererBase::DenoiseImage(const RegionContext &) (internal/RendererCPU.h:661-787): joint NLM filter (7x7 window,
 * 3x3 patches, base-colour and depth-normals features) of the accumulated image inside `rect`; writes the filtered
 * linear image to RC_BUF_RAW and its tonemapped version to RC_BUF_FINAL, updates required-samples.  Uses the variance
 * threshold and gamma of the last rc_render; `iteration` = RegionContext::iteration.  Blocking. */
int rc_denoise_nlm(rc_ctx *ctx, const rc_rect *rect, int iteration);
/* RendererBase::DenoiseImage(int pass, const RegionContext &) / InitUNetFilter (internal/RendererCPU.h:790-1007,
 * :1261-1279): the 16-pass UNet denoiser over the accumulated colour, base-colour and normal planes.
 * rc_unet_set_weights: the 16 convolutions in pass order (enc_conv0, enc_conv1..4, enc_conv5a, enc_conv5b, dec_conv4a,
 *   dec_conv4b, dec_conv3a, dec_conv3b, dec_conv2a, dec_conv2b, dec_conv1a, dec_conv1b, dec_conv0), each as fp16 OIHW
 *   weights [cout][cin][3][3] + fp16 biases [cout] -- the layout of OIDN's weight blobs the reference embeds
 *   (internal/precomputed/__oidn_weights_hdr_alb_nrm.inl).  Channel counts are checked against the network's shape.
 * rc_denoise_unet: pass 0..15 runs that pass over `rect` (frame coordinates), pass -1 runs all 16.  Passes < 15
 *   compute at least `rect` rounded outward to the 16-pixel grid of the frame (origin down, end up to a multiple of 16)
 *   and may compute more of their tensor; pass 15 writes exactly the pixels of `rect`.  To filter a frame region by
 *   region, call pass k for every region of a partition of the frame before pass k + 1 (pass-major): the regions of a
 *   pass then write the whole intermediate tensor the next pass reads.  Pass 15 writes the filtered linear image to
 *   RC_BUF_RAW and its tonemapped version to RC_BUF_FINAL.  flags: RC_UNET_TENSOR_CORES (default path) computes the
 *   convolutions in fp16 on the tensor cores with fp32 accumulation, RC_UNET_FP32 in fp32 FFMA (the parity anchor).
 *   Blocking. */
typedef struct rc_unet_layer {
    const uint16_t *weights; /* fp16 bits, cout * cin * 9 */
    const uint16_t *bias;    /* fp16 bits, cout */
    int32_t cin, cout;
} rc_unet_layer;
enum { RC_UNET_TENSOR_CORES = 0, RC_UNET_FP32 = 1 };
int rc_unet_set_weights(rc_ctx *ctx, const rc_unet_layer layers[16]);
int rc_denoise_unet(rc_ctx *ctx, int pass, const rc_rect *rect, uint32_t flags);

/* Incremental scene update for animated instance transforms (reference: Cpu::Scene::SetMeshInstanceTransform ->
 * RebuildTLAS_nolock, SceneCPU.cpp:884-905 / 1021-1056): re-reads from `scene` ONLY the top-level nodes
 * wnodes[first_tlas_node ..), mesh_instances, lights, light_cwnodes, the light counts, tlas_root and the bounds; every
 * other array (BLAS nodes below first_tlas_node, triangles, vertices, materials, textures, environment) is taken to be
 * what the last rc_upload_scene got and is neither read nor copied.  The node count may differ from the uploaded one
 * (a rebuilt top level rarely has the same size); the instance count may not.  Blocking. */
int rc_update_instances(rc_ctx *ctx, const rc_scene_view *scene, uint32_t first_tlas_node);
/* AgX / Filmic view transforms (reference: TonemapFilmic, TonemapRef.cpp:29-66): hands over the 48^3 table of packed
 * 10-10-10-2 colours for eViewTransform value `view_transform` (1..15; Ray::transform_luts[] in the reference tree --
 * the tables are reference data and are not part of this library).  lut = NULL drops the table.  rc_render with
 * cam.view_transform != 0 fails unless its table was set.  The denoisers use the transform of the last rc_render. */
int rc_set_view_lut(rc_ctx *ctx, uint32_t view_transform, const uint32_t *lut, int dims /* 48 */);

/* Cumulative host->device bytes rc_upload_scene and rc_update_instances have copied on this context. */
uint64_t rc_scene_upload_bytes(const rc_ctx *ctx);

/* Device build of a binary BVH over n primitive boxes (the fast builder of SURVEY.md section 8(f) row 4; reference:
 * PreprocessPrims_HLBVH, internal/Core.cpp:574-720): Morton order of the box centroids, Karras' parallel radix tree,
 * bottom-up box fit.  boxes: n x {min xyz, max xyz}.  nodes_out: 2n - 1 records {min[3], max[3], left, right, first,
 * count}: internal nodes 0 .. n-2 (root 0, count 0, children = node indices), leaves n-1 .. 2n-2 (count 1, first = rank
 * in Morton order).  order_out[rank] = index of the primitive.  n >= 2.  Blocking; all buffers are the caller's (host). */
typedef struct rc_lbvh_node {
    float mn[3], mx[3];
    uint32_t left, right, first, count;
} rc_lbvh_node;
int rc_build_lbvh(rc_ctx *ctx, const float *boxes, uint32_t n, rc_lbvh_node *nodes_out, uint32_t *order_out);

/* dst: rect.w*rect.h RGBA float pixels written with the given pitch (in pixels). */
int rc_readback(rc_ctx *ctx, int which, const rc_rect *rect, float *dst, int pitch);
int rc_readback_required_samples(rc_ctx *ctx, uint16_t *dst);

int rc_enable_stats(rc_ctx *ctx, int enable);
int rc_get_stats(rc_ctx *ctx, uint64_t us[11]); /* order of RendererBase::stats_t */
int rc_get_counters(rc_ctx *ctx, rc_counters *out);
int rc_reset_stats(rc_ctx *ctx);
/* device-side time (ms, CUDA events on the context stream) of each kernel family accumulated since rc_reset_stats:
 * [0] raygen [1] trace_closest [2] shade [3] trace_shadow [4] sort [5] resolve */
int rc_get_kernel_ms(rc_ctx *ctx, double ms[6], uint64_t launches[6]);

/* ---- helpers for callers that time or stage data themselves ---- */
/* pinned (page-locked) host memory for readback mirrors / staging; NULL on failure */
void *rc_host_alloc(size_t bytes);
void rc_host_free(void *p);
/* device address of a frame buffer plane (RC_BUF_*), for zero-copy consumers in the same process (e.g. an NCCL gather
 * of the accumulated image); the plane is w*h RGBA float, row pitch = w pixels */
void *rc_device_ptr(rc_ctx *ctx, int which);
/* user timing events on the context's stream: slot 0..7 */
int rc_event_record(rc_ctx *ctx, int slot);
int rc_event_elapsed_ms(rc_ctx *ctx, int slot_a, int slot_b, float *ms);

/* asynchronous variant of rc_readback: enqueues the 2-D copy on the context's stream and returns; `dst` should be
 * page-locked (rc_host_alloc) for the copy to overlap; complete after rc_sync */
int rc_readback_async(rc_ctx *ctx, int which, const rc_rect *rect, float *dst, int pitch);

/* ---- multi-GPU (SURVEY.md section 8(b)/(e)): one process, one rc_ctx per device, the frame sharded in row strips ----
 * A communicator groups n contexts that were sized (rc_resize) to the SAME full frame and hold the same scene and
 * tables.  The rows of the frame are owned by a fixed device: band r = rc_comm_strip({0,0,W,H}, n, r) (heights differ
 * by <= 1 row), because a pixel's running means must keep accumulating where their history lives.  rc_comm_render
 * intersects pass->rect with every band, enqueues one sample of each non-empty piece on its device and, unless
 * RC_RENDER_ASYNC is set, waits for all of them.  There is no inter-bounce communication: a pixel depends only on
 * (x, y, iteration, scene).
 * rc_gather   : every device copies ITS rows of plane `which` inside `rect` (NULL = the rect of the last
 *               rc_comm_render) straight into the caller's host image (dst = top-left pixel of `rect`, pitch in
 *               pixels), n PCIe links in parallel; `dst` should be page-locked (rc_host_alloc).  Blocking.
 * rc_gather_device : peer copies (NVLink) of the other devices' rows into ctxs[0]'s plane, so device 0 holds the whole
 *               rect (for a consumer on the device: denoiser, display).  Blocking. */
typedef struct rc_comm rc_comm;
int rc_comm_init(rc_ctx **ctxs, int n, rc_comm **out_comm);
void rc_comm_destroy(rc_comm *comm);
const char *rc_comm_last_error(const rc_comm *comm);
/* strip of `rect` owned by context `rank` of an n-context communicator */
int rc_comm_strip(const rc_rect *rect, int n, int rank, rc_rect *out);
int rc_comm_upload_scene(rc_comm *comm, const rc_scene_view *scene);
int rc_comm_upload_tables(rc_comm *comm, const uint32_t *pmj, int dims, int samples, const float *filter_table,
                          int filter_table_size);
int rc_comm_render(rc_comm *comm, const rc_pass_desc *pass);
int rc_comm_sync(rc_comm *comm);
int rc_gather(rc_comm *comm, int which, const rc_rect *rect, float *dst, int pitch);
int rc_gather_device(rc_comm *comm, int which, const rc_rect *rect);
int rc_comm_get_counters(rc_comm *comm, rc_counters *out); /* summed over the devices */

/* ---- stage entry points (host AoS buffers in the reference's layouts; see header comment) ---- */
/* rays_out: ray_data_t[rect.w*rect.h] (72 B), hits_out: hit_data_t[...] (20 B); *count_out = rays generated. */
int rc_stage_generate_primary_rays(rc_ctx *ctx, const rc_pass_desc *pass, void *rays_out, void *hits_out,
                                   int *count_out);
/* the same for a Geo camera (pass->cam.type == 2): the rays and hit records of the covered texels; like a Geo pass of
 * rc_render it also writes 0 into the RC_BUF_TEMP pixels of the uncovered texels */
int rc_stage_generate_geo_rays(rc_ctx *ctx, const rc_pass_desc *pass, void *rays_out, void *hits_out, int *count_out);
/* rays: in/out (transparency updates c/depth), hits: in/out.  trace_lights != 0 adds IntersectAreaLights. */
int rc_stage_trace_rays(rc_ctx *ctx, const rc_pass_desc *pass, void *rays, void *hits, int count, int trace_lights);
/* primary != 0: ShadePrimary (stores colour, updates AOVs) else ShadeSecondary (adds).  bounce selects the clamp as
 * RenderScene does.  Outputs are unordered (append order is not the reference's); compare by pixel key `xy`. */
int rc_stage_shade(rc_ctx *ctx, const rc_pass_desc *pass, int primary, int bounce, const void *rays, const void *hits,
                   int count, void *secondary_out, int *secondary_count, void *shadow_out, int *shadow_count);
/* adds the shadow rays' contribution into the TEMP buffer (read it back with rc_readback(RC_BUF_TEMP)) */
int rc_stage_trace_shadow_rays(rc_ctx *ctx, const rc_pass_desc *pass, const void *shadow_rays, int count,
                               float clamp_val);
/* results-neutral: reorders rays in place by the reference's ray hash; returns the hash of each output ray */
int rc_stage_sort_rays(rc_ctx *ctx, void *rays, int count, uint32_t *hashes_out);
/* overwrite the TEMP buffer (stage tests) */
int rc_debug_fill_temp(rc_ctx *ctx, const float rgba[4]);
/* overwrite frame plane `which` (RC_BUF_FINAL .. RC_BUF_TEMP; not an SH plane) with w*h RGBA floats from `src`, e.g. to
 * feed the UNet synthetic colour / base-colour / depth-normals planes without rendering */
int rc_debug_write_plane(rc_ctx *ctx, int which, const float *src);
/* read back an intermediate tensor of the UNet path `flags` selects (RC_UNET_FP32 or RC_UNET_TENSOR_CORES), exactly as
 * stored.  tensor 0..14: output of pass `tensor`; 15: the network input of the tensor-core path (9 features).
 * dims = {rows, cols, channel stride} of the stored layout:
 *   fp32 path:        (hr >> s, wr >> s, cout) with wr x hr the frame rounded up to 16 and s the tensor's down-scale
 *   tensor-core path: (H + 2, W + 2, Cs) with the one-pixel zero border and the channel stride padded to 64; W x H is
 *                     the stored grid, twice the level's grid for a tensor stored already up-sampled for the next pass
 * Rows [row0, row0 + nrows) of that layout go to `dst` as floats (fp16 converted exactly); with dst == NULL only `dims`
 * is filled.  Refused when the path has not run at the current rounded frame size, or tensor / rows are out of range. */
int rc_debug_unet_tensor(rc_ctx *ctx, uint32_t flags, int tensor, int row0, int nrows, float *dst, int32_t dims[3]);
/* sizeof() of the ABI structs as compiled into the library: 0 rc_array, 1 rc_scene_view, 2 rc_camera, 3 rc_rect,
 * 4 rc_pass_desc, 5 rc_counters; -1 for an unknown id.  Lets a binding verify its struct mirrors. */
int rc_abi_sizeof(int which);

#ifdef __cplusplus
}
#endif
#endif /* RAY_CUDA_H */
