// ray_cuda.cu -- implementation of the C-ABI in include/ray_cuda.h (libray_cuda.so).
//
// Owns the device context: scene arrays, PMJ/filter tables, frame buffers, ray/hit/shadow streams, counters, and the
// per-sample kernel sequence that stands in for Cpu::Renderer<P>::RenderScene (reference internal/RendererCPU.h:374-659).
// There is no CPU fallback anywhere in this file: every entry point either runs the sm_100a kernels or fails.
#include "../../include/ray_cuda.h"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include <cuda_runtime.h>
#include <cub/device/device_scan.cuh>

#include "dev_buf.h"
#include "rt_kernels.cuh"
#include "rt_bake.cuh"
#include "rt_trace.cuh"
#include "rt_sort.cuh"
#include "rt_denoise.cuh"
#include "rt_unet.cuh"
#include "rt_unet_tc.cuh"
#include "rt_lbvh.cuh"

using namespace rt;

namespace {

enum { EV_START = 0, EV_RAYGEN, EV_PTRACE, EV_PSHADE, EV_PSHADOW, EV_BOUNCE0 };
constexpr int kEventsPerBounce = 4; // sort, trace, shade, shadow
constexpr int EV_END = EV_BOUNCE0 + kEventsPerBounce * kMaxBounces;
constexpr int EV_SH1 = EV_END + 2, EV_SH2 = EV_END + 3; // after k_sh_primary / k_sh_direct (RC_RENDER_OUTPUT_SH)
constexpr int kMaxEvents = EV_END + 4;
enum { KF_RAYGEN = 0, KF_TRACE, KF_SHADE, KF_SHADOW, KF_SORT, KF_RESOLVE, KF_COUNT };

struct DevArray {
    DevBuf<uint8_t> buf;
    size_t bytes = 0;
    uint32_t count = 0;

    void *ptr() const { return buf.get(); }
    // A non-empty array whose size did not change keeps its block (the common re-upload: animated transforms, edited
    // materials): a free and a new allocation cost milliseconds and synchronise the device.
    bool fits(size_t new_bytes) const { return buf.get() && new_bytes != 0 && bytes == new_bytes; }
    // Sizes the array for `new_bytes` bytes of `new_count` records, contents undefined.  An empty array is a 256-byte
    // placeholder, so kernels can form (never dereferenced) addresses.
    cudaError_t resize(size_t new_bytes, uint32_t new_count) {
        if (!fits(new_bytes)) {
            bytes = count = 0;
            const cudaError_t e = buf.alloc(new_bytes ? new_bytes : 256);
            if (e != cudaSuccess) {
                return e;
            }
        }
        bytes = new_bytes;
        count = new_count;
        return cudaSuccess;
    }
};

} // namespace

struct rc_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaDeviceProp prop{};
    std::string last_error;
    std::string device_name;
    int num_sms = 0;

    int w = 0, h = 0;
    // fb / rays / hits / shadow are the kernels' views of the per-pixel blocks owned by the DevBufs after them, which
    // rc_resize allocates
    FrameBufs fb{};
    RayBuf rays[2]{};
    HitBuf hits{};
    ShadowBuf shadow{};
    DevBuf<float4> fb_planes[7]; // temp, full, half, raw, final, base_color, depth_normals
    DevBuf<uint16_t> fb_required_samples;
    DevBuf<float4> ray_planes[2][4]; // o_cw, d_cs, c_pdf, ior of each list
    DevBuf<uint2> ray_xy_depth[2];
    DevBuf<float4> hit_tuvp;
    DevBuf<int> hit_obj;
    DevBuf<float4> shadow_planes[3]; // o_depth, d_dist, c_xy
    SortBufs sort{};
    size_t ray_capacity = 0;

    DevBuf<uint32_t> d_counters;
    DevBuf<unsigned long long> d_totals;
    DevBuf<uint32_t> d_pmj;
    DevBuf<float> d_filter_table;
    bool have_tables = false;

    DevArray wnodes, mtris, tri_indices, tri_materials, materials, mesh_instances, vertices, vtx_indices, lights,
        light_cwnodes;
    DevArray tex_descs, tex_texels, qtree;
    DevArray dnodes, blas_roots, dmtris; // device-built traversal copies (rt_trace.cuh)
    uint32_t tlas_root_word = kEmptyChild;
    int trace_fin_min = 32;         // lanes of a warp that must have finished before their epilogue + refill is issued
    // UNet denoiser (rt_unet.cuh): weights as uploaded + the 15 intermediate tensors of the current frame size
    DevBuf<float> unet_w[kUNetLayers], unet_b[kUNetLayers];
    DevBuf<float> unet_t[15];
    int unet_tw = 0, unet_th = 0; // rounded frame the tensors were sized for
    bool unet_ready = false;
    // tensor-core path (rt_unet_tc.cuh): fp16 weights [9][n][in_cs], fp32 biases [n], bordered fp16 tensors
    DevBuf<__half> unet_hw[kUNetLayers];
    DevBuf<float> unet_hb[kUNetLayers];
    DevBuf<__half> unet_ht[15], unet_hx0, unet_hs;
    int unet_htw = 0, unet_hth = 0;
    void *tensor_map_encode = nullptr; // cuTensorMapEncodeTiled through cudaGetDriverEntryPoint
    DevBuf<float4> nlm_scratch; // 3 planes of the largest region denoised so far (rt_denoise.cuh)
    DevBuf<uint32_t> d_view_lut[16]; // AgX / Filmic view-transform tables by eViewTransform (rc_set_view_lut)
    DisplayXf last_xf{nullptr, 1.0f}; // tonemap_params_ of the reference: what the denoisers' display transform uses
    float last_variance_threshold = 0.0f; // tonemap_params_ / variance_threshold_ of the reference
    SceneEnv env{};
    DevBuf<float> d_srgb_lut;
    bool have_scene = false;
    rc_scene_view scene_info{};
    uint32_t li_count = 0;
    bool no_shadow_lights = false; // a light NEE samples casts no shadow (see rc_render)
    uint64_t scene_h2d_bytes = 0; // host->device bytes rc_upload_scene / rc_update_instances have copied so far
    std::map<uint32_t, uint32_t> tex_dense; // (storage << 28 | index) -> dense texture id of the uploaded scene

    // Geo camera candidate lists (rt_bake.cuh) of one (scene upload, triangle range, frame size)
    DevBuf<uint32_t> geo_offsets, geo_cursor, geo_list; // geo_list only grows
    bool geo_valid = false;
    uint32_t geo_first = 0, geo_count = 0;
    // L1 SH planes (RC_BUF_SH_*) + per-sample scratch, allocated by the first RC_RENDER_OUTPUT_SH pass; `sh` is the
    // kernels' view of sh_planes
    ShPlanes sh{};
    DevBuf<float4> sh_planes[7]; // coef[0..2], e0, direct, dir0, dir1
    bool have_sh = false;
    uint32_t sample_tag = 0;

    bool stats_enabled = true;
    std::vector<cudaEvent_t> events;
    cudaEvent_t user_events[10] = {}; // 0..7: rc_event_record slots, 8..9: rc_denoise_nlm timing
    bool sample_pending = false;
    int pending_bounces = 0;
    bool pending_sh = false;
    uint64_t stats_us[11] = {};
    double kernel_ms[KF_COUNT] = {};
    uint64_t kernel_launches[KF_COUNT] = {};
};

namespace {

int fail(rc_ctx *ctx, const char *fmt, ...) {
    char buf[1024];
    va_list vl;
    va_start(vl, fmt);
    vsnprintf(buf, sizeof(buf), fmt, vl);
    va_end(vl);
    if (ctx) {
        ctx->last_error = buf;
    }
    return 1;
}

#define CU_CHECK(ctx, call)                                                                                            \
    do {                                                                                                               \
        const cudaError_t _e = (call);                                                                                 \
        if (_e != cudaSuccess) {                                                                                       \
            return fail(ctx, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__);              \
        }                                                                                                              \
    } while (0)

// (Re)allocates `own` for n elements and points the kernel-side view `view` at it (null while it has no block).
template <typename T> int alloc_view(rc_ctx *ctx, DevBuf<T> &own, T *&view, size_t n) {
    view = nullptr;
    CU_CHECK(ctx, own.alloc(n));
    view = own.get();
    return 0;
}

int upload_array(rc_ctx *ctx, DevArray &dst, const rc_array &src, uint32_t expected_stride, const char *name) {
    if (src.count != 0 && src.stride != expected_stride) {
        return fail(ctx, "rc_upload_scene: %s stride %u != %u", name, src.stride, expected_stride);
    }
    const size_t new_bytes = size_t(src.count) * expected_stride;
    if (new_bytes != 0 && !src.ptr) {
        return fail(ctx, "rc_upload_scene: %s has count %u but a null pointer", name, src.count);
    }
    CU_CHECK(ctx, dst.resize(new_bytes, src.count));
    if (new_bytes == 0) {
        CU_CHECK(ctx, cudaMemsetAsync(dst.ptr(), 0, 256, ctx->stream));
        return 0;
    }
    CU_CHECK(ctx, cudaMemcpyAsync(dst.ptr(), src.ptr, dst.bytes, cudaMemcpyHostToDevice, ctx->stream));
    ctx->scene_h2d_bytes += dst.bytes;
    return 0;
}

// murmur3 finaliser on the host (reference CoreRef.h:133-141) for rand_seed = hash((iteration - 1) / 4096)
uint32_t host_hash(uint32_t x) {
    x ^= x >> 16;
    x *= 0x85ebca6bu;
    x ^= x >> 13;
    x *= 0xc2b2ae35u;
    x ^= x >> 16;
    return x;
}

int host_popcount(unsigned x) {
    int c = 0;
    for (; x != 0; x &= x - 1) {
        c++;
    }
    return c;
}

int fill_params(rc_ctx *ctx, const rc_pass_desc *pass, KParams &p) {
    if (!ctx->have_scene) {
        return fail(ctx, "no scene uploaded");
    }
    if (!ctx->have_tables) {
        return fail(ctx, "no sampler table uploaded (rc_upload_tables)");
    }
    if (ctx->w == 0 || ctx->h == 0) {
        return fail(ctx, "frame buffer has zero size (rc_resize)");
    }
    const rc_camera &c = pass->cam;
    if (c.type != 0 && c.type != 2) {
        return fail(ctx, "camera type %u is not supported by the CUDA backend (Persp and Geo only)", c.type);
    }
    if (c.type == 2) {
        if (pass->geo_instance >= ctx->mesh_instances.count) {
            return fail(ctx, "Geo camera: mesh instance %u outside the %u uploaded", pass->geo_instance,
                        ctx->mesh_instances.count);
        }
        const uint64_t end = uint64_t(pass->geo_tri_first) + pass->geo_tri_count;
        if (end > ctx->tri_materials.count || 3 * end > ctx->vtx_indices.count) {
            return fail(ctx, "Geo camera: triangle range [%u, %llu) outside the %u uploaded triangles", pass->geo_tri_first,
                        (unsigned long long)end, ctx->tri_materials.count);
        }
        if (uint64_t(ctx->w) * ctx->h >= (1ull << 31)) {
            return fail(ctx, "Geo camera: a %dx%d lightmap has more than 2^31 texels", ctx->w, ctx->h);
        }
    }
    if (c.view_transform != 0 && (c.view_transform >= 16 || !ctx->d_view_lut[c.view_transform].get())) {
        return fail(ctx, "view transform %u needs its table (rc_set_view_lut)", c.view_transform);
    }
    if (c.filter != 0 && !ctx->d_filter_table.get()) {
        return fail(ctx, "pixel filter %u needs a filter table (rc_upload_tables)", c.filter);
    }
    if (c.max_total_depth + 1 >= uint32_t(kMaxBounces)) {
        return fail(ctx, "max_total_depth %u exceeds the backend limit %d", c.max_total_depth, kMaxBounces - 2);
    }
    const rc_rect &r = pass->rect;
    if (r.x < 0 || r.y < 0 || r.w <= 0 || r.h <= 0 || r.x + r.w > ctx->w || r.y + r.h > ctx->h) {
        return fail(ctx, "rect (%d,%d,%d,%d) is outside the %dx%d frame", r.x, r.y, r.w, r.h, ctx->w, ctx->h);
    }
    if (pass->iteration < 1) {
        return fail(ctx, "iteration must be >= 1");
    }

    memset(&p, 0, sizeof(p));
    p.sc.geo.nodes = static_cast<const WNode *>(ctx->wnodes.ptr());
    p.sc.geo.dnodes = static_cast<const WNode *>(ctx->dnodes.ptr());
    p.sc.geo.blas_roots = static_cast<const uint32_t *>(ctx->blas_roots.ptr());
    p.sc.geo.dmtris = ctx->dmtris.ptr();
    p.sc.geo.tlas_root_word = ctx->tlas_root_word;
    p.sc.geo.mtris = static_cast<const MTri *>(ctx->mtris.ptr());
    p.sc.geo.tri_indices = static_cast<const uint32_t *>(ctx->tri_indices.ptr());
    p.sc.geo.tri_materials = static_cast<const TriMat *>(ctx->tri_materials.ptr());
    p.sc.geo.instances = static_cast<const MeshInstance *>(ctx->mesh_instances.ptr());
    p.sc.geo.tlas_root = ctx->scene_info.tlas_root;
    p.sc.surf.vertices = static_cast<const Vertex *>(ctx->vertices.ptr());
    p.sc.surf.vtx_indices = static_cast<const uint32_t *>(ctx->vtx_indices.ptr());
    p.sc.surf.materials = static_cast<const Material *>(ctx->materials.ptr());
    p.sc.tex.descs = ctx->tex_descs.count ? static_cast<const TexDesc *>(ctx->tex_descs.ptr()) : nullptr;
    p.sc.tex.texels = static_cast<const uint32_t *>(ctx->tex_texels.ptr());
    p.sc.tex.srgb_lut = ctx->d_srgb_lut.get();
    p.sc.lights.env = ctx->env;
    p.sc.lights.env.qtree = static_cast<const float4 *>(ctx->qtree.ptr());
    p.sc.lights.lights = static_cast<const Light *>(ctx->lights.ptr());
    p.sc.lights.nodes = static_cast<const LightCWNode *>(ctx->light_cwnodes.ptr());
    p.sc.lights.nodes_count = ctx->light_cwnodes.count;
    p.sc.lights.visible_lights_count = ctx->scene_info.visible_lights_count;
    p.sc.lights.blocker_lights_count = ctx->scene_info.blocker_lights_count;
    p.sc.lights.env_light_index = ctx->scene_info.env_light_index;
    for (int i = 0; i < 3; ++i) {
        p.sc.lights.env_col[i] = ctx->scene_info.env_col[i];
        p.sc.lights.back_col[i] = ctx->scene_info.back_col[i];
    }
    p.sc.rand_seq = ctx->d_pmj.get();
    p.sc.li_count = ctx->li_count;

    p.ps.max_diff_depth = int(c.max_diff_depth);
    p.ps.max_spec_depth = int(c.max_spec_depth);
    p.ps.max_refr_depth = int(c.max_refr_depth);
    p.ps.max_transp_depth = int(c.max_transp_depth);
    p.ps.max_total_depth = int(c.max_total_depth);
    p.ps.min_total_depth = int(c.min_total_depth);
    p.ps.min_transp_depth = int(c.min_transp_depth);
    p.ps.clamp_direct = c.clamp_direct;
    p.ps.clamp_indirect = c.clamp_indirect;
    p.ps.regularize_alpha = c.regularize_alpha;

    // camera-derived constants, computed with the host libm exactly like GeneratePrimaryRays (CoreRef.cpp:1434-1442)
    const float PI = 3.141592653589793238463f;
    p.cam.origin = v3{c.origin[0], c.origin[1], c.origin[2]};
    p.cam.fwd = v3{c.fwd[0], c.fwd[1], c.fwd[2]};
    p.cam.side = v3{c.side[0], c.side[1], c.side[2]};
    p.cam.up = v3{c.up[0], c.up[1], c.up[2]};
    p.cam.shift_x = c.shift[0];
    p.cam.shift_y = c.shift[1];
    p.cam.focus_distance = c.focus_distance;
    p.cam.k = float(ctx->w) / float(ctx->h);
    const float temp = tanf(0.5f * c.fov * PI / 180.0f);
    p.cam.fov_k = temp * c.focus_distance;
    p.cam.spread_angle = atanf(2.0f * temp / float(ctx->h));
    p.cam.fstop = c.fstop;
    p.cam.focal_length = c.focal_length;
    p.cam.sensor_height = c.sensor_height;
    p.cam.lens_rotation = c.lens_rotation;
    p.cam.lens_ratio = c.lens_ratio;
    p.cam.lens_blades = c.lens_blades;
    p.cam.clip_start = c.clip_start;
    p.cam.clip_end = c.clip_end;
    p.cam.filter = int(c.filter);

    p.fb = ctx->fb;
    p.filter_table = ctx->d_filter_table.get();
    p.counters = ctx->d_counters.get();
    p.totals = ctx->d_totals.get();
    p.rect_x = r.x;
    p.rect_y = r.y;
    p.rect_w = r.w;
    p.rect_h = r.h;
    p.iteration = pass->iteration;
    p.rand_seed = host_hash(uint32_t((pass->iteration - 1) / kRandSamples));
    return 0;
}

// Walk the hierarchy the way a ray would (TLAS nodes -> instance -> its BLAS) over the caller's arrays and check what
// the trace kernels rely on: child / instance / triangle-block indices inside their arrays, leaves that fit the
// 27-bit + 4-bit leaf word of rt_trace.cuh.  Only nodes REACHABLE from the TLAS root are looked at: freed SparseStorage
// slots inside the arrays' capacity hold stale bytes.  Shared BLASes are walked once.
int validate_bvh(rc_ctx *ctx, const rc_scene_view *sv) {
    if (sv->tlas_root == 0xffffffffu) {
        return 0;
    }
    const uint32_t n_nodes = sv->wnodes.count, n_inst = sv->mesh_instances.count, n_blocks = sv->mtris.count;
    const WNode *nodes = static_cast<const WNode *>(sv->wnodes.ptr);
    const MeshInstance *inst = static_cast<const MeshInstance *>(sv->mesh_instances.ptr);
    if (sv->tlas_root >= n_nodes) {
        return fail(ctx, "rc_upload_scene: tlas_root %u outside the node array (%u)", sv->tlas_root, n_nodes);
    }
    std::vector<uint8_t> seen(n_nodes, 0); // bit 0: visited as a TLAS node, bit 1: as a BLAS node
    std::vector<std::pair<uint32_t, bool>> stack;
    stack.emplace_back(sv->tlas_root, false);
    while (!stack.empty()) {
        const uint32_t n = stack.back().first;
        const bool blas = stack.back().second;
        stack.pop_back();
        const uint8_t bit = blas ? 2 : 1;
        if (seen[n] & bit) {
            continue;
        }
        seen[n] |= bit;
        const WNode &nd = nodes[n];
        if (nd.child[0] & kLeafBit) {
            const uint32_t first = nd.child[0] & kPrimIndexBits, cnt = nd.child[1];
            if (first >= kLeafFirstBits) {
                return fail(ctx, "rc_upload_scene: leaf %u starts at primitive %u >= 2^27 - 1 (backend limit)", n, first);
            }
            if (!blas) {
                if (first >= n_inst) {
                    return fail(ctx, "rc_upload_scene: TLAS leaf %u names mesh instance %u of %u", n, first, n_inst);
                }
                const uint32_t root = inst[first].node_index;
                if (root >= n_nodes) {
                    return fail(ctx, "rc_upload_scene: mesh instance %u has BLAS root %u outside the node array", first, root);
                }
                stack.emplace_back(root, true);
            } else {
                const uint32_t blocks = ((first & 7u) + cnt + 7u) / 8u;
                if (blocks == 0 || blocks > 16 || first / 8u + blocks > n_blocks) {
                    return fail(ctx, "rc_upload_scene: BLAS leaf %u (first %u, count %u) outside the %u triangle blocks or "
                                     "longer than 128 triangles", n, first, cnt, n_blocks);
                }
            }
            continue;
        }
        for (int c = 0; c < 8; ++c) {
            const uint32_t ch = nd.child[c];
            if (ch == kEmptyChild) {
                continue;
            }
            if (ch >= n_nodes) {
                return fail(ctx, "rc_upload_scene: node %u child %d = %u outside the node array (%u)", n, c, ch, n_nodes);
            }
            stack.emplace_back(ch, blas);
        }
    }
    return 0;
}

// device-side copies the trace kernels walk (rt_trace.cuh): nodes with resolved child words + unhittable empty slots,
// BLAS root word per instance, TLAS root word
int build_traversal_copies(rc_ctx *ctx, const rc_scene_view *sv) {
    const uint32_t n_nodes = sv->wnodes.count, n_inst = sv->mesh_instances.count;
    const uint32_t n_blocks = sv->mtris.count;
    CU_CHECK(ctx, ctx->dnodes.resize(size_t(n_nodes) * sizeof(WNode), n_nodes));
    CU_CHECK(ctx, ctx->blas_roots.resize(size_t(n_inst) * 4, n_inst));
    CU_CHECK(ctx, ctx->dmtris.resize(size_t(n_blocks) * sizeof(MTri), n_blocks));
    if (n_blocks != 0) {
        k_build_dmtris<<<(n_blocks * 4 + 255) / 256, 256, 0, ctx->stream>>>(static_cast<const MTri *>(ctx->mtris.ptr()),
                                                                          static_cast<float4 *>(ctx->dmtris.ptr()), n_blocks);
    }
    ctx->tlas_root_word = kEmptyChild;
    if (validate_bvh(ctx, sv)) {
        return 1;
    }
    if (n_nodes != 0) {
        k_build_dnodes<<<(n_nodes * 8 + 255) / 256, 256, 0, ctx->stream>>>(
            static_cast<const WNode *>(ctx->wnodes.ptr()), static_cast<WNode *>(ctx->dnodes.ptr()), 0u, n_nodes);
    }
    if (n_inst != 0) {
        k_build_blas_roots<<<(n_inst + 255) / 256, 256, 0, ctx->stream>>>(
            static_cast<const WNode *>(ctx->wnodes.ptr()), static_cast<const MeshInstance *>(ctx->mesh_instances.ptr()), n_inst,
            n_nodes, static_cast<uint32_t *>(ctx->blas_roots.ptr()));
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    CU_CHECK(ctx, cudaGetLastError());
    if (sv->tlas_root != 0xffffffffu) {
        if (sv->tlas_root >= n_nodes) {
            return fail(ctx, "rc_upload_scene: tlas_root %u outside the node array (%u)", sv->tlas_root, n_nodes);
        }
        // the root may itself be a leaf (a scene with one instance): read its two words from the caller's array
        const WNode *host_nodes = static_cast<const WNode *>(sv->wnodes.ptr);
        const uint32_t c0 = host_nodes[sv->tlas_root].child[0], c1 = host_nodes[sv->tlas_root].child[1];
        if (c0 & kLeafBit) {
            const uint32_t first = c0 & kPrimIndexBits;
            const uint32_t blocks = ((first & 7u) + c1 + 7u) / 8u;
            if (first >= kLeafFirstBits || blocks == 0 || blocks > 16) {
                return fail(ctx, "rc_upload_scene: the TLAS root leaf cannot be encoded");
            }
            ctx->tlas_root_word = kLeafBit | ((blocks - 1u) << kLeafBlocksShift) | first;
        } else {
            ctx->tlas_root_word = sv->tlas_root;
        }
    }
    return 0;
}

const float4 *plane_of(const rc_ctx *ctx, int which) {
    switch (which) {
    case RC_BUF_FINAL: return ctx->fb.final;
    case RC_BUF_RAW: return ctx->fb.raw;
    case RC_BUF_BASE_COLOR: return ctx->fb.base_color;
    case RC_BUF_DEPTH_NORMALS: return ctx->fb.depth_normals;
    case RC_BUF_FULL: return ctx->fb.full;
    case RC_BUF_HALF: return ctx->fb.half;
    case RC_BUF_TEMP: return ctx->fb.temp;
    case RC_BUF_SH_R:
    case RC_BUF_SH_G:
    case RC_BUF_SH_B: return ctx->have_sh ? ctx->sh.coef[which - RC_BUF_SH_R] : nullptr;
    default: return nullptr;
    }
}

// plane `which` or an error naming why it is missing
int plane_or_fail(rc_ctx *ctx, int which, const char *what, const float4 **out) {
    *out = plane_of(ctx, which);
    if (*out) {
        return 0;
    }
    if (which >= RC_BUF_SH_R && which <= RC_BUF_SH_B) {
        return fail(ctx, "%s: the SH planes exist from the first pass with RC_RENDER_OUTPUT_SH on", what);
    }
    return fail(ctx, "%s: unknown buffer %d", what, which);
}

float clamp_limit(float v) { return (v != 0.0f) ? 3.0f * v : 3.402823466e+38F; }

int persistent_grid(const rc_ctx *ctx, int blocks_per_sm) { return ctx->num_sms * blocks_per_sm; }

// Does next-event estimation sample a light that casts no shadow?  (lights reachable through li_indices; without
// that list every light of the array is looked at)
bool has_no_shadow_lights(const rc_scene_view *sv) {
    const Light *l = static_cast<const Light *>(sv->lights.ptr);
    if (!l || sv->lights.count == 0) {
        return false;
    }
    const uint32_t *li = static_cast<const uint32_t *>(sv->li_indices.ptr);
    const uint32_t n = li ? sv->li_indices.count : sv->lights.count;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t k = li ? li[i] : i;
        if (k < sv->lights.count && ((l[k].bits >> 4) & 1u) == 0) {
            return true;
        }
    }
    return false;
}

void record(rc_ctx *ctx, int ev) {
    if (ctx->stats_enabled) {
        cudaEventRecord(ctx->events[ev], ctx->stream);
    }
}

// fold the event timings of the last enqueued sample into stats_t / per-kernel totals
int harvest_stats(rc_ctx *ctx) {
    if (!ctx->sample_pending || !ctx->stats_enabled) {
        ctx->sample_pending = false;
        return 0;
    }
    ctx->sample_pending = false;
    auto ms = [&](int a, int b) {
        float v = 0.0f;
        cudaEventElapsedTime(&v, ctx->events[a], ctx->events[b]);
        return double(v);
    };
    const double raygen = ms(EV_START, EV_RAYGEN), ptrace = ms(EV_RAYGEN, EV_PTRACE), pshade = ms(EV_PTRACE, EV_PSHADE);
    const double pshadow = ctx->pending_sh ? ms(EV_SH1, EV_PSHADOW) : ms(EV_PSHADE, EV_PSHADOW);
    const double sh = ctx->pending_sh ? ms(EV_PSHADE, EV_SH1) + ms(EV_PSHADOW, EV_SH2) : 0.0;
    double ssort = 0, strace = 0, sshade = 0, sshadow = 0;
    int prev = ctx->pending_sh ? EV_SH2 : EV_PSHADOW;
    for (int b = 0; b < ctx->pending_bounces; ++b) {
        const int e = EV_BOUNCE0 + b * kEventsPerBounce;
        ssort += ms(prev, e + 0);
        strace += ms(e + 0, e + 1);
        sshade += ms(e + 1, e + 2);
        sshadow += ms(e + 2, e + 3);
        prev = e + 3;
    }
    const double resolve = ms(prev, EV_END) + sh;
    ctx->stats_us[0] += uint64_t(raygen * 1000.0);
    ctx->stats_us[1] += uint64_t(ptrace * 1000.0);
    ctx->stats_us[2] += uint64_t(pshade * 1000.0);
    ctx->stats_us[3] += uint64_t(pshadow * 1000.0);
    ctx->stats_us[4] += uint64_t(ssort * 1000.0);
    ctx->stats_us[5] += uint64_t(strace * 1000.0);
    ctx->stats_us[6] += uint64_t(sshade * 1000.0);
    ctx->stats_us[7] += uint64_t(sshadow * 1000.0);
    ctx->kernel_ms[KF_RAYGEN] += raygen;
    ctx->kernel_ms[KF_TRACE] += ptrace + strace;
    ctx->kernel_ms[KF_SHADE] += pshade + sshade;
    ctx->kernel_ms[KF_SHADOW] += pshadow + sshadow;
    ctx->kernel_ms[KF_SORT] += ssort;
    ctx->kernel_ms[KF_RESOLVE] += resolve;
    return 0;
}

// k_shade comes in a textured and an untextured build (all texture branches folded away); the scene decides.
template <bool PRIMARY>
void launch_shade(rc_ctx *ctx, int grid, cudaStream_t s, const KParams &p, RayBuf in, RayBuf out, int bounce, float limit0,
                  float limit1, float mix_factor) {
    if (ctx->tex_descs.count != 0) {
        k_shade<PRIMARY, true><<<grid, RT_SHADE_THREADS, 0, s>>>(p, in, ctx->hits, out, ctx->shadow, bounce, limit0, limit1,
                                                                  mix_factor);
    } else {
        k_shade<PRIMARY, false><<<grid, RT_SHADE_THREADS, 0, s>>>(p, in, ctx->hits, out, ctx->shadow, bounce, limit0,
                                                                   limit1, mix_factor);
    }
}

GeoTarget geo_target(const rc_ctx *ctx, const rc_pass_desc *pass) {
    return GeoTarget{static_cast<const Vertex *>(ctx->vertices.ptr()), static_cast<const uint32_t *>(ctx->vtx_indices.ptr()),
                     pass->geo_tri_first, pass->geo_tri_count, ctx->w, ctx->h};
}

// Build (or reuse) the per-texel candidate lists of a Geo pass (rt_bake.cuh).  Blocking when it builds.
int ensure_geo_lists(rc_ctx *ctx, const rc_pass_desc *pass) {
    if (ctx->geo_valid && ctx->geo_first == pass->geo_tri_first && ctx->geo_count == pass->geo_tri_count) {
        return 0;
    }
    ctx->geo_valid = false;
    cudaStream_t s = ctx->stream;
    const GeoTarget g = geo_target(ctx, pass);
    const size_t n = size_t(ctx->w) * ctx->h;
    if (!ctx->geo_offsets.get()) {
        CU_CHECK(ctx, ctx->geo_offsets.alloc(n + 1));
        CU_CHECK(ctx, ctx->geo_cursor.alloc(n + 1));
    }
    const uint32_t tris = g.tri_count;
    unsigned long long total = 0;
    {
        DevBuf<unsigned long long> d_total;
        CU_CHECK(ctx, d_total.alloc(1));
        cudaMemsetAsync(d_total.get(), 0, sizeof(total), s);
        if (tris != 0) {
            k_geo_box_total<<<(tris + 255) / 256, 256, 0, s>>>(g, d_total.get());
        }
        const cudaError_t e = cudaMemcpyAsync(&total, d_total.get(), sizeof(total), cudaMemcpyDeviceToHost, s);
        cudaStreamSynchronize(s);
        CU_CHECK(ctx, e);
    }
    CU_CHECK(ctx, cudaGetLastError());
    if (total > kGeoMaxEntries) {
        return fail(ctx, "Geo camera: the candidate lists of triangles [%u, %u) at %dx%d would hold %llu entries, more than "
                         "the 2^28 (1 GiB) the backend allows",
                    g.tri_first, g.tri_first + g.tri_count, ctx->w, ctx->h, total);
    }
    if (!ctx->geo_list.get() || total > ctx->geo_list.count()) {
        CU_CHECK(ctx, ctx->geo_list.alloc(size_t(total ? total : 1)));
    }
    CU_CHECK(ctx, cudaMemsetAsync(ctx->geo_cursor.get(), 0, (n + 1) * sizeof(uint32_t), s));
    const int warp_blocks = int(std::min<uint64_t>((uint64_t(tris) * 32 + 255) / 256, uint64_t(ctx->num_sms) * 64));
    if (tris != 0) {
        k_geo_walk<false><<<warp_blocks, 256, 0, s>>>(g, ctx->geo_cursor.get(), nullptr);
    }
    {
        size_t temp_bytes = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, ctx->geo_cursor.get(), ctx->geo_offsets.get(), int(n + 1), s);
        DevBuf<uint8_t> d_temp;
        CU_CHECK(ctx, d_temp.alloc(temp_bytes ? temp_bytes : 16));
        cub::DeviceScan::ExclusiveSum(d_temp.get(), temp_bytes, ctx->geo_cursor.get(), ctx->geo_offsets.get(), int(n + 1), s);
        const cudaError_t e = cudaMemcpyAsync(ctx->geo_cursor.get(), ctx->geo_offsets.get(), n * sizeof(uint32_t),
                                              cudaMemcpyDeviceToDevice, s);
        if (e == cudaSuccess && tris != 0) {
            k_geo_walk<true><<<warp_blocks, 256, 0, s>>>(g, ctx->geo_cursor.get(), ctx->geo_list.get());
        }
        cudaStreamSynchronize(s);
        CU_CHECK(ctx, e);
    }
    CU_CHECK(ctx, cudaGetLastError());
    ctx->geo_first = pass->geo_tri_first;
    ctx->geo_count = pass->geo_tri_count;
    ctx->geo_valid = true;
    return 0;
}

GeoParams geo_params(const rc_ctx *ctx, const rc_pass_desc *pass) {
    return GeoParams{geo_target(ctx, pass), ctx->geo_offsets.get(), ctx->geo_list.get(),
                     static_cast<const MeshInstance *>(ctx->mesh_instances.ptr()) + pass->geo_instance, pass->geo_instance};
}

// the SH planes (zeroed) + scratch at the current frame size
int alloc_sh(rc_ctx *ctx) {
    const size_t n = size_t(ctx->w) * ctx->h;
    ShPlanes &sh = ctx->sh;
    float4 **views[7] = {&sh.coef[0], &sh.coef[1], &sh.coef[2], &sh.e0, &sh.direct, &sh.dir0, &sh.dir1};
    for (int i = 0; i < 7; ++i) {
        if (alloc_view(ctx, ctx->sh_planes[i], *views[i], n)) {
            return 1;
        }
        CU_CHECK(ctx, cudaMemsetAsync(*views[i], 0, n * sizeof(float4), ctx->stream));
    }
    ctx->have_sh = true;
    return 0;
}

// Enqueue the kernels of one sample.
int enqueue_sample(rc_ctx *ctx, const rc_pass_desc *pass, KParams &p) {
    cudaStream_t s = ctx->stream;
    const int max_bounces = p.ps.max_total_depth;
    const bool do_sort = (pass->flags & RC_RENDER_NO_SORT) == 0;
    const bool geo = pass->cam.type == 2;
    const bool skip_direct = (pass->flags & RC_RENDER_SKIP_DIRECT) != 0;
    // RC_RENDER_SKIP_INDIRECT: the bounce loop ends after the bounce-1 shading
    const int last_bounce = (pass->flags & RC_RENDER_SKIP_INDIRECT) ? std::min(1, max_bounces) : max_bounces;
    const bool want_sh = (pass->flags & RC_RENDER_OUTPUT_SH) != 0;
    uint32_t shadow_traced = ~0u;
    if (skip_direct) {
        shadow_traced &= ~1u;
    }
    if (pass->flags & RC_RENDER_SKIP_INDIRECT) {
        shadow_traced &= 1u;
    }
    const uint32_t tag = ++ctx->sample_tag;

    if (ctx->sample_pending && ctx->stats_enabled) {
        // event slots are reused per sample: collect the previous sample's timings first.  Without statistics nothing
        // is harvested and samples queue up back to back (RC_RENDER_ASYNC keeps the GPU fed across samples).
        CU_CHECK(ctx, cudaStreamSynchronize(s));
        harvest_stats(ctx);
    }

    CU_CHECK(ctx, cudaMemsetAsync(ctx->d_counters.get(), 0, CNT_TOTAL * sizeof(uint32_t), s));
    if (do_sort) {
        // k_shade emits sort keys + per-list histograms while it writes the secondary rays
        CU_CHECK(ctx, cudaMemsetAsync(ctx->sort.hist.get(), 0, size_t(max_bounces + 2) * kSortBins * sizeof(uint32_t), s));
        p.sort_grid = SortGrid{ctx->sort.root_min[0], ctx->sort.root_min[1], ctx->sort.root_min[2],
                               ctx->sort.inv_cell[0], ctx->sort.inv_cell[1], ctx->sort.inv_cell[2]};
        p.sort_keys = ctx->sort.keys.get();
        p.sort_hist = ctx->sort.hist.get();
    }
    record(ctx, EV_START);

    const int n_pix_tiles = ((p.rect_w + 7) / 8) * ((p.rect_h + 3) / 4);
    const int raygen_blocks = (n_pix_tiles * 32 + 255) / 256;
    if (geo) {
        k_raygen_geo<<<raygen_blocks, 256, 0, s>>>(p, geo_params(ctx, pass), ctx->rays[0], ctx->hits);
    } else {
        k_raygen<<<raygen_blocks, 256, 0, s>>>(p, ctx->rays[0], ctx->hits);
    }
    ctx->kernel_launches[KF_RAYGEN]++;
    record(ctx, EV_RAYGEN);

    const int trace_grid = persistent_grid(ctx, RT_TRACE_BLOCKS);
    const int shade_grid = persistent_grid(ctx, RT_SHADE_BLOCKS);
    const bool have_geo = ctx->scene_info.tlas_root != 0xffffffffu;

    if (have_geo && !geo) { // k_raygen_geo writes the hit records itself
        k_trace_closest<false, false><<<trace_grid, kTraceThreads, 0, s>>>(p, ctx->rays[0], ctx->hits, 0, ctx->trace_fin_min);
        ctx->kernel_launches[KF_TRACE]++;
    }
    record(ctx, EV_PTRACE);

    const float mix_factor = 1.0f / float(p.iteration);
    {
        const float lim = clamp_limit(p.ps.clamp_direct);
        KParams pp = p;
        pp.flags = (pass->flags & RC_RENDER_LIGHTING_ONLY) ? KP_LIGHTING_ONLY : 0u;
        launch_shade<true>(ctx, shade_grid, s, pp, ctx->rays[0], ctx->rays[1], 0, lim, lim, mix_factor);
        ctx->kernel_launches[KF_SHADE]++;
        if (pass->flags & RC_RENDER_NO_BACKGROUND) {
            k_no_background<<<shade_grid, 256, 0, s>>>(p, ctx->rays[0], ctx->hits);
            ctx->kernel_launches[KF_SHADE]++;
        }
    }
    record(ctx, EV_PSHADE);
    const int n_rect = p.rect_w * p.rect_h;
    const int sh_grid = std::min((n_rect + 255) / 256, ctx->num_sms * 8);
    if (want_sh) { // before the sort of bounce 1 reorders list 1
        k_sh_primary<<<sh_grid, 256, 0, s>>>(p, ctx->sh, ctx->rays[1], tag);
        ctx->kernel_launches[KF_RESOLVE]++;
        record(ctx, EV_SH1);
    }

    if (have_geo && !skip_direct) {
        k_trace_shadow<<<trace_grid, kTraceThreads, 0, s>>>(p, ctx->shadow, 0, clamp_limit(p.ps.clamp_direct), ctx->trace_fin_min);
        ctx->kernel_launches[KF_SHADOW]++;
    }
    record(ctx, EV_PSHADOW);
    if (want_sh) {
        k_sh_direct<<<sh_grid, 256, 0, s>>>(p, ctx->sh, ctx->shadow, tag);
        ctx->kernel_launches[KF_RESOLVE]++;
        record(ctx, EV_SH2);
    }

    int cur = 1; // list index holding the rays of the current bounce
    for (int bounce = 1; bounce <= last_bounce; ++bounce) {
        const int e = EV_BOUNCE0 + (bounce - 1) * kEventsPerBounce;
        if (do_sort) {
            sort_rays(ctx->sort, p, ctx->rays[cur], ctx->rays[cur ^ 1], bounce, ctx->num_sms, /*have_hist*/ true,
                      /*want_sorted_keys*/ false, s);
            cur ^= 1; // the reordered list now lives in the other buffer; the old one is free for this bounce's output
            ctx->kernel_launches[KF_SORT] += 2;
        }
        record(ctx, e + 0);
        if (have_geo) {
            if (ctx->scene_info.visible_lights_count != 0) {
                k_trace_closest<true, true><<<trace_grid, kTraceThreads, 0, s>>>(p, ctx->rays[cur], ctx->hits, bounce, ctx->trace_fin_min);
            } else {
                k_trace_closest<false, true><<<trace_grid, kTraceThreads, 0, s>>>(p, ctx->rays[cur], ctx->hits, bounce, ctx->trace_fin_min);
            }
        } else {
            k_init_hits<<<shade_grid, 128, 0, s>>>(p, ctx->hits, bounce);
        }
        ctx->kernel_launches[KF_TRACE]++;
        record(ctx, e + 1);
        {
            const float cd = (bounce == 1) ? p.ps.clamp_direct : p.ps.clamp_indirect;
            KParams pp = p;
            pp.flags = (bounce == 1 && skip_direct) ? KP_DROP_COL : 0u;
            launch_shade<false>(ctx, shade_grid, s, pp, ctx->rays[cur], ctx->rays[cur ^ 1], bounce, clamp_limit(cd),
                                clamp_limit(p.ps.clamp_indirect), mix_factor);
            ctx->kernel_launches[KF_SHADE]++;
        }
        record(ctx, e + 2);
        if (have_geo && ((shadow_traced >> bounce) & 1u)) {
            k_trace_shadow<<<trace_grid, kTraceThreads, 0, s>>>(p, ctx->shadow, bounce, clamp_limit(p.ps.clamp_indirect), ctx->trace_fin_min);
            ctx->kernel_launches[KF_SHADOW]++;
        }
        record(ctx, e + 3);
        cur ^= 1;
    }

    {
        const float exposure_mul = powf(2.0f, pass->cam.exposure);
        const int is_class_a = host_popcount(uint32_t(p.iteration - 1) & 0xaaaaaaaau) & 1;
        const float half_mix_factor = 1.0f / float((p.iteration + 1) / 2);
        const float inv_gamma = 1.0f / pass->cam.gamma;
        const float vt = p.iteration > pass->cam.min_samples
                             ? 0.5f * pass->cam.variance_threshold * pass->cam.variance_threshold
                             : 0.0f;
        const DisplayXf xf{pass->cam.view_transform ? ctx->d_view_lut[pass->cam.view_transform].get() : nullptr, inv_gamma};
        if (want_sh) { // reads temp before k_resolve overwrites it with the variance
            k_sh_resolve<<<(n_rect + 255) / 256, 256, 0, s>>>(p, ctx->sh, tag, exposure_mul, mix_factor);
            ctx->kernel_launches[KF_RESOLVE]++;
        }
        k_resolve<<<(n_rect + 255) / 256, 256, 0, s>>>(p, exposure_mul, mix_factor, half_mix_factor, is_class_a, xf, vt);
        ctx->last_xf = xf;
        ctx->last_variance_threshold = vt;
        ctx->kernel_launches[KF_RESOLVE]++;
        k_accumulate_totals<<<1, 32, 0, s>>>(p, last_bounce, shadow_traced);
    }
    record(ctx, EV_END);
    ctx->sample_pending = ctx->stats_enabled;
    ctx->pending_bounces = last_bounce;
    ctx->pending_sh = want_sh;
    CU_CHECK(ctx, cudaGetLastError());
    return 0;
}

// ---- AoS <-> SoA staging for the stage entry points ----------------------------------------------------------------
int upload_rays_aos(rc_ctx *ctx, const RayBuf &b, const RayAoS *src, int n) {
    std::vector<float4> p0(n), p1(n), p2(n), p3(n);
    std::vector<uint2> p4(n);
    for (int i = 0; i < n; ++i) {
        const RayAoS &r = src[i];
        p0[i] = make_float4(r.o[0], r.o[1], r.o[2], r.cone_width);
        p1[i] = make_float4(r.d[0], r.d[1], r.d[2], r.cone_spread);
        p2[i] = make_float4(r.c[0], r.c[1], r.c[2], r.pdf);
        p3[i] = make_float4(r.ior[0], r.ior[1], r.ior[2], r.ior[3]);
        p4[i] = make_uint2(r.xy, r.depth);
    }
    CU_CHECK(ctx, cudaMemcpy(b.o_cw, p0.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
    CU_CHECK(ctx, cudaMemcpy(b.d_cs, p1.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
    CU_CHECK(ctx, cudaMemcpy(b.c_pdf, p2.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
    CU_CHECK(ctx, cudaMemcpy(b.ior, p3.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
    CU_CHECK(ctx, cudaMemcpy(b.xy_depth, p4.data(), n * sizeof(uint2), cudaMemcpyHostToDevice));
    return 0;
}

int download_rays_aos(rc_ctx *ctx, const RayBuf &b, RayAoS *dst, int n) {
    std::vector<float4> p0(n), p1(n), p2(n), p3(n);
    std::vector<uint2> p4(n);
    CU_CHECK(ctx, cudaMemcpy(p0.data(), b.o_cw, n * sizeof(float4), cudaMemcpyDeviceToHost));
    CU_CHECK(ctx, cudaMemcpy(p1.data(), b.d_cs, n * sizeof(float4), cudaMemcpyDeviceToHost));
    CU_CHECK(ctx, cudaMemcpy(p2.data(), b.c_pdf, n * sizeof(float4), cudaMemcpyDeviceToHost));
    CU_CHECK(ctx, cudaMemcpy(p3.data(), b.ior, n * sizeof(float4), cudaMemcpyDeviceToHost));
    CU_CHECK(ctx, cudaMemcpy(p4.data(), b.xy_depth, n * sizeof(uint2), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) {
        RayAoS &r = dst[i];
        r.o[0] = p0[i].x, r.o[1] = p0[i].y, r.o[2] = p0[i].z, r.cone_width = p0[i].w;
        r.d[0] = p1[i].x, r.d[1] = p1[i].y, r.d[2] = p1[i].z, r.cone_spread = p1[i].w;
        r.c[0] = p2[i].x, r.c[1] = p2[i].y, r.c[2] = p2[i].z, r.pdf = p2[i].w;
        r.ior[0] = p3[i].x, r.ior[1] = p3[i].y, r.ior[2] = p3[i].z, r.ior[3] = p3[i].w;
        r.xy = p4[i].x, r.depth = p4[i].y;
    }
    return 0;
}

int upload_hits_aos(rc_ctx *ctx, const HitBuf &b, const HitAoS *src, int n) {
    std::vector<float4> p0(n);
    std::vector<int> p1(n);
    for (int i = 0; i < n; ++i) {
        float pf;
        memcpy(&pf, &src[i].prim_index, 4);
        p0[i] = make_float4(src[i].t, src[i].u, src[i].v, pf);
        p1[i] = src[i].obj_index;
    }
    CU_CHECK(ctx, cudaMemcpy(b.tuvp, p0.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
    CU_CHECK(ctx, cudaMemcpy(b.obj, p1.data(), n * sizeof(int), cudaMemcpyHostToDevice));
    return 0;
}

int download_hits_aos(rc_ctx *ctx, const HitBuf &b, HitAoS *dst, int n) {
    std::vector<float4> p0(n);
    std::vector<int> p1(n);
    CU_CHECK(ctx, cudaMemcpy(p0.data(), b.tuvp, n * sizeof(float4), cudaMemcpyDeviceToHost));
    CU_CHECK(ctx, cudaMemcpy(p1.data(), b.obj, n * sizeof(int), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) {
        dst[i].t = p0[i].x, dst[i].u = p0[i].y, dst[i].v = p0[i].z;
        memcpy(&dst[i].prim_index, &p0[i].w, 4);
        dst[i].obj_index = p1[i];
    }
    return 0;
}

int upload_shadow_aos(rc_ctx *ctx, const ShadowBuf &b, const ShadowRayAoS *src, int n) {
    std::vector<float4> p0(n), p1(n), p2(n);
    for (int i = 0; i < n; ++i) {
        float df, xf;
        memcpy(&df, &src[i].depth, 4);
        memcpy(&xf, &src[i].xy, 4);
        p0[i] = make_float4(src[i].o[0], src[i].o[1], src[i].o[2], df);
        p1[i] = make_float4(src[i].d[0], src[i].d[1], src[i].d[2], src[i].dist);
        p2[i] = make_float4(src[i].c[0], src[i].c[1], src[i].c[2], xf);
    }
    CU_CHECK(ctx, cudaMemcpy(b.o_depth, p0.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
    CU_CHECK(ctx, cudaMemcpy(b.d_dist, p1.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
    CU_CHECK(ctx, cudaMemcpy(b.c_xy, p2.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
    return 0;
}

int download_shadow_aos(rc_ctx *ctx, const ShadowBuf &b, ShadowRayAoS *dst, int n) {
    std::vector<float4> p0(n), p1(n), p2(n);
    CU_CHECK(ctx, cudaMemcpy(p0.data(), b.o_depth, n * sizeof(float4), cudaMemcpyDeviceToHost));
    CU_CHECK(ctx, cudaMemcpy(p1.data(), b.d_dist, n * sizeof(float4), cudaMemcpyDeviceToHost));
    CU_CHECK(ctx, cudaMemcpy(p2.data(), b.c_xy, n * sizeof(float4), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) {
        dst[i].o[0] = p0[i].x, dst[i].o[1] = p0[i].y, dst[i].o[2] = p0[i].z;
        memcpy(&dst[i].depth, &p0[i].w, 4);
        dst[i].d[0] = p1[i].x, dst[i].d[1] = p1[i].y, dst[i].d[2] = p1[i].z, dst[i].dist = p1[i].w;
        dst[i].c[0] = p2[i].x, dst[i].c[1] = p2[i].y, dst[i].c[2] = p2[i].z;
        memcpy(&dst[i].xy, &p2[i].w, 4);
    }
    return 0;
}

int set_counter(rc_ctx *ctx, int slot, uint32_t v) {
    CU_CHECK(ctx, cudaMemcpy(ctx->d_counters.get() + slot, &v, sizeof(v), cudaMemcpyHostToDevice));
    return 0;
}

int get_counter(rc_ctx *ctx, int slot, uint32_t *v) {
    CU_CHECK(ctx, cudaMemcpy(v, ctx->d_counters.get() + slot, sizeof(*v), cudaMemcpyDeviceToHost));
    return 0;
}

} // namespace

extern "C" {

int rc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int rc_create(int device, rc_ctx **out_ctx) {
    if (!out_ctx) {
        return 1;
    }
    *out_ctx = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
        cudaGetLastError();
        return 2; // no such device: Cuda::Renderer's ctor turns this into std::runtime_error
    }
    rc_ctx *ctx = new rc_ctx();
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&ctx->prop, device) != cudaSuccess) {
        delete ctx;
        return 3;
    }
    if (ctx->prop.major < 10) {
        // the fatbin only holds sm_100a code
        delete ctx;
        return 4;
    }
    ctx->device_name = ctx->prop.name;
    ctx->num_sms = ctx->prop.multiProcessorCount;
    // every failure below returns through `delete ctx`: what was allocated so far frees itself, with the device current
    if (ctx->d_counters.alloc(CNT_TOTAL) != cudaSuccess || ctx->d_totals.alloc(TOT_COUNT) != cudaSuccess) {
        delete ctx;
        return 6;
    }
    cudaMemset(ctx->d_counters.get(), 0, CNT_TOTAL * sizeof(uint32_t));
    cudaMemset(ctx->d_totals.get(), 0, TOT_COUNT * sizeof(unsigned long long));
    { // srgb_to_linear (CoreRef.h:208-220) of the 256 values a texel channel can hold, with the HOST powf like the reference
        float lut[256];
        for (int i = 0; i < 256; ++i) {
            const float c = float(i) / 255.0f;
            lut[i] = (c > 0.04045f) ? powf((c + 0.055f) / 1.055f, 2.4f) : (c / 12.92f);
        }
        if (ctx->d_srgb_lut.alloc(256) != cudaSuccess ||
            cudaMemcpy(ctx->d_srgb_lut.get(), lut, sizeof(lut), cudaMemcpyHostToDevice) != cudaSuccess) {
            delete ctx;
            return 6;
        }
    }
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return 5;
    }
    ctx->events.resize(kMaxEvents);
    for (auto &e : ctx->events) {
        cudaEventCreate(&e);
    }
    for (auto &e : ctx->user_events) {
        cudaEventCreate(&e);
    }
    // the trace kernels keep their stacks in static shared memory (rt_trace.cuh): RT_TRACE_BLOCKS blocks must fit, the
    // rest of the unified array stays L1
    {
        const int pct = int((sizeof(TraceSmem) + 1024) * RT_TRACE_BLOCKS * 100 / (228 * 1024)) + 1;
        const int carve = pct > 100 ? 100 : pct;
        cudaFuncSetAttribute(k_trace_closest<false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
        cudaFuncSetAttribute(k_trace_closest<true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
        cudaFuncSetAttribute(k_trace_closest<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
        cudaFuncSetAttribute(k_trace_closest<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
        cudaFuncSetAttribute(k_trace_shadow, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
    }
    if (const char *e = getenv("RC_TRACE_FIN_MIN")) { // development knob
        ctx->trace_fin_min = atoi(e);
    }
    cudaFuncSetAttribute(k_shade<true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 0);
    cudaFuncSetAttribute(k_shade<false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 0);
    cudaFuncSetAttribute(k_shade<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 0);
    cudaFuncSetAttribute(k_shade<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 0);
    // function attributes apply to the current device: each context sets them for its own
    cudaFuncSetAttribute(tc::k_unet_conv_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemBudget + 1024);
    *out_ctx = ctx;
    return 0;
}

void rc_destroy(rc_ctx *ctx) {
    if (!ctx) {
        return;
    }
    cudaSetDevice(ctx->device); // the members' destructors free their blocks on this device
    cudaStreamSynchronize(ctx->stream);
    for (auto &e : ctx->events) {
        cudaEventDestroy(e);
    }
    for (auto &e : ctx->user_events) {
        cudaEventDestroy(e);
    }
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *rc_last_error(const rc_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
const char *rc_device_name(const rc_ctx *ctx) { return ctx ? ctx->device_name.c_str() : ""; }

int rc_resize(rc_ctx *ctx, int w, int h) {
    if (!ctx || w < 0 || h < 0 || w > 65535 || h > 65535) {
        return fail(ctx, "rc_resize: bad size %dx%d", w, h);
    }
    cudaSetDevice(ctx->device);
    if (w == ctx->w && h == ctx->h) {
        return 0; // idempotent like Cpu::Renderer::Resize (RendererCPU.h:266-295)
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t n = size_t(w) * h;
    // the old buffers go one by one below: a failure half-way must leave the context unrenderable (fill_params checks
    // for a zero-size frame), not pointing at freed or mis-sized planes
    ctx->w = ctx->h = ctx->fb.w = ctx->fb.h = 0;
    ctx->ray_capacity = 0;
    ctx->geo_offsets.reset();
    ctx->geo_cursor.reset();
    ctx->geo_list.reset();
    ctx->geo_valid = false;
    const bool had_sh = ctx->have_sh;
    ctx->have_sh = false;
    for (DevBuf<float4> &b : ctx->sh_planes) {
        b.reset();
    }
    FrameBufs &fb = ctx->fb;
    float4 **planes[7] = {&fb.temp, &fb.full, &fb.half, &fb.raw, &fb.final, &fb.base_color, &fb.depth_normals};
    for (int i = 0; i < 7; ++i) {
        if (alloc_view(ctx, ctx->fb_planes[i], *planes[i], n)) {
            return 1;
        }
    }
    if (alloc_view(ctx, ctx->fb_required_samples, fb.required_samples, n)) {
        return 1;
    }
    if (n) {
        for (float4 **b : planes) {
            CU_CHECK(ctx, cudaMemsetAsync(*b, 0, n * sizeof(float4), ctx->stream));
        }
        CU_CHECK(ctx, cudaMemsetAsync(fb.required_samples, 0xff, n * sizeof(uint16_t), ctx->stream));
    }
    for (int l = 0; l < 2; ++l) {
        RayBuf &r = ctx->rays[l];
        if (alloc_view(ctx, ctx->ray_planes[l][0], r.o_cw, n) || alloc_view(ctx, ctx->ray_planes[l][1], r.d_cs, n) ||
            alloc_view(ctx, ctx->ray_planes[l][2], r.c_pdf, n) || alloc_view(ctx, ctx->ray_planes[l][3], r.ior, n) ||
            alloc_view(ctx, ctx->ray_xy_depth[l], r.xy_depth, n)) {
            return 1;
        }
    }
    if (alloc_view(ctx, ctx->hit_tuvp, ctx->hits.tuvp, n) || alloc_view(ctx, ctx->hit_obj, ctx->hits.obj, n) ||
        alloc_view(ctx, ctx->shadow_planes[0], ctx->shadow.o_depth, n) ||
        alloc_view(ctx, ctx->shadow_planes[1], ctx->shadow.d_dist, n) ||
        alloc_view(ctx, ctx->shadow_planes[2], ctx->shadow.c_xy, n)) {
        return 1;
    }
    SortBufs &so = ctx->sort;
    if (!so.hist.get()) {
        CU_CHECK(ctx, so.hist.alloc(size_t(kMaxBounces) * kSortBins));
    }
    if (!so.chunk_totals.get()) {
        CU_CHECK(ctx, so.chunk_totals.alloc(size_t(kMaxBounces) * 64));
    }
    CU_CHECK(ctx, so.keys.alloc(n));
    CU_CHECK(ctx, so.keys_sorted.alloc(n));
    ctx->ray_capacity = n;
    ctx->fb.w = w;
    ctx->fb.h = h;
    ctx->w = w;
    ctx->h = h;
    if (had_sh && n && alloc_sh(ctx)) {
        return 1;
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

__global__ void k_fill4(float4 *dst, float4 v, size_t n) {
    for (size_t i = blockIdx.x * size_t(blockDim.x) + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        dst[i] = v;
    }
}

int rc_clear(rc_ctx *ctx, const float rgba[4]) {
    if (!ctx) {
        return 1;
    }
    cudaSetDevice(ctx->device);
    const size_t n = size_t(ctx->w) * ctx->h;
    if (n == 0) {
        return 0;
    }
    const float4 v = make_float4(rgba[0], rgba[1], rgba[2], rgba[3]);
    k_fill4<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(ctx->fb.full, v, n);
    k_fill4<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(ctx->fb.half, v, n);
    if (ctx->have_sh) {
        for (float4 *c : ctx->sh.coef) {
            CU_CHECK(ctx, cudaMemsetAsync(c, 0, n * sizeof(float4), ctx->stream));
        }
    }
    CU_CHECK(ctx, cudaMemsetAsync(ctx->fb.required_samples, 0xff, n * sizeof(uint16_t), ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rc_debug_fill_temp(rc_ctx *ctx, const float rgba[4]) {
    if (!ctx) {
        return 1;
    }
    cudaSetDevice(ctx->device);
    const size_t n = size_t(ctx->w) * ctx->h;
    if (n == 0) {
        return 0;
    }
    k_fill4<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(ctx->fb.temp, make_float4(rgba[0], rgba[1], rgba[2], rgba[3]), n);
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rc_upload_tables(rc_ctx *ctx, const uint32_t *pmj, int dims, int samples, const float *filter_table,
                     int filter_table_size) {
    if (!ctx || !pmj) {
        return fail(ctx, "rc_upload_tables: null argument");
    }
    if (dims != kRandDims || samples != kRandSamples) {
        return fail(ctx, "rc_upload_tables: table must be %d dims x %d samples", kRandDims, kRandSamples);
    }
    cudaSetDevice(ctx->device);
    const size_t n = size_t(dims) * samples * 2;
    CU_CHECK(ctx, ctx->d_pmj.alloc(n));
    CU_CHECK(ctx, cudaMemcpy(ctx->d_pmj.get(), pmj, n * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (filter_table) {
        if (filter_table_size != kFilterTableSize) {
            return fail(ctx, "rc_upload_tables: filter table must have %d entries", kFilterTableSize);
        }
        CU_CHECK(ctx, ctx->d_filter_table.alloc(kFilterTableSize));
        CU_CHECK(ctx, cudaMemcpy(ctx->d_filter_table.get(), filter_table, kFilterTableSize * sizeof(float),
                                 cudaMemcpyHostToDevice));
    }
    ctx->have_tables = true;
    return 0;
}

int rc_upload_scene(rc_ctx *ctx, const rc_scene_view *sv) {
    if (!ctx || !sv) {
        return fail(ctx, "rc_upload_scene: null argument");
    }
    cudaSetDevice(ctx->device);
    if (sv->sky_map_spread_angle != 0.0f) {
        return fail(ctx, "rc_upload_scene: procedural sky is not supported by the CUDA backend");
    }
    // ---- textures: decoded RGBA8 pool + descriptor table; handles in the device copies of the materials and triangle
    // lights become flags | dense id (rt_tex.cuh) ----
    std::vector<Material> mats;
    std::vector<Light> lts;
    if (sv->materials.count != 0) {
        if (sv->materials.stride != sizeof(Material) || !sv->materials.ptr) {
            return fail(ctx, "rc_upload_scene: materials stride %u != %zu", sv->materials.stride, sizeof(Material));
        }
        const Material *m = static_cast<const Material *>(sv->materials.ptr);
        mats.assign(m, m + sv->materials.count);
    }
    if (sv->lights.count != 0) {
        if (sv->lights.stride != sizeof(Light) || !sv->lights.ptr) {
            return fail(ctx, "rc_upload_scene: lights stride %u != %zu", sv->lights.stride, sizeof(Light));
        }
        const Light *l = static_cast<const Light *>(sv->lights.ptr);
        lts.assign(l, l + sv->lights.count);
    }
    std::vector<TexDesc> descs;
    std::vector<uint32_t> texels;
    std::map<uint32_t, uint32_t> dense; // (storage << 28 | index) -> id
    if (sv->texture_count != 0 && !sv->textures) {
        return fail(ctx, "rc_upload_scene: texture_count %u but a null textures pointer", sv->texture_count);
    }
    for (uint32_t ti = 0; ti < sv->texture_count; ++ti) {
        const rc_texture &t = sv->textures[ti];
        if (t.channels < 1 || t.channels > 4) {
            return fail(ctx, "rc_upload_scene: texture %u has %u channels", ti, t.channels);
        }
        TexDesc d{};
        for (int lod = 0; lod < RC_TEX_MIP_LEVELS; ++lod) {
            const int w = t.res[lod][0], h = t.res[lod][1];
            if (w <= 0 || h <= 0 || !t.pixels[lod]) {
                return fail(ctx, "rc_upload_scene: texture %u level %d is empty (absent levels must alias the last real one)",
                            ti, lod);
            }
            d.w[lod] = uint16_t(w);
            d.h[lod] = uint16_t(h);
            int alias = -1;
            for (int k = 0; k < lod; ++k) {
                if (t.pixels[k] == t.pixels[lod] && t.res[k][0] == w && t.res[k][1] == h) {
                    alias = k;
                    break;
                }
            }
            if (alias >= 0) {
                d.offset[lod] = d.offset[alias];
                continue;
            }
            if (texels.size() + size_t(w) * h > 0xffffffffull) {
                return fail(ctx, "rc_upload_scene: more than 2^32 texels");
            }
            d.offset[lod] = uint32_t(texels.size());
            const uint8_t *src = t.pixels[lod];
            const uint32_t n = t.channels;
            for (size_t i = 0; i < size_t(w) * h; ++i) {
                uint32_t c[4];
                for (uint32_t k = 0; k < 4; ++k) {
                    c[k] = src[i * n + (k < n ? k : n - 1)]; // TexStorage*::Fetch: missing channels repeat the last one
                }
                texels.push_back(c[0] | (c[1] << 8) | (c[2] << 16) | (c[3] << 24));
            }
        }
        dense[t.handle & 0xf0ffffffu] = uint32_t(descs.size());
        descs.push_back(d);
    }
    auto patch = [&](uint32_t &h, const char *what, uint32_t owner, int slot) -> int {
        if (h == 0xffffffffu) {
            return 0;
        }
        const auto it = dense.find(h & 0xf0ffffffu);
        if (it == dense.end()) {
            return fail(ctx, "rc_upload_scene: %s %u slot %d references texture 0x%08x which is not in rc_scene_view::textures",
                        what, owner, slot, h);
        }
        h = (h & 0x0f000000u) | it->second; // colour-space flags (sRGB, reconstruct-z, YCoCg) | dense id
        return 0;
    };
    for (uint32_t i = 0; i < mats.size(); ++i) {
        Material &m = mats[i];
        if (m.type > NODE_PRINCIPLED) {
            continue; // dead SparseStorage slot
        }
        // only the slots ShadeSurface reads for this node type are meaningful: AddMaterial zero-initialises material_t
        // and leaves the others at 0 (SceneCPU.cpp:208-247); Mix keeps child material ids in slots 3/4
        const int n_slots = (m.type == NODE_PRINCIPLED) ? 5 : 3;
        for (int t = 0; t < n_slots; ++t) {
            if (m.type == NODE_MIX && t != kTexBase) {
                continue;
            }
            if (patch(m.textures[t], "material", i, t)) {
                return 1;
            }
        }
    }
    for (uint32_t i = 0; i < lts.size(); ++i) {
        if ((lts[i].bits & 7u) == LIGHT_TRI) {
            uint32_t h;
            memcpy(&h, &lts[i].p[2], 4); // light_t::tri.tex_index
            if (patch(h, "triangle light", i, 0)) {
                return 1;
            }
            memcpy(&lts[i].p[2], &h, 4);
        }
    }
    // environment: map handles -> dense ids, quad-tree levels concatenated
    SceneEnv env{};
    env.env_map = sv->env_map;
    env.back_map = sv->back_map;
    if (patch(env.env_map, "environment map", 0, 0) || patch(env.back_map, "background map", 0, 0)) {
        return 1;
    }
    if (env.env_map != 0xffffffffu) {
        env.env_map &= kTexIdBits;
    }
    if (env.back_map != 0xffffffffu) {
        env.back_map &= kTexIdBits;
    }
    env.env_map_rotation = sv->env_map_rotation;
    env.back_map_rotation = sv->back_map_rotation;
    env.qtree_levels = sv->qtree_levels;
    std::vector<float> qtree;
    if (sv->qtree_levels < 0 || sv->qtree_levels > kMaxQTreeLevels) {
        return fail(ctx, "rc_upload_scene: qtree_levels %d out of range", sv->qtree_levels);
    }
    for (int i = 0; i < sv->qtree_levels; ++i) {
        if (!sv->qtree_mips[i]) {
            return fail(ctx, "rc_upload_scene: quad-tree level %d is null", i);
        }
        const size_t quads = size_t(1) << (2 * (sv->qtree_levels - 1 - i));
        env.qtree_offset[i] = uint32_t(qtree.size() / 4);
        qtree.insert(qtree.end(), sv->qtree_mips[i], sv->qtree_mips[i] + quads * 4);
    }
    rc_scene_view patched = *sv;
    patched.materials.ptr = mats.data();
    patched.lights.ptr = lts.data();
    sv = &patched;
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->have_scene = false; // a failed upload must not leave a half-replaced scene renderable
    if (upload_array(ctx, ctx->wnodes, sv->wnodes, sizeof(WNode), "wnodes") ||
        upload_array(ctx, ctx->mtris, sv->mtris, sizeof(MTri), "mtris") ||
        upload_array(ctx, ctx->tri_indices, sv->tri_indices, 4, "tri_indices") ||
        upload_array(ctx, ctx->tri_materials, sv->tri_materials, sizeof(TriMat), "tri_materials") ||
        upload_array(ctx, ctx->materials, sv->materials, sizeof(Material), "materials") ||
        upload_array(ctx, ctx->mesh_instances, sv->mesh_instances, sizeof(MeshInstance), "mesh_instances") ||
        upload_array(ctx, ctx->vertices, sv->vertices, sizeof(Vertex), "vertices") ||
        upload_array(ctx, ctx->vtx_indices, sv->vtx_indices, 4, "vtx_indices") ||
        upload_array(ctx, ctx->lights, sv->lights, sizeof(Light), "lights") ||
        upload_array(ctx, ctx->light_cwnodes, sv->light_cwnodes, sizeof(LightCWNode), "light_cwnodes")) {
        return 1;
    }
    {
        const rc_array da{descs.data(), uint32_t(descs.size()), uint32_t(sizeof(TexDesc))};
        const rc_array ta{texels.data(), uint32_t(texels.size()), 4u};
        const rc_array qa{qtree.data(), uint32_t(qtree.size() / 4), 16u};
        if (upload_array(ctx, ctx->tex_descs, da, sizeof(TexDesc), "texture descriptors") ||
            upload_array(ctx, ctx->tex_texels, ta, 4, "texels") || upload_array(ctx, ctx->qtree, qa, 16, "env quad-tree")) {
            return 1;
        }
        ctx->env = env;
        CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream)); // descs / texels / mats / lts are locals
    }
    ctx->scene_info = *sv;
    ctx->scene_info.materials.ptr = nullptr;
    ctx->scene_info.lights.ptr = nullptr;
    ctx->scene_info.textures = nullptr;
    for (const float *&q : ctx->scene_info.qtree_mips) {
        q = nullptr;
    }
    ctx->li_count = sv->li_indices.count;
    ctx->no_shadow_lights = has_no_shadow_lights(sv);
    ctx->tex_dense = dense;
    ctx->geo_valid = false; // the candidate lists depend on the uvs of the uploaded triangles
    set_sort_bounds(ctx->sort, sv->bounds_min, sv->bounds_max);
    if (build_traversal_copies(ctx, sv)) {
        return 1;
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->have_scene = true;
    return 0;
}

namespace {
// grow / shrink a node array to new_count records keeping the first `keep` ones (device-to-device)
int resize_keep(rc_ctx *ctx, DevArray &a, uint32_t keep, uint32_t new_count) {
    const size_t want = size_t(new_count) * sizeof(WNode);
    if (a.fits(want)) {
        return 0;
    }
    DevArray fresh;
    CU_CHECK(ctx, fresh.resize(want, new_count));
    if (a.ptr() && keep != 0) {
        CU_CHECK(ctx, cudaMemcpyAsync(fresh.ptr(), a.ptr(), size_t(keep) * sizeof(WNode), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    a = std::move(fresh); // frees the old block
    return 0;
}
} // namespace

int rc_set_view_lut(rc_ctx *ctx, uint32_t view_transform, const uint32_t *lut, int dims) {
    if (!ctx || view_transform == 0 || view_transform >= 16 || dims != kViewLutDims) {
        return fail(ctx, "rc_set_view_lut: view transform %u / table size %d^3 not accepted (1..15, %d^3)", view_transform, dims,
                    kViewLutDims);
    }
    cudaSetDevice(ctx->device);
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->last_xf.lut == ctx->d_view_lut[view_transform].get()) {
        ctx->last_xf.lut = nullptr;
    }
    DevBuf<uint32_t> &table = ctx->d_view_lut[view_transform];
    table.reset();
    if (lut) {
        const size_t n = size_t(dims) * dims * dims;
        CU_CHECK(ctx, table.alloc(n));
        CU_CHECK(ctx, cudaMemcpy(table.get(), lut, n * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    return 0;
}

uint64_t rc_scene_upload_bytes(const rc_ctx *ctx) { return ctx ? ctx->scene_h2d_bytes : 0; }

int rc_update_instances(rc_ctx *ctx, const rc_scene_view *sv, uint32_t first_node) {
    if (!ctx || !sv) {
        return fail(ctx, "rc_update_instances: null argument");
    }
    if (!ctx->have_scene) {
        return fail(ctx, "rc_update_instances: no scene uploaded");
    }
    cudaSetDevice(ctx->device);
    const rc_scene_view &old = ctx->scene_info;
    const uint32_t n_nodes = sv->wnodes.count, n_inst = sv->mesh_instances.count;
    if (sv->mtris.count != old.mtris.count || sv->tri_indices.count != old.tri_indices.count ||
        sv->tri_materials.count != old.tri_materials.count || sv->materials.count != old.materials.count ||
        sv->vertices.count != old.vertices.count || sv->vtx_indices.count != old.vtx_indices.count ||
        sv->texture_count != old.texture_count || n_inst != old.mesh_instances.count) {
        return fail(ctx, "rc_update_instances: geometry, materials or the instance count changed since rc_upload_scene");
    }
    if (first_node > n_nodes || first_node > old.wnodes.count || sv->wnodes.stride != sizeof(WNode) ||
        (n_inst != 0 && sv->mesh_instances.stride != sizeof(MeshInstance)) ||
        (sv->lights.count != 0 && (sv->lights.stride != sizeof(Light) || !sv->lights.ptr)) ||
        (n_nodes != 0 && !sv->wnodes.ptr) || (n_inst != 0 && !sv->mesh_instances.ptr)) {
        return fail(ctx, "rc_update_instances: bad node range or array strides");
    }
    // ---- validate the new top level: nodes [first_node, n_nodes) reference each other or mesh instances only ----
    const WNode *nodes = static_cast<const WNode *>(sv->wnodes.ptr);
    const MeshInstance *inst = static_cast<const MeshInstance *>(sv->mesh_instances.ptr);
    uint32_t root_word = kEmptyChild;
    if (sv->tlas_root != 0xffffffffu) {
        if (sv->tlas_root < first_node || sv->tlas_root >= n_nodes) {
            return fail(ctx, "rc_update_instances: tlas_root %u outside [%u, %u)", sv->tlas_root, first_node, n_nodes);
        }
        for (uint32_t n = first_node; n < n_nodes; ++n) {
            const WNode &nd = nodes[n];
            if (nd.child[0] & kLeafBit) {
                const uint32_t first = nd.child[0] & kPrimIndexBits;
                if (first >= n_inst || inst[first].node_index >= first_node) {
                    return fail(ctx, "rc_update_instances: top-level leaf %u names instance %u (of %u) or a BLAS root past %u",
                                n, first, n_inst, first_node);
                }
                continue;
            }
            for (int c = 0; c < 8; ++c) {
                const uint32_t ch = nd.child[c];
                if (ch != kEmptyChild && (ch < first_node || ch >= n_nodes)) {
                    return fail(ctx, "rc_update_instances: top-level node %u child %d = %u outside [%u, %u)", n, c, ch,
                                first_node, n_nodes);
                }
            }
        }
        const uint32_t c0 = nodes[sv->tlas_root].child[0], c1 = nodes[sv->tlas_root].child[1];
        if (c0 & kLeafBit) {
            const uint32_t first = c0 & kPrimIndexBits, blocks = ((first & 7u) + c1 + 7u) / 8u;
            if (first >= kLeafFirstBits || blocks == 0 || blocks > 16) {
                return fail(ctx, "rc_update_instances: the TLAS root leaf cannot be encoded");
            }
            root_word = kLeafBit | ((blocks - 1u) << kLeafBlocksShift) | first;
        } else {
            root_word = sv->tlas_root;
        }
    }
    // ---- lights: texture handles of triangle lights -> dense ids of the uploaded texture table ----
    std::vector<Light> lts;
    if (sv->lights.count != 0) {
        const Light *l = static_cast<const Light *>(sv->lights.ptr);
        lts.assign(l, l + sv->lights.count);
        for (uint32_t i = 0; i < lts.size(); ++i) {
            if ((lts[i].bits & 7u) == LIGHT_TRI) {
                uint32_t h;
                memcpy(&h, &lts[i].p[2], 4);
                if (h != 0xffffffffu) {
                    const auto it = ctx->tex_dense.find(h & 0xf0ffffffu);
                    if (it == ctx->tex_dense.end()) {
                        return fail(ctx, "rc_update_instances: triangle light %u references texture 0x%08x which was not uploaded", i, h);
                    }
                    h = (h & 0x0f000000u) | it->second;
                    memcpy(&lts[i].p[2], &h, 4);
                }
            }
        }
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream)); // samples in flight still read the old top level
    ctx->have_scene = false;
    if (resize_keep(ctx, ctx->wnodes, first_node, n_nodes) || resize_keep(ctx, ctx->dnodes, first_node, n_nodes)) {
        return 1;
    }
    ctx->wnodes.count = ctx->dnodes.count = n_nodes;
    if (n_nodes > first_node) {
        CU_CHECK(ctx, cudaMemcpyAsync(static_cast<WNode *>(ctx->wnodes.ptr()) + first_node, nodes + first_node,
                                      size_t(n_nodes - first_node) * sizeof(WNode), cudaMemcpyHostToDevice, ctx->stream));
        ctx->scene_h2d_bytes += size_t(n_nodes - first_node) * sizeof(WNode);
    }
    rc_array la = sv->lights;
    la.ptr = lts.data();
    if (upload_array(ctx, ctx->mesh_instances, sv->mesh_instances, sizeof(MeshInstance), "mesh_instances") ||
        upload_array(ctx, ctx->lights, la, sizeof(Light), "lights") ||
        upload_array(ctx, ctx->light_cwnodes, sv->light_cwnodes, sizeof(LightCWNode), "light_cwnodes")) {
        return 1;
    }
    if (n_nodes > first_node) {
        k_build_dnodes<<<((n_nodes - first_node) * 8 + 255) / 256, 256, 0, ctx->stream>>>(
            static_cast<const WNode *>(ctx->wnodes.ptr()), static_cast<WNode *>(ctx->dnodes.ptr()), first_node, n_nodes);
    }
    if (n_inst != 0) {
        k_build_blas_roots<<<(n_inst + 255) / 256, 256, 0, ctx->stream>>>(
            static_cast<const WNode *>(ctx->wnodes.ptr()), static_cast<const MeshInstance *>(ctx->mesh_instances.ptr()), n_inst,
            n_nodes, static_cast<uint32_t *>(ctx->blas_roots.ptr()));
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream)); // lts is a local
    CU_CHECK(ctx, cudaGetLastError());
    ctx->tlas_root_word = root_word;
    rc_scene_view &info = ctx->scene_info;
    info.wnodes.count = n_nodes;
    info.lights.count = sv->lights.count;
    info.li_indices.count = sv->li_indices.count;
    info.light_cwnodes.count = sv->light_cwnodes.count;
    info.tlas_root = sv->tlas_root;
    info.visible_lights_count = sv->visible_lights_count;
    info.blocker_lights_count = sv->blocker_lights_count;
    info.env_light_index = sv->env_light_index;
    memcpy(info.bounds_min, sv->bounds_min, sizeof(info.bounds_min));
    memcpy(info.bounds_max, sv->bounds_max, sizeof(info.bounds_max));
    ctx->li_count = sv->li_indices.count;
    ctx->no_shadow_lights = has_no_shadow_lights(sv);
    set_sort_bounds(ctx->sort, sv->bounds_min, sv->bounds_max);
    ctx->have_scene = true;
    return 0;
}

int rc_render(rc_ctx *ctx, const rc_pass_desc *pass) {
    if (!ctx || !pass) {
        return fail(ctx, "rc_render: null argument");
    }
    cudaSetDevice(ctx->device);
    KParams p;
    if (fill_params(ctx, pass, p)) {
        return 1;
    }
    const uint32_t split_flags = RC_RENDER_SKIP_DIRECT | RC_RENDER_SKIP_INDIRECT | RC_RENDER_OUTPUT_SH;
    if ((pass->flags & split_flags) && ctx->no_shadow_lights) {
        // the shading adds such a light's contribution straight into the colour of the surface it lights, with no
        // shadow ray: the kernels cannot tell it from that surface's emission, so the split would be wrong
        return fail(ctx, "RC_RENDER_SKIP_DIRECT / SKIP_INDIRECT / OUTPUT_SH need every sampled light to cast shadows; "
                         "the scene has a light with cast_shadow = 0");
    }
    if (pass->cam.type == 2 && ensure_geo_lists(ctx, pass)) {
        return 1;
    }
    if ((pass->flags & RC_RENDER_OUTPUT_SH) && !ctx->have_sh && alloc_sh(ctx)) {
        return 1;
    }
    if (enqueue_sample(ctx, pass, p)) {
        return 1;
    }
    if ((pass->flags & RC_RENDER_ASYNC) == 0) {
        return rc_sync(ctx);
    }
    return 0;
}

// ---- UNet denoiser (rt_unet.cuh) ----------------------------------------------------------------------------------
namespace {
float half_bits_to_float(uint16_t h) {
    const uint32_t sign = uint32_t(h & 0x8000u) << 16, exp = (h >> 10) & 0x1fu, man = h & 0x3ffu;
    uint32_t bits;
    if (exp == 0) {
        if (man == 0) {
            bits = sign;
        } else { // subnormal
            int e = -1;
            uint32_t m = man;
            do {
                ++e;
                m <<= 1;
            } while ((m & 0x400u) == 0);
            bits = sign | uint32_t(127 - 15 - e) << 23 | (m & 0x3ffu) << 13;
        }
    } else if (exp == 31) {
        bits = sign | 0x7f800000u | man << 13;
    } else {
        bits = sign | (exp + 127 - 15) << 23 | man << 13;
    }
    float f;
    memcpy(&f, &bits, 4);
    return f;
}

// tensor i of the network (output of pass i, i < 15): channels and down-scale shift
void unet_tensor_shape(int i, int &channels, int &shift) {
    const UNetLayerShape L = unet_layer(i);
    channels = L.cout;
    shift = L.level + (L.pool ? 1 : 0);
}

int unet_alloc_tensors(rc_ctx *ctx) {
    const int wr = (ctx->w + 15) / 16 * 16, hr = (ctx->h + 15) / 16 * 16;
    if (ctx->unet_tw == wr && ctx->unet_th == hr && ctx->unet_t[0].get()) {
        return 0;
    }
    ctx->unet_tw = ctx->unet_th = 0;
    for (int i = 0; i < 15; ++i) {
        int c, sh;
        unet_tensor_shape(i, c, sh);
        const size_t n = size_t(wr >> sh) * size_t(hr >> sh) * size_t(c);
        CU_CHECK(ctx, ctx->unet_t[i].alloc(n ? n : 1));
        CU_CHECK(ctx, cudaMemsetAsync(ctx->unet_t[i].get(), 0, (n ? n : 1) * sizeof(float), ctx->stream));
    }
    ctx->unet_tw = wr;
    ctx->unet_th = hr;
    return 0;
}
} // namespace

// ---- tensor-core path of the UNet (rt_unet_tc.cuh) -------------------------------------------------------------------
namespace {
int round_up_i(int v, int a) { return (v + a - 1) / a * a; }

// K layout of layer i on the tensor-core path: the first input tensor's channels in nkb1 blocks of 64, then (decoder
// layers) the skip tensor's channels in nkb2 blocks; real channels are padded to 16 inside their last block
int unet_tc_nkb1(int i) { return (round_up_i(unet_layer(i).cin1, 16) + 63) / 64; }
int unet_tc_nkb2(int i) { return unet_layer(i).cin2 ? (round_up_i(unet_layer(i).cin2, 16) + 63) / 64 : 0; }
int unet_tc_in_cs(int i) { return (unet_tc_nkb1(i) + unet_tc_nkb2(i)) * 64; }
int unet_tc_cin_pos(int i, int ci) {
    const UNetLayerShape L = unet_layer(i);
    return ci < L.cin1 ? ci : unet_tc_nkb1(i) * 64 + (ci - L.cin1);
}
// layers whose output feeds a decoder's up-sampling: they write every pixel to a 2 x 2 block of the finer grid
bool unet_tc_writes_upsampled(int i) { return i + 1 < kUNetLayers && unet_layer(i + 1).up; }

size_t unet_h_elems(int w, int h, int cs) { return size_t(w + 2) * size_t(h + 2) * size_t(cs); }

int unet_tc_alloc(rc_ctx *ctx) {
    const int wr = (ctx->w + 15) / 16 * 16, hr = (ctx->h + 15) / 16 * 16;
    if (ctx->unet_htw == wr && ctx->unet_hth == hr && ctx->unet_hx0.get()) {
        return 0;
    }
    ctx->unet_htw = ctx->unet_hth = 0;
    auto alloc0 = [&](DevBuf<__half> &b, size_t n) -> int {
        CU_CHECK(ctx, b.alloc(n));
        CU_CHECK(ctx, cudaMemsetAsync(b.get(), 0, n * sizeof(__half), ctx->stream)); // borders and padded channels stay zero for good
        return 0;
    };
    for (int i = 0; i < 15; ++i) {
        int c, sh;
        unet_tensor_shape(i, c, sh);
        if (unet_tc_writes_upsampled(i)) {
            --sh; // stored already up-sampled (the convolution's epilogue replicates)
        }
        if (alloc0(ctx->unet_ht[i], unet_h_elems(wr >> sh, hr >> sh, round_up_i(c, 64)))) {
            return 1;
        }
    }
    // network input (64-channel stride) and the pre-pooling output of the encoder convolutions (sized for level 0)
    if (alloc0(ctx->unet_hx0, unet_h_elems(wr, hr, 64)) || alloc0(ctx->unet_hs, unet_h_elems(wr, hr, 128))) {
        return 1;
    }
    ctx->unet_htw = wr;
    ctx->unet_hth = hr;
    return 0;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D fp16 tensor map: `rows` rows of `cs` channels, box = [box_rows][64 channels], 128-byte swizzle
int make_map(rc_ctx *ctx, CUtensorMap *m, const void *base, int cs, size_t rows, int box_rows) {
    if (!ctx->tensor_map_encode) {
        cudaDriverEntryPointQueryResult q;
        void *fn = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) {
            return fail(ctx, "rc_denoise_unet: cuTensorMapEncodeTiled is not available from the driver");
        }
        ctx->tensor_map_encode = fn;
    }
    const cuuint64_t dims[2] = {cuuint64_t(cs), cuuint64_t(rows)};
    const cuuint64_t strides[1] = {cuuint64_t(cs) * 2};
    const cuuint32_t box[2] = {64, cuuint32_t(box_rows)};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = reinterpret_cast<EncodeTiledFn>(ctx->tensor_map_encode)(
        m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        return fail(ctx, "rc_denoise_unet: cuTensorMapEncodeTiled failed (%d)", int(r));
    }
    return 0;
}

// one convolution on the tensor cores: in1 (bordered, stride cs1) [++ in2 (stride cs2)] -> out
int unet_conv_tc(rc_ctx *ctx, int layer, const __half *in1, int cs1, const __half *in2, int cs2, int w, int h, __half *out,
                 int out_cs, bool up, const rc_rect &r) {
    const UNetLayerShape L = unet_layer(layer);
    const int n = round_up_i(L.cout, 16);
    const size_t rows = size_t(w + 2) * size_t(h + 2);
    CUtensorMap map_a1, map_a2, map_b;
    if (make_map(ctx, &map_a1, in1, cs1, rows, tc::kHaloRows) ||
        make_map(ctx, &map_a2, in2 ? in2 : in1, in2 ? cs2 : cs1, rows, tc::kHaloRows) ||
        make_map(ctx, &map_b, ctx->unet_hw[layer].get(), unet_tc_in_cs(layer), size_t(9) * n, n)) {
        return 1;
    }
    tc::ConvTcParams p{};
    p.bias = ctx->unet_hb[layer].get();
    p.out = out;
    p.fb = ctx->fb;
    p.w = w;
    p.h = h;
    p.cin1 = round_up_i(L.cin1, 16);
    p.nkb1 = unet_tc_nkb1(layer);
    p.cin2 = L.cin2 ? round_up_i(L.cin2, 16) : 0;
    p.nkb2 = unet_tc_nkb2(layer);
    p.n = n;
    p.cout = L.cout;
    p.out_cs = out_cs;
    p.up = up ? 1 : 0;
    p.tmem_cols = n <= 32 ? 32 : (n <= 64 ? 64 : 128);
    const int b_slot_bytes = (n * tc::kBlockK * 2 + 1023) & ~1023;
    const int nkb = p.nkb1 + p.nkb2;
    p.base_offset = 0; // measured: the swizzle is a function of the absolute shared address, a shifted start needs no base offset
    p.tiles_x = (w + tc::kTileM - 1) / tc::kTileM;
    p.tiles = p.tiles_x * h;
    p.last = (layer == kUNetLayers - 1);
    p.rx = r.x, p.ry = r.y, p.rw = r.w, p.rh = r.h;
    p.xf = ctx->last_xf;
    // Shared memory plan.  Every CTA asks for more than a third of an SM's 227 KB whatever the layer, so that at most two
    // CTAs (2 x 2 accumulators of <= 128 columns = the 512 TMEM columns) are ever resident on an SM.  A filter that fits
    // next to a >= 3-slot activation ring stays resident; otherwise the weights stream through a B ring.
    const int b_all_bytes = 9 * nkb * b_slot_bytes;
    const int smem = tc::kSmemBudget + 1024;
    if (b_all_bytes + 3 * tc::kASlotBytes <= tc::kSmemBudget) {
        p.b_resident = 1;
        p.a_slots = std::min(tc::kMaxASlots, (tc::kSmemBudget - b_all_bytes) / tc::kASlotBytes);
        p.stages = 1;
    } else {
        p.b_resident = 0;
        p.a_slots = 3;
        p.stages = std::min(tc::kMaxStages, (tc::kSmemBudget - p.a_slots * tc::kASlotBytes) / b_slot_bytes);
    }
    const int grid = std::min(p.tiles, 2 * ctx->num_sms);
    tc::k_unet_conv_tc<<<grid, tc::kThreads, smem, ctx->stream>>>(map_a1, map_a2, map_b, p);
    return 0;
}

int unet_run_tc(rc_ctx *ctx, int pass, const rc_rect &r) {
    if (unet_tc_alloc(ctx)) {
        return 1;
    }
    cudaStream_t s = ctx->stream;
    const int wr = ctx->unet_htw, hr = ctx->unet_hth;
    static const int skip_of[16] = {-1, -1, -1, -1, -1, -1, -1, 3, -1, 2, -1, 1, -1, -2, -1, -1};
    for (int i = (pass < 0 ? 0 : pass); i <= (pass < 0 ? kUNetLayers - 1 : pass); ++i) {
        const UNetLayerShape L = unet_layer(i);
        const int w = wr >> L.level, h = hr >> L.level;
        const __half *in1, *in2 = nullptr;
        int cs1, cs2 = 0;
        if (i == 0) {
            tc::k_unet_feat_h<<<dim3((wr + 127) / 128, hr), 128, 0, s>>>(ctx->fb, ctx->unet_hx0.get(), wr, hr, 64);
            in1 = ctx->unet_hx0.get();
            cs1 = 64;
        } else {
            // decoder (L.up): the previous layer already stored its output up-sampled; the skip tensor (or the network
            // input) is the second K range of the same GEMM -- no gather pass
            in1 = ctx->unet_ht[i - 1].get();
            cs1 = round_up_i(L.cin1, 64);
            if (L.up) {
                in2 = skip_of[i] == -2 ? ctx->unet_hx0.get() : ctx->unet_ht[skip_of[i]].get();
                cs2 = skip_of[i] == -2 ? 64 : round_up_i(L.cin2, 64);
            }
        }
        const int out_cs = round_up_i(L.cout, 64);
        if (i == kUNetLayers - 1) {
            if (unet_conv_tc(ctx, i, in1, cs1, in2, cs2, w, h, nullptr, 0, false, r)) {
                return 1;
            }
        } else if (L.pool) {
            if (unet_conv_tc(ctx, i, in1, cs1, in2, cs2, w, h, ctx->unet_hs.get(), out_cs, false, r)) {
                return 1;
            }
            const int c8 = round_up_i(L.cout, 8) / 8;
            const size_t work = size_t(w >> 1) * size_t(h >> 1) * size_t(c8);
            tc::k_unet_pool_h<<<unsigned((work + 255) / 256), 256, 0, s>>>(ctx->unet_hs.get(), out_cs, ctx->unet_ht[i].get(), out_cs, c8, w, h);
        } else if (unet_conv_tc(ctx, i, in1, cs1, in2, cs2, w, h, ctx->unet_ht[i].get(), out_cs, unet_tc_writes_upsampled(i), r)) {
            return 1;
        }
    }
    return 0;
}
} // namespace

int rc_unet_set_weights(rc_ctx *ctx, const rc_unet_layer layers[16]) {
    if (!ctx || !layers) {
        return fail(ctx, "rc_unet_set_weights: null argument");
    }
    cudaSetDevice(ctx->device);
    ctx->unet_ready = false;
    for (int i = 0; i < kUNetLayers; ++i) {
        const UNetLayerShape L = unet_layer(i);
        const int cin = L.cin1 + L.cin2;
        if (!layers[i].weights || !layers[i].bias || layers[i].cin != cin || layers[i].cout != L.cout) {
            return fail(ctx, "rc_unet_set_weights: layer %d must be %d -> %d channels (got %d -> %d)", i, cin, L.cout,
                        layers[i].cin, layers[i].cout);
        }
        // OIHW fp16 -> [cout][tap][cin] fp32 (exact)
        std::vector<float> w(size_t(L.cout) * 9 * cin), b(L.cout);
        for (int co = 0; co < L.cout; ++co) {
            b[co] = half_bits_to_float(layers[i].bias[co]);
            for (int ci = 0; ci < cin; ++ci) {
                for (int t = 0; t < 9; ++t) {
                    w[(size_t(co) * 9 + t) * cin + ci] = half_bits_to_float(layers[i].weights[(size_t(co) * cin + ci) * 9 + t]);
                }
            }
        }
        CU_CHECK(ctx, ctx->unet_w[i].alloc(w.size()));
        CU_CHECK(ctx, ctx->unet_b[i].alloc(b.size()));
        CU_CHECK(ctx, cudaMemcpy(ctx->unet_w[i].get(), w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
        CU_CHECK(ctx, cudaMemcpy(ctx->unet_b[i].get(), b.data(), b.size() * sizeof(float), cudaMemcpyHostToDevice));
        // tensor-core path: the fp16 bits as they came, [tap][cout padded to 16][input channel stride], zero padded
        const int n = round_up_i(L.cout, 16), in_cs = unet_tc_in_cs(i);
        std::vector<uint16_t> hw(size_t(9) * n * in_cs, 0);
        std::vector<float> hb(n, 0.0f);
        for (int co = 0; co < L.cout; ++co) {
            hb[co] = b[co];
            for (int ci = 0; ci < cin; ++ci) {
                for (int t = 0; t < 9; ++t) {
                    hw[(size_t(t) * n + co) * in_cs + unet_tc_cin_pos(i, ci)] = layers[i].weights[(size_t(co) * cin + ci) * 9 + t];
                }
            }
        }
        CU_CHECK(ctx, ctx->unet_hw[i].alloc(hw.size()));
        CU_CHECK(ctx, ctx->unet_hb[i].alloc(hb.size()));
        CU_CHECK(ctx, cudaMemcpy(ctx->unet_hw[i].get(), hw.data(), hw.size() * 2, cudaMemcpyHostToDevice));
        CU_CHECK(ctx, cudaMemcpy(ctx->unet_hb[i].get(), hb.data(), hb.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    ctx->unet_ready = true;
    return 0;
}

int rc_denoise_unet(rc_ctx *ctx, int pass, const rc_rect *rect, uint32_t flags) {
    if (!ctx || !rect) {
        return fail(ctx, "rc_denoise_unet: null argument");
    }
    cudaSetDevice(ctx->device);
    if (!ctx->unet_ready) {
        return fail(ctx, "rc_denoise_unet: no weights (rc_unet_set_weights)");
    }
    if (pass < -1 || pass >= kUNetLayers) {
        return fail(ctx, "rc_denoise_unet: pass %d out of range", pass);
    }
    const rc_rect &r = *rect;
    if (r.x < 0 || r.y < 0 || r.w <= 0 || r.h <= 0 || r.x + r.w > ctx->w || r.y + r.h > ctx->h) {
        return fail(ctx, "rc_denoise_unet: rect (%d,%d,%d,%d) is outside the %dx%d frame", r.x, r.y, r.w, r.h, ctx->w, ctx->h);
    }
    cudaStream_t s = ctx->stream;
    cudaEvent_t e0 = ctx->user_events[8], e1 = ctx->user_events[9];
    if (e0 && e1) {
        cudaEventRecord(e0, s);
    }
    if ((flags & RC_UNET_FP32) == 0) {
        if (unet_run_tc(ctx, pass, r)) {
            return 1;
        }
        if (e0 && e1) {
            cudaEventRecord(e1, s);
        }
        CU_CHECK(ctx, cudaStreamSynchronize(s));
        CU_CHECK(ctx, cudaGetLastError());
        if (e0 && e1) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, e0, e1);
            ctx->stats_us[8] += uint64_t(double(ms) * 1000.0);
        }
        return 0;
    }
    if (unet_alloc_tensors(ctx)) {
        return 1;
    }
    const int wr = ctx->unet_tw, hr = ctx->unet_th;
    // which tensors each pass reads: main input, skip input (-1 none, -2 the frame's feature planes)
    static const int in1_of[16] = {-2, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14};
    static const int in2_of[16] = {-1, -1, -1, -1, -1, -1, -1, 3, -1, 2, -1, 1, -1, -2, -1, -1};
    for (int i = (pass < 0 ? 0 : pass); i <= (pass < 0 ? kUNetLayers - 1 : pass); ++i) {
        const UNetLayerShape L = unet_layer(i);
        UNetConvParams p{};
        p.fb = ctx->fb;
        p.cin1 = L.cin1;
        p.cin2 = L.cin2;
        p.cout = L.cout;
        p.w = wr >> L.level;
        p.h = hr >> L.level;
        p.up = L.up ? 1 : 0;
        p.pool = L.pool ? 1 : 0;
        p.feat_in1 = in1_of[i] == -2;
        p.feat_in2 = in2_of[i] == -2;
        p.last = (i == kUNetLayers - 1);
        p.xf = ctx->last_xf;
        p.in1 = in1_of[i] >= 0 ? ctx->unet_t[in1_of[i]].get() : nullptr;
        p.in2 = in2_of[i] >= 0 ? ctx->unet_t[in2_of[i]].get() : nullptr;
        p.weights = ctx->unet_w[i].get();
        p.bias = ctx->unet_b[i].get();
        p.out = (i < 15) ? ctx->unet_t[i].get() : nullptr;
        // the region on this level's grid: passes < 15 round the frame rect outward to the 16-pixel grid first.  Then the
        // origin is even on every pooled level (k_unet_conv_f32 pools the lane quads of tiles that start at p.rx, p.ry),
        // and the regions of a partition cover the rounded frame.  Pixels outside the rect are recomputed with the same
        // inputs, which is harmless when all regions of pass k run before pass k + 1.
        int x0 = r.x, y0 = r.y, x1 = r.x + r.w, y1 = r.y + r.h;
        if (i < 15) {
            x0 &= ~15;
            y0 &= ~15;
            x1 = (x1 + 15) & ~15;
            y1 = (y1 + 15) & ~15;
        }
        const int sh = L.level;
        p.rx = x0 >> sh;
        p.ry = y0 >> sh;
        p.rw = min(((x1 + (1 << sh) - 1) >> sh), p.w) - p.rx;
        p.rh = min(((y1 + (1 << sh) - 1) >> sh), p.h) - p.ry;
        const dim3 grid((p.rw + kConvTile - 1) / kConvTile, (p.rh + kConvTile - 1) / kConvTile,
                        (p.cout + kConvCoutBlk - 1) / kConvCoutBlk);
        k_unet_conv_f32<<<grid, 64, 0, s>>>(p);
    }
    if (e0 && e1) {
        cudaEventRecord(e1, s);
    }
    CU_CHECK(ctx, cudaStreamSynchronize(s));
    CU_CHECK(ctx, cudaGetLastError());
    if (e0 && e1) {
        float ms = 0.0f;
        cudaEventElapsedTime(&ms, e0, e1);
        ctx->stats_us[8] += uint64_t(double(ms) * 1000.0);
    }
    return 0;
}

int rc_debug_write_plane(rc_ctx *ctx, int which, const float *src) {
    if (!ctx || !src) {
        return fail(ctx, "rc_debug_write_plane: null argument");
    }
    if (which < RC_BUF_FINAL || which > RC_BUF_TEMP) {
        return fail(ctx, "rc_debug_write_plane: buffer %d is not a frame plane (RC_BUF_FINAL .. RC_BUF_TEMP)", which);
    }
    cudaSetDevice(ctx->device);
    const size_t n = size_t(ctx->w) * ctx->h;
    if (n == 0) {
        return 0;
    }
    CU_CHECK(ctx, cudaMemcpyAsync(const_cast<float4 *>(plane_of(ctx, which)), src, n * sizeof(float4), cudaMemcpyHostToDevice,
                                  ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rc_debug_unet_tensor(rc_ctx *ctx, uint32_t flags, int tensor, int row0, int nrows, float *dst, int32_t dims[3]) {
    if (!ctx || !dims) {
        return fail(ctx, "rc_debug_unet_tensor: null argument");
    }
    cudaSetDevice(ctx->device);
    const bool fp32 = (flags & RC_UNET_FP32) != 0;
    const int wr = (ctx->w + 15) / 16 * 16, hr = (ctx->h + 15) / 16 * 16;
    if (tensor < 0 || tensor > (fp32 ? 14 : 15)) {
        return fail(ctx, "rc_debug_unet_tensor: tensor %d out of range for the %s path", tensor, fp32 ? "fp32" : "tensor-core");
    }
    const bool ran = fp32 ? (ctx->unet_tw == wr && ctx->unet_th == hr && ctx->unet_t[0].get())
                          : (ctx->unet_htw == wr && ctx->unet_hth == hr && ctx->unet_hx0.get());
    if (!ran) {
        return fail(ctx, "rc_debug_unet_tensor: the %s path has not run at the %dx%d rounded frame", fp32 ? "fp32" : "tensor-core",
                    wr, hr);
    }
    int c = 64, sh = 0;
    if (tensor < 15) {
        unet_tensor_shape(tensor, c, sh);
    }
    if (fp32) {
        dims[0] = hr >> sh;
        dims[1] = wr >> sh;
        dims[2] = c;
    } else {
        if (tensor < 15 && unet_tc_writes_upsampled(tensor)) {
            --sh;
        }
        dims[0] = (hr >> sh) + 2;
        dims[1] = (wr >> sh) + 2;
        dims[2] = round_up_i(c, 64);
    }
    if (row0 < 0 || nrows < 0 || row0 + nrows > dims[0]) {
        return fail(ctx, "rc_debug_unet_tensor: rows [%d, %d) outside the %d rows of tensor %d", row0, row0 + nrows, dims[0], tensor);
    }
    if (!dst || nrows == 0) {
        return 0;
    }
    const size_t row = size_t(dims[1]) * size_t(dims[2]), n = row * size_t(nrows);
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (fp32) {
        CU_CHECK(ctx, cudaMemcpy(dst, ctx->unet_t[tensor].get() + row * size_t(row0), n * sizeof(float), cudaMemcpyDeviceToHost));
        return 0;
    }
    const __half *src = (tensor < 15 ? ctx->unet_ht[tensor].get() : ctx->unet_hx0.get()) + row * size_t(row0);
    std::vector<uint16_t> bits(n);
    CU_CHECK(ctx, cudaMemcpy(bits.data(), src, n * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; ++i) {
        dst[i] = half_bits_to_float(bits[i]);
    }
    return 0;
}

int rc_build_lbvh(rc_ctx *ctx, const float *boxes, uint32_t n, rc_lbvh_node *nodes_out, uint32_t *order_out) {
    if (!ctx || !boxes || !nodes_out || !order_out || n < 2 || n > 0x3fffffffu) {
        return fail(ctx, "rc_build_lbvh: bad argument");
    }
    static_assert(sizeof(rc_lbvh_node) == sizeof(LbvhNode), "layout");
    cudaSetDevice(ctx->device);
    cudaStream_t s = ctx->stream;
    DevBuf<float> d_boxes, d_bounds;
    DevBuf<uint32_t> d_codes, d_codes2, d_ids, d_ids2, d_parent, d_visits;
    DevBuf<LbvhNode> d_nodes;
    if (d_boxes.alloc(size_t(n) * 6) != cudaSuccess || d_bounds.alloc(6) != cudaSuccess || d_codes.alloc(n) != cudaSuccess ||
        d_codes2.alloc(n) != cudaSuccess || d_ids.alloc(n) != cudaSuccess || d_ids2.alloc(n) != cudaSuccess ||
        d_parent.alloc(size_t(2) * n - 1) != cudaSuccess || d_visits.alloc(n) != cudaSuccess ||
        d_nodes.alloc(size_t(2) * n - 1) != cudaSuccess) {
        return fail(ctx, "rc_build_lbvh: out of device memory");
    }
    cudaMemcpyAsync(d_boxes.get(), boxes, size_t(n) * 6 * sizeof(float), cudaMemcpyHostToDevice, s);
    const int init[6] = {0x7fffffff, 0x7fffffff, 0x7fffffff, int(0x80000000), int(0x80000000), int(0x80000000)};
    cudaMemcpyAsync(d_bounds.get(), init, sizeof(init), cudaMemcpyHostToDevice, s);
    cudaMemsetAsync(d_visits.get(), 0, size_t(n) * 4, s);
    const unsigned blocks = (n + 255) / 256;
    k_lbvh_bounds<<<min(blocks, 1024u), 256, 0, s>>>(d_boxes.get(), n, d_bounds.get());
    k_lbvh_codes<<<blocks, 256, 0, s>>>(d_boxes.get(), n, d_bounds.get(), d_codes.get(), d_ids.get());
    size_t temp_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, d_codes.get(), d_codes2.get(), d_ids.get(), d_ids2.get(), int(n), 0,
                                    30, s);
    DevBuf<uint8_t> d_temp;
    if (d_temp.alloc(temp_bytes ? temp_bytes : 16) != cudaSuccess) {
        return fail(ctx, "rc_build_lbvh: out of device memory");
    }
    cub::DeviceRadixSort::SortPairs(d_temp.get(), temp_bytes, d_codes.get(), d_codes2.get(), d_ids.get(), d_ids2.get(),
                                    int(n), 0, 30, s);
    k_lbvh_hierarchy<<<blocks, 256, 0, s>>>(d_codes2.get(), int(n), d_nodes.get(), d_parent.get());
    k_lbvh_fit<<<blocks, 256, 0, s>>>(d_boxes.get(), d_ids2.get(), int(n), d_nodes.get(), d_parent.get(), d_visits.get());
    cudaMemcpyAsync(nodes_out, d_nodes.get(), (size_t(2) * n - 1) * sizeof(LbvhNode), cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(order_out, d_ids2.get(), size_t(n) * 4, cudaMemcpyDeviceToHost, s);
    const cudaError_t e = cudaStreamSynchronize(s);
    if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) {
        return fail(ctx, "rc_build_lbvh: %s", cudaGetErrorString(e));
    }
    return 0;
}

int rc_denoise_nlm(rc_ctx *ctx, const rc_rect *rect, int iteration) {
    if (!ctx || !rect) {
        return fail(ctx, "rc_denoise_nlm: null argument");
    }
    cudaSetDevice(ctx->device);
    const rc_rect &r = *rect;
    if (r.x < 0 || r.y < 0 || r.w <= 0 || r.h <= 0 || r.x + r.w > ctx->w || r.y + r.h > ctx->h) {
        return fail(ctx, "rc_denoise_nlm: rect (%d,%d,%d,%d) is outside the %dx%d frame", r.x, r.y, r.w, r.h, ctx->w, ctx->h);
    }
    NlmParams p{};
    p.fb = ctx->fb;
    p.rx = r.x, p.ry = r.y, p.rw = r.w, p.rh = r.h;
    p.ex = r.x - kNlmExt, p.ey = r.y - kNlmExt, p.ew = r.w + 2 * kNlmExt, p.eh = r.h + 2 * kNlmExt;
    const size_t plane = size_t(p.ew) * p.eh;
    if (ctx->nlm_scratch.count() < 3 * plane) {
        CU_CHECK(ctx, ctx->nlm_scratch.alloc(3 * plane));
    }
    p.temp_final = ctx->nlm_scratch.get();
    p.var_h = ctx->nlm_scratch.get() + plane;
    p.var_f = ctx->nlm_scratch.get() + 2 * plane;
    p.variance_threshold = ctx->last_variance_threshold;
    p.iteration = iteration;
    p.xf = ctx->last_xf;
    cudaStream_t s = ctx->stream;
    cudaEvent_t e0 = ctx->user_events[8], e1 = ctx->user_events[9];
    if (e0 && e1) {
        cudaEventRecord(e0, s);
    }
    k_nlm_prep<<<unsigned((plane + 255) / 256), 256, 0, s>>>(p);
    const size_t inner = size_t(p.ew - 8) * (p.eh - 8);
    k_nlm_vblur<<<unsigned((inner + 255) / 256), 256, 0, s>>>(p);
    k_nlm_filter<<<dim3((r.w + kNlmBx - 1) / kNlmBx, (r.h + kNlmBy - 1) / kNlmBy), dim3(kNlmBx, kNlmBy), 0, s>>>(p);
    if (e0 && e1) {
        cudaEventRecord(e1, s);
    }
    CU_CHECK(ctx, cudaStreamSynchronize(s));
    CU_CHECK(ctx, cudaGetLastError());
    if (e0 && e1) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) {
            ctx->stats_us[8] += uint64_t(ms * 1000.0f); // stats_t::time_denoise_us
        }
    }
    return 0;
}

int rc_sync(rc_ctx *ctx) {
    if (!ctx) {
        return 1;
    }
    cudaSetDevice(ctx->device);
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    harvest_stats(ctx);
    return 0;
}

int rc_readback(rc_ctx *ctx, int which, const rc_rect *rect, float *dst, int pitch) {
    if (!ctx || !rect || !dst) {
        return fail(ctx, "rc_readback: null argument");
    }
    cudaSetDevice(ctx->device);
    const float4 *src = nullptr;
    if (plane_or_fail(ctx, which, "rc_readback", &src)) {
        return 1;
    }
    if (rect->x < 0 || rect->y < 0 || rect->w <= 0 || rect->h <= 0 || rect->x + rect->w > ctx->w ||
        rect->y + rect->h > ctx->h || pitch < rect->w) {
        return fail(ctx, "rc_readback: bad rect/pitch");
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    CU_CHECK(ctx, cudaMemcpy2D(dst, size_t(pitch) * sizeof(float4), src + size_t(rect->y) * ctx->w + rect->x,
                               size_t(ctx->w) * sizeof(float4), size_t(rect->w) * sizeof(float4), rect->h,
                               cudaMemcpyDeviceToHost));
    return 0;
}

int rc_readback_async(rc_ctx *ctx, int which, const rc_rect *rect, float *dst, int pitch) {
    if (!ctx || !rect || !dst) {
        return fail(ctx, "rc_readback_async: null argument");
    }
    cudaSetDevice(ctx->device);
    const float4 *src = nullptr;
    if (plane_or_fail(ctx, which, "rc_readback_async", &src)) {
        return 1;
    }
    if (rect->x < 0 || rect->y < 0 || rect->w <= 0 || rect->h <= 0 || rect->x + rect->w > ctx->w ||
        rect->y + rect->h > ctx->h || pitch < rect->w) {
        return fail(ctx, "rc_readback_async: bad rect/pitch");
    }
    CU_CHECK(ctx, cudaMemcpy2DAsync(dst, size_t(pitch) * sizeof(float4), src + size_t(rect->y) * ctx->w + rect->x,
                                    size_t(ctx->w) * sizeof(float4), size_t(rect->w) * sizeof(float4), rect->h,
                                    cudaMemcpyDeviceToHost, ctx->stream));
    return 0;
}

// ---- multi-GPU: one process, one context per device, row strips (SURVEY.md section 8(e)) ---------------------------
struct rc_comm {
    std::vector<rc_ctx *> ctxs;
    std::vector<char> peer_ok; // ctxs[0] can address ctxs[r]'s memory
    rc_rect last_rect{0, 0, 0, 0};
    std::string last_error;
};

namespace {
int comm_fail(rc_comm *c, const char *fmt, ...) {
    char buf[1024];
    va_list vl;
    va_start(vl, fmt);
    vsnprintf(buf, sizeof(buf), fmt, vl);
    va_end(vl);
    if (c) {
        c->last_error = buf;
    }
    return 1;
}
} // namespace

int rc_comm_strip(const rc_rect *rect, int n, int rank, rc_rect *out);

namespace {
// Rows of the FRAME are owned by a fixed device (band r of the full height), whatever region a call renders: the
// running means of a pixel (full / half / AOV planes) must keep accumulating on the device that holds their history.
// Returns false when `rect` does not touch band r.
bool comm_band(const rc_comm *comm, int r, const rc_rect &rect, rc_rect *out) {
    const rc_ctx *c0 = comm->ctxs[0];
    const rc_rect frame{0, 0, c0->w, c0->h};
    rc_rect band;
    rc_comm_strip(&frame, int(comm->ctxs.size()), r, &band);
    const int y0 = rect.y > band.y ? rect.y : band.y;
    const int y1 = (rect.y + rect.h) < (band.y + band.h) ? (rect.y + rect.h) : (band.y + band.h);
    if (y1 <= y0 || rect.w <= 0) {
        return false;
    }
    *out = rc_rect{rect.x, y0, rect.w, y1 - y0};
    return true;
}
} // namespace

int rc_comm_strip(const rc_rect *rect, int n, int rank, rc_rect *out) {
    if (!rect || !out || n <= 0 || rank < 0 || rank >= n) {
        return 1;
    }
    const int base = rect->h / n, rem = rect->h % n;
    out->x = rect->x;
    out->w = rect->w;
    out->y = rect->y + rank * base + (rank < rem ? rank : rem);
    out->h = base + (rank < rem ? 1 : 0);
    return 0;
}

int rc_comm_init(rc_ctx **ctxs, int n, rc_comm **out_comm) {
    if (!ctxs || n <= 0 || !out_comm) {
        return 1;
    }
    auto *c = new rc_comm();
    for (int i = 0; i < n; ++i) {
        if (!ctxs[i]) {
            delete c;
            return 1;
        }
        for (int j = 0; j < i; ++j) {
            if (ctxs[j]->device == ctxs[i]->device) {
                delete c;
                return 1; // one context per device
            }
        }
        c->ctxs.push_back(ctxs[i]);
    }
    c->peer_ok.assign(n, 0);
    c->peer_ok[0] = 1;
    cudaSetDevice(ctxs[0]->device);
    for (int i = 1; i < n; ++i) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, ctxs[0]->device, ctxs[i]->device);
        if (can) {
            const cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[i]->device, 0);
            if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) {
                c->peer_ok[i] = 1;
            }
            cudaGetLastError();
        }
    }
    *out_comm = c;
    return 0;
}

void rc_comm_destroy(rc_comm *comm) { delete comm; }

const char *rc_comm_last_error(const rc_comm *comm) { return comm ? comm->last_error.c_str() : "null communicator"; }

int rc_comm_upload_scene(rc_comm *comm, const rc_scene_view *scene) {
    if (!comm) {
        return 1;
    }
    for (rc_ctx *ctx : comm->ctxs) { // replicated: the whole scene is needed by every strip
        if (rc_upload_scene(ctx, scene) != 0) {
            return comm_fail(comm, "device %d: %s", ctx->device, rc_last_error(ctx));
        }
    }
    return 0;
}

int rc_comm_upload_tables(rc_comm *comm, const uint32_t *pmj, int dims, int samples, const float *filter_table,
                          int filter_table_size) {
    if (!comm) {
        return 1;
    }
    for (rc_ctx *ctx : comm->ctxs) {
        if (rc_upload_tables(ctx, pmj, dims, samples, filter_table, filter_table_size) != 0) {
            return comm_fail(comm, "device %d: %s", ctx->device, rc_last_error(ctx));
        }
    }
    return 0;
}

int rc_comm_sync(rc_comm *comm) {
    if (!comm) {
        return 1;
    }
    int rc = 0;
    for (rc_ctx *ctx : comm->ctxs) {
        if (rc_sync(ctx) != 0) {
            rc = comm_fail(comm, "device %d: %s", ctx->device, rc_last_error(ctx));
        }
    }
    return rc;
}

int rc_comm_render(rc_comm *comm, const rc_pass_desc *pass) {
    if (!comm || !pass) {
        return 1;
    }
    const int n = int(comm->ctxs.size());
    for (int r = 0; r < n; ++r) {
        rc_ctx *ctx = comm->ctxs[r];
        if (ctx->w != comm->ctxs[0]->w || ctx->h != comm->ctxs[0]->h) {
            return comm_fail(comm, "rc_comm_render: context %d is sized %dx%d, context 0 %dx%d", r, ctx->w, ctx->h,
                             comm->ctxs[0]->w, comm->ctxs[0]->h);
        }
        rc_pass_desc p = *pass;
        if ((pass->flags & RC_RENDER_OUTPUT_SH) && !ctx->have_sh) {
            // every device holds the planes, also one whose band this pass does not touch: rc_gather reads them all
            cudaSetDevice(ctx->device);
            if (alloc_sh(ctx) || cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
                return comm_fail(comm, "device %d: %s", ctx->device, rc_last_error(ctx));
            }
        }
        if (!comm_band(comm, r, pass->rect, &p.rect)) {
            continue;
        }
        p.flags |= RC_RENDER_ASYNC; // every device gets its strip queued before anyone is waited for
        if (rc_render(ctx, &p) != 0) {
            return comm_fail(comm, "device %d: %s", ctx->device, rc_last_error(ctx));
        }
    }
    comm->last_rect = pass->rect;
    if ((pass->flags & RC_RENDER_ASYNC) == 0) {
        return rc_comm_sync(comm);
    }
    return 0;
}

int rc_gather(rc_comm *comm, int which, const rc_rect *rect, float *dst, int pitch) {
    if (!comm || !dst) {
        return 1;
    }
    const rc_rect full = rect ? *rect : comm->last_rect;
    const int n = int(comm->ctxs.size());
    if (pitch < full.w || full.w <= 0 || full.h <= 0) {
        return comm_fail(comm, "rc_gather: bad rect/pitch");
    }
    for (int r = 0; r < n; ++r) { // n independent device->host copies, each on its own device's link
        rc_rect s;
        if (!comm_band(comm, r, full, &s)) {
            continue;
        }
        float *d = dst + (size_t(s.y - full.y) * size_t(pitch)) * 4; // dst addresses the top-left pixel of `rect`
        if (rc_readback_async(comm->ctxs[r], which, &s, d, pitch) != 0) {
            return comm_fail(comm, "device %d: %s", comm->ctxs[r]->device, rc_last_error(comm->ctxs[r]));
        }
    }
    return rc_comm_sync(comm);
}

int rc_gather_device(rc_comm *comm, int which, const rc_rect *rect) {
    if (!comm) {
        return 1;
    }
    const rc_rect full = rect ? *rect : comm->last_rect;
    const int n = int(comm->ctxs.size());
    rc_ctx *c0 = comm->ctxs[0];
    float4 *dst = const_cast<float4 *>(plane_of(c0, which));
    if (!dst) {
        return comm_fail(comm, "rc_gather_device: buffer %d does not exist on device %d", which, c0->device);
    }
    if (rc_comm_sync(comm) != 0) {
        return 1;
    }
    for (int r = 1; r < n; ++r) {
        rc_ctx *cr = comm->ctxs[r];
        rc_rect s;
        if (!comm_band(comm, r, full, &s)) {
            continue;
        }
        const float4 *src = plane_of(cr, which);
        if (!src) {
            return comm_fail(comm, "rc_gather_device: buffer %d does not exist on device %d", which, cr->device);
        }
        cudaSetDevice(cr->device);
        cudaMemcpy3DPeerParms pp = {};
        pp.srcDevice = cr->device;
        pp.dstDevice = c0->device;
        pp.srcPtr = make_cudaPitchedPtr(const_cast<float4 *>(src), size_t(cr->w) * sizeof(float4), cr->w, cr->h);
        pp.dstPtr = make_cudaPitchedPtr(dst, size_t(c0->w) * sizeof(float4), c0->w, c0->h);
        pp.srcPos = make_cudaPos(size_t(s.x) * sizeof(float4), s.y, 0);
        pp.dstPos = make_cudaPos(size_t(s.x) * sizeof(float4), s.y, 0);
        pp.extent = make_cudaExtent(size_t(s.w) * sizeof(float4), s.h, 1);
        const cudaError_t e = cudaMemcpy3DPeerAsync(&pp, cr->stream); // NVLink when peer access is on, staged otherwise
        if (e != cudaSuccess) {
            return comm_fail(comm, "rc_gather_device: peer copy %d -> %d failed: %s", cr->device, c0->device,
                             cudaGetErrorString(e));
        }
    }
    return rc_comm_sync(comm);
}

int rc_comm_get_counters(rc_comm *comm, rc_counters *out) {
    if (!comm || !out) {
        return 1;
    }
    memset(out, 0, sizeof(*out));
    for (rc_ctx *ctx : comm->ctxs) {
        rc_counters c;
        if (rc_get_counters(ctx, &c) != 0) {
            return comm_fail(comm, "device %d: %s", ctx->device, rc_last_error(ctx));
        }
        out->primary_rays += c.primary_rays;
        out->secondary_rays += c.secondary_rays;
        out->shadow_rays += c.shadow_rays;
        out->nodes_visited += c.nodes_visited;
        out->leaves_tested += c.leaves_tested;
        out->samples = c.samples > out->samples ? c.samples : out->samples;
    }
    return 0;
}

int rc_readback_required_samples(rc_ctx *ctx, uint16_t *dst) {
    if (!ctx || !dst) {
        return 1;
    }
    cudaSetDevice(ctx->device);
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    CU_CHECK(ctx, cudaMemcpy(dst, ctx->fb.required_samples, size_t(ctx->w) * ctx->h * sizeof(uint16_t),
                             cudaMemcpyDeviceToHost));
    return 0;
}

int rc_enable_stats(rc_ctx *ctx, int enable) {
    if (!ctx) {
        return 1;
    }
    rc_sync(ctx);
    ctx->stats_enabled = enable != 0;
    return 0;
}

int rc_get_stats(rc_ctx *ctx, uint64_t us[11]) {
    if (!ctx || !us) {
        return 1;
    }
    rc_sync(ctx);
    memcpy(us, ctx->stats_us, sizeof(ctx->stats_us));
    return 0;
}

int rc_get_counters(rc_ctx *ctx, rc_counters *out) {
    if (!ctx || !out) {
        return 1;
    }
    cudaSetDevice(ctx->device);
    rc_sync(ctx);
    unsigned long long t[TOT_COUNT];
    CU_CHECK(ctx, cudaMemcpy(t, ctx->d_totals.get(), sizeof(t), cudaMemcpyDeviceToHost));
    out->primary_rays = t[TOT_PRIMARY];
    out->secondary_rays = t[TOT_SECONDARY];
    out->shadow_rays = t[TOT_SHADOW];
    out->nodes_visited = t[TOT_NODES];
    out->leaves_tested = t[TOT_LEAVES];
    out->samples = t[TOT_SAMPLES];
    return 0;
}

int rc_reset_stats(rc_ctx *ctx) {
    if (!ctx) {
        return 1;
    }
    cudaSetDevice(ctx->device);
    rc_sync(ctx);
    memset(ctx->stats_us, 0, sizeof(ctx->stats_us));
    memset(ctx->kernel_ms, 0, sizeof(ctx->kernel_ms));
    memset(ctx->kernel_launches, 0, sizeof(ctx->kernel_launches));
    CU_CHECK(ctx, cudaMemset(ctx->d_totals.get(), 0, TOT_COUNT * sizeof(unsigned long long)));
    return 0;
}

int rc_get_kernel_ms(rc_ctx *ctx, double ms[6], uint64_t launches[6]) {
    if (!ctx) {
        return 1;
    }
    rc_sync(ctx);
    for (int i = 0; i < KF_COUNT; ++i) {
        if (ms) {
            ms[i] = ctx->kernel_ms[i];
        }
        if (launches) {
            launches[i] = ctx->kernel_launches[i];
        }
    }
    return 0;
}

// ---- stage entry points ---------------------------------------------------------------------------------------------
int rc_stage_generate_primary_rays(rc_ctx *ctx, const rc_pass_desc *pass, void *rays_out, void *hits_out,
                                   int *count_out) {
    if (!ctx || !pass || !rays_out || !hits_out || !count_out) {
        return fail(ctx, "rc_stage_generate_primary_rays: null argument");
    }
    cudaSetDevice(ctx->device);
    KParams p;
    if (fill_params(ctx, pass, p)) {
        return 1;
    }
    CU_CHECK(ctx, cudaMemsetAsync(ctx->d_counters.get(), 0, CNT_TOTAL * sizeof(uint32_t), ctx->stream));
    const int n_pix_tiles = ((p.rect_w + 7) / 8) * ((p.rect_h + 3) / 4);
    k_raygen<<<(n_pix_tiles * 32 + 255) / 256, 256, 0, ctx->stream>>>(p, ctx->rays[0], ctx->hits);
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    uint32_t n = 0;
    if (get_counter(ctx, CNT_RAYS + 0, &n)) {
        return 1;
    }
    *count_out = int(n);
    if (n) {
        if (download_rays_aos(ctx, ctx->rays[0], static_cast<RayAoS *>(rays_out), int(n)) ||
            download_hits_aos(ctx, ctx->hits, static_cast<HitAoS *>(hits_out), int(n))) {
            return 1;
        }
    }
    return 0;
}

int rc_stage_generate_geo_rays(rc_ctx *ctx, const rc_pass_desc *pass, void *rays_out, void *hits_out, int *count_out) {
    if (!ctx || !pass || !rays_out || !hits_out || !count_out) {
        return fail(ctx, "rc_stage_generate_geo_rays: null argument");
    }
    if (pass->cam.type != 2) {
        return fail(ctx, "rc_stage_generate_geo_rays: camera type %u is not Geo (2)", pass->cam.type);
    }
    cudaSetDevice(ctx->device);
    KParams p;
    if (fill_params(ctx, pass, p) || ensure_geo_lists(ctx, pass)) {
        return 1;
    }
    CU_CHECK(ctx, cudaMemsetAsync(ctx->d_counters.get(), 0, CNT_TOTAL * sizeof(uint32_t), ctx->stream));
    const int n_pix_tiles = ((p.rect_w + 7) / 8) * ((p.rect_h + 3) / 4);
    k_raygen_geo<<<(n_pix_tiles * 32 + 255) / 256, 256, 0, ctx->stream>>>(p, geo_params(ctx, pass), ctx->rays[0], ctx->hits);
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    CU_CHECK(ctx, cudaGetLastError());
    uint32_t n = 0;
    if (get_counter(ctx, CNT_RAYS + 0, &n)) {
        return 1;
    }
    *count_out = int(n);
    if (n) {
        if (download_rays_aos(ctx, ctx->rays[0], static_cast<RayAoS *>(rays_out), int(n)) ||
            download_hits_aos(ctx, ctx->hits, static_cast<HitAoS *>(hits_out), int(n))) {
            return 1;
        }
    }
    return 0;
}

int rc_stage_trace_rays(rc_ctx *ctx, const rc_pass_desc *pass, void *rays, void *hits, int count, int trace_lights) {
    if (!ctx || !pass || !rays || !hits || count < 0) {
        return fail(ctx, "rc_stage_trace_rays: bad argument");
    }
    cudaSetDevice(ctx->device);
    if (size_t(count) > ctx->ray_capacity) {
        return fail(ctx, "rc_stage_trace_rays: %d rays exceed the capacity %zu (w*h)", count, ctx->ray_capacity);
    }
    KParams p;
    if (fill_params(ctx, pass, p)) {
        return 1;
    }
    if (count == 0) {
        return 0;
    }
    CU_CHECK(ctx, cudaMemsetAsync(ctx->d_counters.get(), 0, CNT_TOTAL * sizeof(uint32_t), ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (upload_rays_aos(ctx, ctx->rays[0], static_cast<const RayAoS *>(rays), count) ||
        upload_hits_aos(ctx, ctx->hits, static_cast<const HitAoS *>(hits), count) ||
        set_counter(ctx, CNT_RAYS + 0, uint32_t(count))) {
        return 1;
    }
    const int grid = persistent_grid(ctx, RT_TRACE_BLOCKS);
    if (ctx->scene_info.tlas_root != 0xffffffffu) {
        if (trace_lights && ctx->scene_info.visible_lights_count != 0) {
            k_trace_closest<true, false><<<grid, kTraceThreads, 0, ctx->stream>>>(p, ctx->rays[0], ctx->hits, 0, ctx->trace_fin_min);
        } else {
            k_trace_closest<false, false><<<grid, kTraceThreads, 0, ctx->stream>>>(p, ctx->rays[0], ctx->hits, 0, ctx->trace_fin_min);
        }
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    CU_CHECK(ctx, cudaGetLastError());
    return download_rays_aos(ctx, ctx->rays[0], static_cast<RayAoS *>(rays), count) ||
           download_hits_aos(ctx, ctx->hits, static_cast<HitAoS *>(hits), count);
}

int rc_stage_shade(rc_ctx *ctx, const rc_pass_desc *pass, int primary, int bounce, const void *rays, const void *hits,
                   int count, void *secondary_out, int *secondary_count, void *shadow_out, int *shadow_count) {
    if (!ctx || !pass || !rays || !hits || count < 0 || !secondary_out || !secondary_count || !shadow_out ||
        !shadow_count) {
        return fail(ctx, "rc_stage_shade: bad argument");
    }
    cudaSetDevice(ctx->device);
    if (size_t(count) > ctx->ray_capacity) {
        return fail(ctx, "rc_stage_shade: %d rays exceed the capacity %zu (w*h)", count, ctx->ray_capacity);
    }
    KParams p;
    if (fill_params(ctx, pass, p)) {
        return 1;
    }
    *secondary_count = *shadow_count = 0;
    if (count == 0) {
        return 0;
    }
    CU_CHECK(ctx, cudaMemsetAsync(ctx->d_counters.get(), 0, CNT_TOTAL * sizeof(uint32_t), ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (upload_rays_aos(ctx, ctx->rays[0], static_cast<const RayAoS *>(rays), count) ||
        upload_hits_aos(ctx, ctx->hits, static_cast<const HitAoS *>(hits), count) ||
        set_counter(ctx, CNT_RAYS + 0, uint32_t(count))) {
        return 1;
    }
    const int grid = persistent_grid(ctx, RT_SHADE_BLOCKS);
    const float mix_factor = 1.0f / float(p.iteration);
    if (primary) {
        const float lim = clamp_limit(p.ps.clamp_direct);
        launch_shade<true>(ctx, grid, ctx->stream, p, ctx->rays[0], ctx->rays[1], 0, lim, lim, mix_factor);
    } else {
        const float cd = (bounce == 1) ? p.ps.clamp_direct : p.ps.clamp_indirect;
        launch_shade<false>(ctx, grid, ctx->stream, p, ctx->rays[0], ctx->rays[1], 0, clamp_limit(cd),
                            clamp_limit(p.ps.clamp_indirect), mix_factor);
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    CU_CHECK(ctx, cudaGetLastError());
    uint32_t ns = 0, nh = 0;
    if (get_counter(ctx, CNT_RAYS + 1, &ns) || get_counter(ctx, CNT_SHADOW + 0, &nh)) {
        return 1;
    }
    *secondary_count = int(ns);
    *shadow_count = int(nh);
    if (ns && download_rays_aos(ctx, ctx->rays[1], static_cast<RayAoS *>(secondary_out), int(ns))) {
        return 1;
    }
    if (nh && download_shadow_aos(ctx, ctx->shadow, static_cast<ShadowRayAoS *>(shadow_out), int(nh))) {
        return 1;
    }
    return 0;
}

int rc_stage_trace_shadow_rays(rc_ctx *ctx, const rc_pass_desc *pass, const void *shadow_rays, int count,
                               float clamp_val) {
    if (!ctx || !pass || !shadow_rays || count < 0) {
        return fail(ctx, "rc_stage_trace_shadow_rays: bad argument");
    }
    cudaSetDevice(ctx->device);
    if (size_t(count) > ctx->ray_capacity) {
        return fail(ctx, "rc_stage_trace_shadow_rays: %d rays exceed the capacity %zu", count, ctx->ray_capacity);
    }
    KParams p;
    if (fill_params(ctx, pass, p)) {
        return 1;
    }
    if (count == 0) {
        return 0;
    }
    CU_CHECK(ctx, cudaMemsetAsync(ctx->d_counters.get(), 0, CNT_TOTAL * sizeof(uint32_t), ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (upload_shadow_aos(ctx, ctx->shadow, static_cast<const ShadowRayAoS *>(shadow_rays), count) ||
        set_counter(ctx, CNT_SHADOW + 0, uint32_t(count))) {
        return 1;
    }
    if (ctx->scene_info.tlas_root != 0xffffffffu) {
        k_trace_shadow<<<persistent_grid(ctx, RT_TRACE_BLOCKS), kTraceThreads, 0, ctx->stream>>>(p, ctx->shadow, 0, clamp_limit(clamp_val), ctx->trace_fin_min);
    }
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    CU_CHECK(ctx, cudaGetLastError());
    return 0;
}

int rc_stage_sort_rays(rc_ctx *ctx, void *rays, int count, uint32_t *hashes_out) {
    if (!ctx || !rays || count < 0) {
        return fail(ctx, "rc_stage_sort_rays: bad argument");
    }
    cudaSetDevice(ctx->device);
    if (size_t(count) > ctx->ray_capacity) {
        return fail(ctx, "rc_stage_sort_rays: %d rays exceed the capacity %zu", count, ctx->ray_capacity);
    }
    if (!ctx->have_scene) {
        return fail(ctx, "no scene uploaded");
    }
    if (count == 0) {
        return 0;
    }
    KParams p;
    memset(&p, 0, sizeof(p));
    p.counters = ctx->d_counters.get();
    CU_CHECK(ctx, cudaMemsetAsync(ctx->d_counters.get(), 0, CNT_TOTAL * sizeof(uint32_t), ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (upload_rays_aos(ctx, ctx->rays[0], static_cast<const RayAoS *>(rays), count) ||
        set_counter(ctx, CNT_RAYS + 1, uint32_t(count))) {
        return 1;
    }
    sort_rays(ctx->sort, p, ctx->rays[0], ctx->rays[1], 1, ctx->num_sms, /*have_hist*/ false,
              /*want_sorted_keys*/ true, ctx->stream);
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    CU_CHECK(ctx, cudaGetLastError());
    if (download_rays_aos(ctx, ctx->rays[1], static_cast<RayAoS *>(rays), count)) {
        return 1;
    }
    if (hashes_out) {
        CU_CHECK(ctx, cudaMemcpy(hashes_out, ctx->sort.keys_sorted.get(), size_t(count) * sizeof(uint32_t),
                                 cudaMemcpyDeviceToHost));
    }
    return 0;
}

void *rc_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void rc_host_free(void *p) {
    if (p) {
        cudaFreeHost(p);
    }
}

void *rc_device_ptr(rc_ctx *ctx, int which) {
    if (!ctx) {
        return nullptr;
    }
    return const_cast<float4 *>(plane_of(ctx, which));
}

int rc_event_record(rc_ctx *ctx, int slot) {
    if (!ctx || slot < 0 || slot >= 8) {
        return fail(ctx, "rc_event_record: bad slot");
    }
    cudaSetDevice(ctx->device);
    CU_CHECK(ctx, cudaEventRecord(ctx->user_events[slot], ctx->stream));
    return 0;
}

int rc_event_elapsed_ms(rc_ctx *ctx, int a, int b, float *ms) {
    if (!ctx || !ms || a < 0 || a >= 8 || b < 0 || b >= 8) {
        return fail(ctx, "rc_event_elapsed_ms: bad argument");
    }
    cudaSetDevice(ctx->device);
    CU_CHECK(ctx, cudaEventSynchronize(ctx->user_events[b]));
    CU_CHECK(ctx, cudaEventElapsedTime(ms, ctx->user_events[a], ctx->user_events[b]));
    return 0;
}

int rc_abi_sizeof(int which) {
    switch (which) {
    case 0: return int(sizeof(rc_array));
    case 1: return int(sizeof(rc_scene_view));
    case 2: return int(sizeof(rc_camera));
    case 3: return int(sizeof(rc_rect));
    case 4: return int(sizeof(rc_pass_desc));
    case 5: return int(sizeof(rc_counters));
    case 6: return int(sizeof(rc_texture));
    default: return -1;
    }
}

} // extern "C"
