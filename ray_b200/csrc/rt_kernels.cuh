// rt_kernels.cuh -- the wavefront kernels: raygen, closest-hit trace, shade, shadow trace, resolve.
//
// One sample of one region = the kernel sequence Cpu::Renderer<P>::RenderScene runs on the host (reference
// internal/RendererCPU.h:374-659), enqueued on one stream with NO host round trip: every kernel reads its work size
// from a device counter written by its producer, so bounces that have run dry cost an empty launch.
//
// Stream layout in HBM (all SoA, 16-byte planes, one coalesced 512 B request per warp per plane):
//   ray    72 B  = float4 {o.xyz, cone_width} | float4 {d.xyz, cone_spread} | float4 {c.rgb, pdf} | float4 ior[4]
//                  | uint2 {xy, depth}                                              (Ref::ray_data_t, CoreRef.h:57-71)
//   hit    20 B  = float4 {t, u, v, bits(prim_index)} | int obj_index              (Ref::hit_data_t, CoreRef.h:89-105)
//   shadow 48 B  = float4 {o.xyz, bits(depth)} | float4 {d.xyz, dist} | float4 {c.rgb, bits(xy)}   (shadow_ray_t)
#pragma once

#include "rt_shade.cuh"

// Launch shapes of the persistent kernels (measured on hall-250k, profiles/README.md "launch shape sweep"):
//  * k_shade is instruction-FETCH bound (177 KB of straight-line SASS walked once per ray, I-cache hit rate 65 %):
//    big blocks whose warps are re-aligned with __syncthreads() between the phases walk the same cache lines together
//    (119 -> 82 ms per 16 samples); 64 registers / thread costs spills but doubles the resident warps.
//  * the trace kernels (rt_trace.cuh) run RT_TRACE_BLOCKS resident 128-thread blocks per SM.
#ifndef RT_SHADE_THREADS
#define RT_SHADE_THREADS 512
#endif
#ifndef RT_SHADE_BLOCKS
#define RT_SHADE_BLOCKS 2
#endif
#ifndef RT_SHADE_SYNC
#define RT_SHADE_SYNC 1
#endif
#ifndef RT_TRACE_BLOCKS
#define RT_TRACE_BLOCKS 6
#endif

namespace rt {

struct RayBuf {
    float4 *o_cw, *d_cs, *c_pdf, *ior;
    uint2 *xy_depth;
};
struct HitBuf {
    float4 *tuvp;
    int *obj;
};
struct ShadowBuf {
    float4 *o_depth, *d_dist, *c_xy;
};

constexpr int kMaxBounces = 16;
// per-sample counter block (uint32), zeroed at the start of every sample
enum : int {
    CNT_RAYS = 0,                         // [kMaxBounces] rays entering the closest-hit trace of bounce b (0 = primary)
    CNT_SHADOW = CNT_RAYS + kMaxBounces,  // [kMaxBounces] shadow rays produced by the shade of bounce b
    CNT_HEAD_TRACE = CNT_SHADOW + kMaxBounces,
    CNT_HEAD_SHADOW = CNT_HEAD_TRACE + kMaxBounces,
    CNT_HEAD_SHADE = CNT_HEAD_SHADOW + kMaxBounces,
    CNT_TOTAL = CNT_HEAD_SHADE + kMaxBounces
};
// persistent totals (uint64)
enum : int { TOT_PRIMARY = 0, TOT_SECONDARY, TOT_SHADOW, TOT_NODES, TOT_LEAVES, TOT_SAMPLES, TOT_COUNT };

// ---- sort key of the inter-bounce ray reordering (rt_sort.cuh) -----------------------------------------------------
// key = direction cell (major) | Morton code of the origin in a (2^kSortCellBits)^3 grid over the scene bounds.
// Direction: 8x8 octahedral cells (6 bits); origin: 16^3 cells (12 bits) -> 18-bit key, 262144 bins.  Measured on
// hall-250k (ms per sample, profiles/README.md): octant + 12-bit Morton 14.35, 6 + 9 bits 13.85, 6 + 12 bits 13.52,
// 8 + 12 bits 13.48 (4x the histogram memory), octant + 15 / 18-bit Morton: no gain -- direction resolution is what pays.
#ifndef RT_SORT_CELL_BITS
#define RT_SORT_CELL_BITS 4
#endif
constexpr int kSortCellBits = RT_SORT_CELL_BITS;
#ifndef RT_SORT_DIR_BITS
#define RT_SORT_DIR_BITS 6 // 3 = octant; 6 / 8 = 8x8 / 16x16 octahedral cells
#endif
constexpr int kSortDirBits = RT_SORT_DIR_BITS;
constexpr int kSortKeyBits = kSortDirBits + 3 * kSortCellBits;
constexpr int kSortBins = 1 << kSortKeyBits;

struct SortGrid {
    float min_x, min_y, min_z, inv_x, inv_y, inv_z;
};

RT_DEV uint32_t spread3(uint32_t v) { // bit i -> bit 3 i
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < kSortCellBits; ++i) {
        r |= ((v >> i) & 1u) << (3 * i);
    }
    return r;
}

RT_DEV uint32_t ray_sort_key(float4 o, float4 d, const SortGrid &g) {
    constexpr int hi = (1 << kSortCellBits) - 1;
    const int cx = min(max(int((o.x - g.min_x) * g.inv_x), 0), hi);
    const int cy = min(max(int((o.y - g.min_y) * g.inv_y), 0), hi);
    const int cz = min(max(int((o.z - g.min_z) * g.inv_z), 0), hi);
    const uint32_t morton = spread3(uint32_t(cx)) | (spread3(uint32_t(cy)) << 1) | (spread3(uint32_t(cz)) << 2);
#if RT_SORT_DIR_BITS == 3
    const uint32_t oct = (d.x < 0.0f ? 1u : 0u) | (d.y < 0.0f ? 2u : 0u) | (d.z < 0.0f ? 4u : 0u);
#else
    // octahedral map of the direction, 2^(bits/2) x 2^(bits/2) cells
    const float inv = 1.0f / (fabsf(d.x) + fabsf(d.y) + fabsf(d.z) + 1e-20f);
    float ux = d.x * inv, uy = d.y * inv;
    if (d.z < 0.0f) {
        const float tx = (1.0f - fabsf(uy)) * (ux >= 0.0f ? 1.0f : -1.0f), ty = (1.0f - fabsf(ux)) * (uy >= 0.0f ? 1.0f : -1.0f);
        ux = tx;
        uy = ty;
    }
    constexpr int dres = 1 << (kSortDirBits / 2);
    const int qx = min(max(int((ux * 0.5f + 0.5f) * float(dres)), 0), dres - 1),
              qy = min(max(int((uy * 0.5f + 0.5f) * float(dres)), 0), dres - 1);
    const uint32_t oct = uint32_t(qy * dres + qx);
#endif
#if defined(RT_SORT_ORIGIN_MAJOR) && RT_SORT_ORIGIN_MAJOR
    return (morton << kSortDirBits) | oct;
#else
    return (oct << (3 * kSortCellBits)) | morton;
#endif
}

struct CamParams { // derived once per pass on the host (tanf/atanf come from the host libm like the reference's)
    v3 origin, fwd, side, up;
    float shift_x, shift_y;
    float k, fov_k, spread_angle, focus_distance;
    float fstop, focal_length, sensor_height, lens_rotation, lens_ratio;
    int lens_blades;
    float clip_start, clip_end;
    int filter; // 0 = Box
};

struct FrameBufs {
    float4 *temp, *full, *half, *raw, *final, *base_color, *depth_normals;
    uint16_t *required_samples;
    int w, h;
};

// pass flags as k_shade sees them (include/ray_cuda.h RC_RENDER_*): LIGHTING_ONLY acts in the PRIMARY instantiation
// only; DROP_COL is set on the bounce-1 launch of a SKIP_DIRECT pass.  (NO_BACKGROUND is k_no_background: the
// test inside k_shade cost the register-capped PRIMARY variants spill stores.)
enum : uint32_t { KP_LIGHTING_ONLY = 1u, KP_DROP_COL = 4u };

struct KParams {
    ShadeScene sc;
    PassSettings ps;
    CamParams cam;
    FrameBufs fb;
    const float *filter_table;
    uint32_t *counters;            // CNT_TOTAL
    unsigned long long *totals;    // TOT_COUNT
    int rect_x, rect_y, rect_w, rect_h;
    int iteration;
    uint32_t rand_seed;
    // ray reordering (rt_sort.cuh): when sort_hist != nullptr, k_shade also emits the sort key of every secondary ray
    // it stores and counts it in the histogram of the list it appends to (sort_hist + list * kSortBins)
    SortGrid sort_grid;
    uint32_t *sort_keys;
    uint32_t *sort_hist;
    uint32_t flags; // KP_* (pass flags that reach the shading kernels; set per launch by the host)
};

RT_DEV RayD load_ray(const RayBuf &b, uint32_t i) {
    RayD r;
    const float4 a = b.o_cw[i], d = b.d_cs[i], c = b.c_pdf[i], io = b.ior[i];
    const uint2 xd = b.xy_depth[i];
    r.o = v3{a.x, a.y, a.z};
    r.cone_width = a.w;
    r.d = v3{d.x, d.y, d.z};
    r.cone_spread = d.w;
    r.c = v3{c.x, c.y, c.z};
    r.pdf = c.w;
    r.ior[0] = io.x;
    r.ior[1] = io.y;
    r.ior[2] = io.z;
    r.ior[3] = io.w;
    r.xy = xd.x;
    r.depth = xd.y;
    return r;
}

RT_DEV void store_ray(const RayBuf &b, uint32_t i, const RayD &r) {
    b.o_cw[i] = make_float4(r.o.x, r.o.y, r.o.z, r.cone_width);
    b.d_cs[i] = make_float4(r.d.x, r.d.y, r.d.z, r.cone_spread);
    b.c_pdf[i] = make_float4(r.c.x, r.c.y, r.c.z, r.pdf);
    b.ior[i] = make_float4(r.ior[0], r.ior[1], r.ior[2], r.ior[3]);
    b.xy_depth[i] = make_uint2(r.xy, r.depth);
}

RT_DEV Hit load_hit(const HitBuf &b, uint32_t i) {
    const float4 h = b.tuvp[i];
    Hit r;
    r.t = h.x;
    r.u = h.y;
    r.v = h.z;
    r.prim = __float_as_int(h.w);
    r.obj = b.obj[i];
    return r;
}

RT_DEV void store_hit(const HitBuf &b, uint32_t i, const Hit &h) {
    b.tuvp[i] = make_float4(h.t, h.u, h.v, __int_as_float(h.prim));
    b.obj[i] = h.obj;
}

RT_DEV void store_shadow(const ShadowBuf &b, uint32_t i, const ShadowRayD &s) {
    b.o_depth[i] = make_float4(s.o.x, s.o.y, s.o.z, __uint_as_float(s.depth));
    b.d_dist[i] = make_float4(s.d.x, s.d.y, s.d.z, s.dist);
    b.c_xy[i] = make_float4(s.c.x, s.c.y, s.c.z, __uint_as_float(s.xy));
}

RT_DEV ShadowRayD load_shadow(const ShadowBuf &b, uint32_t i) {
    const float4 a = b.o_depth[i], d = b.d_dist[i], c = b.c_xy[i];
    ShadowRayD s;
    s.o = v3{a.x, a.y, a.z};
    s.depth = __float_as_uint(a.w);
    s.d = v3{d.x, d.y, d.z};
    s.dist = d.w;
    s.c = v3{c.x, c.y, c.z};
    s.xy = __float_as_uint(c.w);
    return s;
}

// warp-aggregated append: returns the slot of this lane's record (valid only where pred)
RT_DEV uint32_t warp_append(uint32_t *counter, bool pred) {
    const uint32_t mask = __ballot_sync(0xffffffffu, pred);
    if (mask == 0) {
        return 0;
    }
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) {
        base = atomicAdd(counter, uint32_t(__popc(mask)));
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + __popc(mask & ((1u << lane) - 1u));
}

// ---- GeneratePrimaryRays (reference internal/CoreRef.cpp:1429-1553) -----------------------------------------------
RT_DEV float lookup_filter_table(const float *__restrict__ table, float x) {
    x *= (kFilterTableSize - 1);
    const int index = min(int(x), kFilterTableSize - 1);
    const int nindex = min(index + 1, kFilterTableSize - 1);
    const float t = x - float(index);
    const float data0 = table[index];
    if (t == 0.0f) {
        return data0;
    }
    const float data1 = table[nindex];
    return (1.0f - t) * data0 + t * data1;
}

RT_DEV float ngon_rad(float theta, float n) {
    return portable_cos(kPi / n) / portable_cos(theta - (2.0f * kPi / n) * floorf((n * theta + kPi) / (2.0f * kPi)));
}

__global__ void __launch_bounds__(256) k_raygen(KParams p, RayBuf rays, HitBuf hits) {
    // one warp = one 8x4 pixel tile of the rect, so a warp's 32 primary rays form a compact frustum
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t tile = gid >> 5, lane = gid & 31;
    const uint32_t tiles_x = (p.rect_w + 7) / 8, tiles_y = (p.rect_h + 3) / 4;
    bool active = tile < tiles_x * tiles_y;
    int x = 0, y = 0;
    if (active) {
        x = p.rect_x + int(tile % tiles_x) * 8 + int(lane & 7);
        y = p.rect_y + int(tile / tiles_x) * 4 + int(lane >> 3);
        active = (x < p.rect_x + p.rect_w) && (y < p.rect_y + p.rect_h);
    }
    if (active && p.fb.required_samples[y * p.fb.w + x] < p.iteration) {
        active = false;
    }
    RayD r;
    float hit_t = 0.0f;
    if (active) {
        const CamParams &cam = p.cam;
        float fx = float(x), fy = float(y);
        const uint32_t px_hash = hash_u32((uint32_t(x) << 16) | uint32_t(y));
        const uint32_t rand_hash = hash_combine(px_hash, p.rand_seed);
        const v2 filter_rand = rand2d(kRandDimFilter, rand_hash, p.iteration - 1, p.sc.rand_seq);
        float rx = filter_rand.x, ry = filter_rand.y;
        if (cam.filter != 0) {
            rx = lookup_filter_table(p.filter_table, rx);
            ry = lookup_filter_table(p.filter_table, ry);
        }
        fx += rx;
        fy += ry;
        float ox = 0.0f, oy = 0.0f;
        if (cam.fstop > 0.0f) {
            const v2 lens_rand = rand2d(kRandDimLens, rand_hash, p.iteration - 1, p.sc.rand_seq);
            ox = 2.0f * lens_rand.x - 1.0f;
            oy = 2.0f * lens_rand.y - 1.0f;
            if (ox != 0.0f && oy != 0.0f) {
                float theta, rr;
                if (fabsf(ox) > fabsf(oy)) {
                    rr = ox;
                    theta = 0.25f * kPi * (oy / ox);
                } else {
                    rr = oy;
                    theta = 0.5f * kPi - 0.25f * kPi * (ox / oy);
                }
                if (cam.lens_blades) {
                    rr *= ngon_rad(theta, float(cam.lens_blades));
                }
                theta += cam.lens_rotation;
                const v2 sc = portable_sincos(theta);
                ox = 0.5f * rr * sc.y / cam.lens_ratio;
                oy = 0.5f * rr * sc.x;
            }
            const float coc = 0.5f * (cam.focal_length / cam.fstop);
            ox *= coc * cam.sensor_height;
            oy *= coc * cam.sensor_height;
        }
        const v3 origin = cam.origin + cam.side * ox + cam.up * oy;
        // get_pix_dir
        const float px = 2 * cam.fov_k * (fx / float(p.fb.w) + cam.shift_x / cam.k) - cam.fov_k;
        const float py = 2 * cam.fov_k * (-fy / float(p.fb.h) + cam.shift_y) + cam.fov_k;
        const v3 pt = cam.origin + cam.k * px * cam.side + py * cam.up + cam.focus_distance * cam.fwd;
        const v3 d = normalize(pt - origin);
        const float clip_start = cam.clip_start / dot(d, cam.fwd);
        r.o = v3{origin.x + d.x * clip_start, origin.y + d.y * clip_start, origin.z + d.z * clip_start};
        r.d = d;
        r.c = v3{1.0f, 1.0f, 1.0f};
        r.ior[0] = r.ior[1] = r.ior[2] = r.ior[3] = -1.0f;
        r.cone_width = 0.0f;
        r.cone_spread = cam.spread_angle;
        r.pdf = 1e6f;
        r.xy = (uint32_t(x) << 16) | uint32_t(y);
        r.depth = (uint32_t(RAY_CAMERA) << 28);
        hit_t = (cam.clip_end / dot(d, cam.fwd)) - clip_start;
    }
    const uint32_t slot = warp_append(&p.counters[CNT_RAYS + 0], active);
    if (active) {
        store_ray(rays, slot, r);
        Hit h;
        h.obj = -1;
        h.prim = -1;
        h.t = hit_t;
        h.u = 0.0f;
        h.v = -1.0f;
        store_hit(hits, slot, h);
    }
}

// ---- ShadePrimary / ShadeSecondary (ShadeRef.cpp:1654-1737) --------------------------------------------------------
// `bounce` = index of the ray list being shaded (0 = primary).  Secondary rays go to list bounce+1.
template <bool PRIMARY, bool TEX>
__global__ void __launch_bounds__(RT_SHADE_THREADS, RT_SHADE_BLOCKS)
    k_shade(KParams p, RayBuf rays, HitBuf hits, RayBuf out_rays, ShadowBuf out_shadow, int bounce, float limit0,
            float limit1, float mix_factor) {
    const uint32_t count = p.counters[CNT_RAYS + bounce];
    uint32_t tl_stack[kMaxStack];
    float tl_factors[kMaxStack];
    // block-uniform trip count, so the warps of a block can be kept in step (RT_SHADE_SYNC): the shading code is a
    // long straight line walked once per ray, and warps that walk it together share instruction-cache lines
    for (uint32_t base = blockIdx.x * blockDim.x; base < count; base += gridDim.x * blockDim.x) {
#if RT_SHADE_SYNC
        __syncthreads();
#endif
        const uint32_t i = base + threadIdx.x;
        const bool valid = i < count;
        ShadeOut out;
        out.has_secondary = out.has_shadow = false;
        uint32_t xy = 0;
        RayD ray;
        Hit inter;
        MatCtx c;
        bool more = false;
        if (valid) {
            ray = load_ray(rays, i);
            inter = load_hit(hits, i);
            xy = ray.xy;
            more = shade_surface_a(TEX, p.ps, limit0, inter, ray, p.rand_seed, p.iteration, p.sc, tl_stack, tl_factors, c, out);
        }
#if RT_SHADE_SYNC
        __syncthreads();
#endif
        if (more) {
            shade_surface_l(TEX, c);
        }
#if RT_SHADE_SYNC
        __syncthreads();
#endif
        if (more) {
            shade_surface_b(TEX, c, limit1, out, PRIMARY && (p.flags & KP_LIGHTING_ONLY));
        }
        if (valid) {
            const int x = int((xy >> 16) & 0xffff), y = int(xy & 0xffff);
            const int pix = y * p.fb.w + x;
            if (PRIMARY) {
                p.fb.temp[pix] = make_float4(out.col.x, out.col.y, out.col.z, out.col.w);
                // running means of the AOVs (ShadeRef.cpp:1677-1698)
                float4 nb = make_float4(out.base_color.x, out.base_color.y, out.base_color.z, 0.0f);
                const float norm_factor = fmaxf(fmaxf(nb.x, nb.y), fmaxf(nb.z, 1.0f));
                nb.x /= norm_factor;
                nb.y /= norm_factor;
                nb.z /= norm_factor;
                nb.w /= norm_factor;
                float4 ob = p.fb.base_color[pix];
                ob.x += (nb.x - ob.x) * mix_factor;
                ob.y += (nb.y - ob.y) * mix_factor;
                ob.z += (nb.z - ob.z) * mix_factor;
                ob.w += (nb.w - ob.w) * mix_factor;
                p.fb.base_color[pix] = ob;
                const float4 nd = make_float4(out.aov_normal.x, out.aov_normal.y, out.aov_normal.z, out.aov_depth);
                float4 od = p.fb.depth_normals[pix];
                od.x += (nd.x - od.x) * mix_factor;
                od.y += (nd.y - od.y) * mix_factor;
                od.z += (nd.z - od.z) * mix_factor;
                od.w += (nd.w - od.w) * mix_factor;
                p.fb.depth_normals[pix] = od;
            } else if (!(p.flags & KP_DROP_COL)) {
                float4 o = p.fb.temp[pix];
                o.x += out.col.x;
                o.y += out.col.y;
                o.z += out.col.z;
                o.w += 0.0f;
                p.fb.temp[pix] = o;
            }
        }
        const uint32_t s_slot = warp_append(&p.counters[CNT_RAYS + bounce + 1], out.has_secondary);
        if (out.has_secondary) {
            store_ray(out_rays, s_slot, out.new_ray);
            if (p.sort_hist) {
                const RayD &nr = out.new_ray;
                const uint32_t key = ray_sort_key(make_float4(nr.o.x, nr.o.y, nr.o.z, 0.0f),
                                                  make_float4(nr.d.x, nr.d.y, nr.d.z, 0.0f), p.sort_grid);
                p.sort_keys[s_slot] = key;
                atomicAdd(&p.sort_hist[size_t(bounce + 1) * kSortBins + key], 1u);
            }
            // initial hit record for the next trace (RendererCPU.h:532-535: `intersections[i] = {}`)
        }
        const uint32_t h_slot = warp_append(&p.counters[CNT_SHADOW + bounce], out.has_shadow);
        if (out.has_shadow) {
            store_shadow(out_shadow, h_slot, out.sh_r);
        }
    }
}

// RC_RENDER_NO_BACKGROUND, after the primary shade: camera rays that missed contribute (0,0,0)
__global__ void k_no_background(KParams p, RayBuf rays, HitBuf hits) {
    const uint32_t count = p.counters[CNT_RAYS + 0];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        if (hits.tuvp[i].z < 0.0f) {
            const uint32_t xy = rays.xy_depth[i].x;
            float4 &t = p.fb.temp[int(xy & 0xffff) * p.fb.w + int(xy >> 16)];
            t.x = t.y = t.z = 0.0f;
        }
    }
}

// Reset the hit records of a ray list to "no intersection" (hit_data_t default ctor, CoreRef.h:97-104)
__global__ void k_init_hits(KParams p, HitBuf hits, int bounce) {
    const uint32_t count = p.counters[CNT_RAYS + bounce];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        hits.tuvp[i] = make_float4(kMaxDist, 0.0f, -1.0f, __int_as_float(-1));
        hits.obj[i] = -1;
    }
}

// ---- accumulate + tonemap + variance (RendererCPU.h:607-658, TonemapRef.h) ---------------------------------------
RT_DEV float tonemap_standard(float c) {
    if (c < 0.0031308f) {
        return 12.92f * c;
    }
    return 1.055f * libm_powf(c, (1.0f / 2.4f)) - 0.055f;
}

// TonemapFilmic (TonemapRef.cpp:29-66): the AgX / Filmic view transforms are 48^3 tables of packed 10-10-10-2 colours
// (handed in through rc_set_view_lut -- the tables are the caller's data), sampled with a trilinear fetch
constexpr int kViewLutDims = 48;
RT_DEV v3 fetch_view_lut(const uint32_t *__restrict__ lut, int ix, int iy, int iz) {
    const uint32_t v = lut[(iz * kViewLutDims + iy) * kViewLutDims + ix];
    return v3{float(int(v & 0x3ffu)) * (1.0f / 1023.0f), float(int((v >> 10) & 0x3ffu)) * (1.0f / 1023.0f),
              float(int((v >> 20) & 0x3ffu)) * (1.0f / 1023.0f)};
}
RT_DEV v3 tonemap_filmic(const uint32_t *__restrict__ lut, v3 color) {
    const v3 uv = v3{color.x / (color.x + 1.0f) * float(kViewLutDims - 1), color.y / (color.y + 1.0f) * float(kViewLutDims - 1),
                     color.z / (color.z + 1.0f) * float(kViewLutDims - 1)};
    // ivec4(uv) truncates; the clamp only guards table reads for non-finite colours (the reference would read out of bounds)
    const int ix = min(max(int(uv.x), 0), kViewLutDims - 1), iy = min(max(int(uv.y), 0), kViewLutDims - 1),
              iz = min(max(int(uv.z), 0), kViewLutDims - 1);
    const float fx = fractf(uv.x), fy = fractf(uv.y), fz = fractf(uv.z);
    const int jx = min(ix + 1, kViewLutDims - 1), jy = min(iy + 1, kViewLutDims - 1), jz = min(iz + 1, kViewLutDims - 1);
    const v3 c000 = fetch_view_lut(lut, ix, iy, iz), c001 = fetch_view_lut(lut, jx, iy, iz),
             c010 = fetch_view_lut(lut, ix, jy, iz), c011 = fetch_view_lut(lut, jx, jy, iz),
             c100 = fetch_view_lut(lut, ix, iy, jz), c101 = fetch_view_lut(lut, jx, iy, jz),
             c110 = fetch_view_lut(lut, ix, jy, jz), c111 = fetch_view_lut(lut, jx, jy, jz);
    const v3 c00x = (1.0f - fx) * c000 + fx * c001, c01x = (1.0f - fx) * c010 + fx * c011,
             c10x = (1.0f - fx) * c100 + fx * c101, c11x = (1.0f - fx) * c110 + fx * c111;
    const v3 c0xx = (1.0f - fy) * c00x + fy * c01x, c1xx = (1.0f - fy) * c10x + fy * c11x;
    return (1.0f - fz) * c0xx + fz * c1xx;
}

// Tonemap (TonemapRef.h:36-48) without the final saturate: view transform (Standard when lut == nullptr), then 1/gamma
struct DisplayXf {
    const uint32_t *lut;
    float inv_gamma;
};
RT_DEV void display_transform(const DisplayXf &xf, float4 &c) {
    if (xf.lut == nullptr) {
        c.x = tonemap_standard(c.x);
        c.y = tonemap_standard(c.y);
        c.z = tonemap_standard(c.z);
    } else {
        const v3 t = tonemap_filmic(xf.lut, v3{c.x, c.y, c.z});
        c.x = t.x;
        c.y = t.y;
        c.z = t.z;
    }
    if (xf.inv_gamma != 1.0f) {
        c.x = libm_powf(c.x, xf.inv_gamma);
        c.y = libm_powf(c.y, xf.inv_gamma);
        c.z = libm_powf(c.z, xf.inv_gamma);
    }
}

__global__ void __launch_bounds__(256) k_resolve(KParams p, float exposure_mul, float mix_factor, float half_mix_factor,
                                                 int is_class_a, DisplayXf xf, float variance_threshold) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p.rect_w * p.rect_h) {
        return;
    }
    const int x = p.rect_x + idx % p.rect_w, y = p.rect_y + idx / p.rect_w;
    const int pix = y * p.fb.w + x;
    float4 full = p.fb.full[pix];
    float4 half = p.fb.half[pix];
    if (!(p.fb.required_samples[pix] < p.iteration)) {
        const float4 t = p.fb.temp[pix];
        const float4 nv = make_float4(t.x * exposure_mul, t.y * exposure_mul, t.z * exposure_mul, t.w * 1.0f);
        full.x += (nv.x - full.x) * mix_factor;
        full.y += (nv.y - full.y) * mix_factor;
        full.z += (nv.z - full.z) * mix_factor;
        full.w += (nv.w - full.w) * mix_factor;
        p.fb.full[pix] = full;
        if (is_class_a) {
            half.x += (nv.x - half.x) * half_mix_factor;
            half.y += (nv.y - half.y) * half_mix_factor;
            half.z += (nv.z - half.z) * half_mix_factor;
            half.w += (nv.w - half.w) * half_mix_factor;
            p.fb.half[pix] = half;
        }
    }
    p.fb.raw[pix] = full;
    float4 c = full;
    display_transform(xf, c);
    // saturate = _mm_max_ps(0, _mm_min_ps(c, 1))
    c.x = sse_max(0.0f, sse_min(c.x, 1.0f));
    c.y = sse_max(0.0f, sse_min(c.y, 1.0f));
    c.z = sse_max(0.0f, sse_min(c.z, 1.0f));
    c.w = sse_max(0.0f, sse_min(c.w, 1.0f));
    p.fb.final[pix] = c;

    // variance estimate from the full/half pair
    float4 a = make_float4(sse_max(2.0f * full.x - half.x, 0.0f), sse_max(2.0f * full.y - half.y, 0.0f),
                           sse_max(2.0f * full.z - half.z, 0.0f), sse_max(2.0f * full.w - half.w, 0.0f));
    const float da = fmaxf(a.x, fmaxf(a.y, a.z)) + 1.0f;
    a = make_float4(a.x / da, a.y / da, a.z / da, a.w / da);
    const float db = fmaxf(half.x, fmaxf(half.y, half.z)) + 1.0f;
    const float4 b = make_float4(half.x / db, half.y / db, half.z / db, half.w / db);
    const float4 var = make_float4(0.5f * (a.x - b.x) * (a.x - b.x), 0.5f * (a.y - b.y) * (a.y - b.y),
                                   0.5f * (a.z - b.z) * (a.z - b.z), 0.5f * (a.w - b.w) * (a.w - b.w));
    p.fb.temp[pix] = var;
    if ((var.x >= variance_threshold) | (var.y >= variance_threshold) | (var.z >= variance_threshold) |
        (var.w >= variance_threshold)) {
        p.fb.required_samples[pix] = uint16_t(p.iteration + 1);
    }
}

// add this sample's counters into the persistent 64-bit totals: the rays of the bounces that were traced, and the
// shadow rays of the lists in `shadow_traced` (bit b = list b; the pass flags can skip a list)
__global__ void k_accumulate_totals(KParams p, int max_bounces, uint32_t shadow_traced) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        p.totals[TOT_PRIMARY] += p.counters[CNT_RAYS + 0];
        unsigned long long sec = 0, sh = 0;
        for (int b = 1; b <= max_bounces; ++b) {
            sec += p.counters[CNT_RAYS + b];
        }
        for (int b = 0; b <= max_bounces; ++b) {
            if ((shadow_traced >> b) & 1u) {
                sh += p.counters[CNT_SHADOW + b];
            }
        }
        p.totals[TOT_SECONDARY] += sec;
        p.totals[TOT_SHADOW] += sh;
        p.totals[TOT_SAMPLES] += 1;
    }
}

} // namespace rt
