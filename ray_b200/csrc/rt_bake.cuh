// rt_bake.cuh -- lightmap baking: the texture-space (Geo) camera and the L1 SH output (include/ray_cuda.h states the
// semantics).
//
// Geo camera.  A texel's sample point is rasterised against the uv triangles of one mesh: per texel, a candidate list
// (CSR: offsets[w*h + 1], tri ids) holds the triangles whose texel-clamped uv bounding box overlaps the texel.  The
// lists are built once per (scene, triangle range, frame size) by
//   k_geo_box_total  thread per triangle: sum of the box areas (checked against the memory cap before anything else)
//   k_geo_count      warp per triangle striding its box (a big triangle does not serialise one thread)
//   exclusive scan   (cub)
//   k_geo_fill       warp per triangle, same walk, appends its id through a per-texel cursor
// The order inside a list is not deterministic and does not need to be: the winner is the MINIMUM containing index.
// k_raygen_geo replaces k_raygen + the primary closest-hit trace: it emits the ray AND its hit record.
//
// SH.  Three small per-sample kernels around the unchanged shade / resolve kernels, all reading list sizes from the
// device counters:
//   k_sh_primary  after the primary shade: snapshot temp (= E0) and scatter the bounce-1 ray directions by pixel
//   k_sh_direct   after the bounce-0 shadow trace: D = temp - E0, and the shadow-ray directions of list 0
//   k_sh_resolve  before k_resolve: I = temp - (E0 + D), running mean of the three coefficient planes
// A scattered direction carries the sample's tag in w, so a pixel that got no ray this sample sees no direction.
#pragma once

#include "rt_kernels.cuh"

namespace rt {

constexpr uint64_t kGeoMaxEntries = 1ull << 28; // candidate-list entries (4 B each): 1 GiB
constexpr float kGeoMinArea2 = 2e-12f;            // |doubled uv area| in texel^2 below which a triangle never wins

struct GeoTarget {
    const Vertex *vertices;
    const uint32_t *vtx_indices;
    uint32_t tri_first, tri_count;
    int w, h;
};

// uv corners of triangle `tri` in texel units
RT_DEV void geo_uv(const GeoTarget &g, uint32_t tri, v2 &a, v2 &b, v2 &c) {
    const Vertex &v0 = g.vertices[g.vtx_indices[tri * 3 + 0]];
    const Vertex &v1 = g.vertices[g.vtx_indices[tri * 3 + 1]];
    const Vertex &v2_ = g.vertices[g.vtx_indices[tri * 3 + 2]];
    const float fw = float(g.w), fh = float(g.h);
    a = v2{v0.t[0] * fw, v0.t[1] * fh};
    b = v2{v1.t[0] * fw, v1.t[1] * fh};
    c = v2{v2_.t[0] * fw, v2_.t[1] * fh};
}

RT_DEV float edge_fn(v2 a, v2 b, v2 p) { return (b.x - a.x) * (p.y - a.y) - (b.y - a.y) * (p.x - a.x); }

// texel box [x0, x1] x [y0, y1] of a triangle's uv bounds clamped to the frame; false when the triangle can never win
// (degenerate, non-finite) or lies outside the frame
RT_DEV bool geo_box(const GeoTarget &g, uint32_t tri, int &x0, int &y0, int &x1, int &y1) {
    v2 a, b, c;
    geo_uv(g, tri, a, b, c);
    const float area2 = edge_fn(a, b, c);
    if (!(fabsf(area2) >= kGeoMinArea2) || !isfinite(area2)) {
        return false;
    }
    const float smin = fminf(a.x, fminf(b.x, c.x)), smax = fmaxf(a.x, fmaxf(b.x, c.x));
    const float tmin = fminf(a.y, fminf(b.y, c.y)), tmax = fmaxf(a.y, fmaxf(b.y, c.y));
    if (!(smax >= 0.0f && tmax >= 0.0f && smin < float(g.w) && tmin < float(g.h))) {
        return false;
    }
    x0 = int(fmaxf(floorf(smin), 0.0f));
    y0 = int(fmaxf(floorf(tmin), 0.0f));
    x1 = int(fminf(floorf(smax), float(g.w - 1)));
    y1 = int(fminf(floorf(tmax), float(g.h - 1)));
    return true;
}

__global__ void k_geo_box_total(GeoTarget g, unsigned long long *total) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long n = 0;
    int x0, y0, x1, y1;
    if (i < g.tri_count && geo_box(g, g.tri_first + i, x0, y0, x1, y1)) {
        n = (unsigned long long)(x1 - x0 + 1) * (unsigned long long)(y1 - y0 + 1);
    }
    for (int o = 16; o > 0; o >>= 1) {
        n += __shfl_down_sync(0xffffffffu, n, o);
    }
    if ((threadIdx.x & 31) == 0 && n != 0) {
        atomicAdd(total, n);
    }
}

// FILL = false: counts[texel]++ for every texel of the box; FILL = true: list[cursor[texel]++] = tri
template <bool FILL> __global__ void k_geo_walk(GeoTarget g, uint32_t *counts_or_cursor, uint32_t *list) {
    const uint32_t lane = threadIdx.x & 31, warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; warp < g.tri_count; warp += warps) {
        const uint32_t tri = g.tri_first + warp;
        int x0, y0, x1, y1;
        if (!geo_box(g, tri, x0, y0, x1, y1)) {
            continue;
        }
        const uint32_t bw = uint32_t(x1 - x0 + 1);
        const uint64_t n = uint64_t(bw) * uint32_t(y1 - y0 + 1);
        for (uint64_t k = lane; k < n; k += 32) {
            const uint32_t tx = uint32_t(x0) + uint32_t(k % bw), ty = uint32_t(y0) + uint32_t(k / bw);
            const size_t texel = size_t(ty) * uint32_t(g.w) + tx;
            const uint32_t slot = atomicAdd(&counts_or_cursor[texel], 1u);
            if (FILL) {
                list[slot] = tri;
            }
        }
    }
}

struct GeoParams {
    GeoTarget g;
    const uint32_t *offsets, *list;
    const MeshInstance *inst; // the baked instance
    uint32_t instance;
};

__global__ void __launch_bounds__(256) k_raygen_geo(KParams p, GeoParams gp, RayBuf rays, HitBuf hits) {
    // one warp = one 8x4 texel tile of the rect, like k_raygen
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
    const GeoTarget &g = gp.g;
    uint32_t best = 0xffffffffu;
    float bu = 0.0f, bv = 0.0f, barea2 = 0.0f;
    if (active) {
        const uint32_t px_hash = hash_u32((uint32_t(x) << 16) | uint32_t(y));
        const uint32_t rand_hash = hash_combine(px_hash, p.rand_seed);
        const v2 jit = rand2d(kRandDimFilter, rand_hash, p.iteration - 1, p.sc.rand_seq);
        const v2 pt = v2{float(x) + jit.x, float(y) + jit.y};
        const size_t texel = size_t(y) * uint32_t(p.fb.w) + uint32_t(x);
        for (uint32_t k = gp.offsets[texel], end = gp.offsets[texel + 1]; k < end; ++k) {
            const uint32_t tri = gp.list[k];
            if (tri >= best) {
                continue;
            }
            v2 a, b, c;
            geo_uv(g, tri, a, b, c);
            float area2 = edge_fn(a, b, c);
            float e0 = edge_fn(b, c, pt), e1 = edge_fn(c, a, pt), e2 = edge_fn(a, b, pt);
            if (area2 < 0.0f) {
                area2 = -area2;
                e0 = -e0;
                e1 = -e1;
                e2 = -e2;
            }
            if (e0 >= 0.0f && e1 >= 0.0f && e2 >= 0.0f) {
                best = tri;
                bu = e1;
                bv = e2;
                barea2 = area2;
            }
        }
        if (best == 0xffffffffu) {
            p.fb.temp[y * p.fb.w + x] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
    }
    const bool emit = best != 0xffffffffu;
    RayD r;
    Hit h;
    if (emit) {
        const float u = bu / barea2, v = bv / barea2, w = 1.0f - u - v;
        const Vertex &v0 = g.vertices[g.vtx_indices[best * 3 + 0]];
        const Vertex &v1 = g.vertices[g.vtx_indices[best * 3 + 1]];
        const Vertex &v2_ = g.vertices[g.vtx_indices[best * 3 + 2]];
        const float *xf = gp.inst->xform, *ixf = gp.inst->inv_xform;
        const v3 P = transform_point(mk3(v0.p) * w + mk3(v1.p) * u + mk3(v2_.p) * v, xf);
        const v3 N = safe_normalize(transform_normal(mk3(v0.n) * w + mk3(v1.n) * u + mk3(v2_.n) * v, ixf));
        const v3 W0 = transform_point(mk3(v0.p), xf), W1 = transform_point(mk3(v1.p), xf), W2 = transform_point(mk3(v2_.p), xf);
        r.o = P;
        r.d = -N;
        r.c = v3{1.0f, 1.0f, 1.0f};
        r.ior[0] = r.ior[1] = r.ior[2] = r.ior[3] = -1.0f;
        r.cone_width = sqrtf(length(cross(W1 - W0, W2 - W0)) / barea2); // both areas doubled
        r.cone_spread = 0.0f;
        r.pdf = 1e6f;
        r.xy = (uint32_t(x) << 16) | uint32_t(y);
        r.depth = (uint32_t(RAY_CAMERA) << 28);
        h.obj = int(gp.instance);
        h.prim = int(best);
        h.t = 0.0f;
        h.u = u;
        h.v = v;
    }
    const uint32_t slot = warp_append(&p.counters[CNT_RAYS + 0], emit);
    if (emit) {
        store_ray(rays, slot, r);
        store_hit(hits, slot, h);
    }
}

// ---- L1 SH ------------------------------------------------------------------------------------------------------
struct ShPlanes {
    float4 *coef[3];     // RC_BUF_SH_R / G / B: 4 coefficients of one channel
    float4 *e0, *direct; // per-sample scratch: temp after the primary shade, D
    float4 *dir0, *dir1; // per-sample scratch: shadow-ray / bounce-1 direction, tag in w
};

RT_DEV int rect_pixel(const KParams &p, int idx) {
    return (p.rect_y + idx / p.rect_w) * p.fb.w + (p.rect_x + idx % p.rect_w);
}

__global__ void k_sh_primary(KParams p, ShPlanes sh, RayBuf bounce1, uint32_t tag) {
    const int stride = gridDim.x * blockDim.x, i0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int idx = i0; idx < p.rect_w * p.rect_h; idx += stride) {
        const int pix = rect_pixel(p, idx);
        sh.e0[pix] = p.fb.temp[pix];
    }
    const uint32_t n = p.counters[CNT_RAYS + 1];
    for (uint32_t i = uint32_t(i0); i < n; i += uint32_t(stride)) {
        const uint32_t xy = bounce1.xy_depth[i].x;
        const float4 d = bounce1.d_cs[i];
        sh.dir1[int(xy & 0xffff) * p.fb.w + int(xy >> 16)] = make_float4(d.x, d.y, d.z, __uint_as_float(tag));
    }
}

__global__ void k_sh_direct(KParams p, ShPlanes sh, ShadowBuf shadow0, uint32_t tag) {
    const int stride = gridDim.x * blockDim.x, i0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int idx = i0; idx < p.rect_w * p.rect_h; idx += stride) {
        const int pix = rect_pixel(p, idx);
        const float4 t = p.fb.temp[pix], e = sh.e0[pix];
        sh.direct[pix] = make_float4(t.x - e.x, t.y - e.y, t.z - e.z, 0.0f);
    }
    const uint32_t n = p.counters[CNT_SHADOW + 0];
    for (uint32_t i = uint32_t(i0); i < n; i += uint32_t(stride)) {
        const uint32_t xy = __float_as_uint(shadow0.c_xy[i].w);
        const float4 d = shadow0.d_dist[i];
        sh.dir0[int(xy & 0xffff) * p.fb.w + int(xy >> 16)] = make_float4(d.x, d.y, d.z, __uint_as_float(tag));
    }
}

RT_DEV float4 sh_basis(float4 d, uint32_t tag) {
    if (__float_as_uint(d.w) != tag) {
        d.x = d.y = d.z = 0.0f;
    }
    return make_float4(0.282095f, 0.488603f * d.y, 0.488603f * d.z, 0.488603f * d.x);
}

__global__ void k_sh_resolve(KParams p, ShPlanes sh, uint32_t tag, float exposure_mul, float mix_factor) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p.rect_w * p.rect_h) {
        return;
    }
    const int pix = rect_pixel(p, idx);
    if (p.fb.required_samples[pix] < p.iteration) {
        return;
    }
    const float4 t = p.fb.temp[pix], e = sh.e0[pix], dd = sh.direct[pix];
    const float D[3] = {dd.x, dd.y, dd.z};
    const float I[3] = {t.x - (e.x + dd.x), t.y - (e.y + dd.y), t.z - (e.z + dd.z)};
    const float4 y0 = sh_basis(sh.dir0[pix], tag), y1 = sh_basis(sh.dir1[pix], tag);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const float4 nv = make_float4((D[ch] * y0.x + I[ch] * y1.x) * exposure_mul, (D[ch] * y0.y + I[ch] * y1.y) * exposure_mul,
                                      (D[ch] * y0.z + I[ch] * y1.z) * exposure_mul, (D[ch] * y0.w + I[ch] * y1.w) * exposure_mul);
        float4 o = sh.coef[ch][pix];
        o.x += (nv.x - o.x) * mix_factor;
        o.y += (nv.y - o.y) * mix_factor;
        o.z += (nv.z - o.z) * mix_factor;
        o.w += (nv.w - o.w) * mix_factor;
        sh.coef[ch][pix] = o;
    }
}

} // namespace rt
