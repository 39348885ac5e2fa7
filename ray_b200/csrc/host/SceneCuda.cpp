#include <stdio.h>
#include <stdlib.h>
// SceneCuda.cpp -- see SceneCuda.h.  Behavioural spec: reference internal/SceneCPU.cpp (file:line cited per function).
#include "SceneCuda.h"

#include <algorithm>
#include <array>
#include <atomic>
#include <cmath>
#include <cstring>

namespace RayB200 {
namespace Cuda {

namespace {
constexpr float PI = 3.141592653589793238463f;
constexpr float MAX_DIST = 3.402823466e+30F;

inline float clampf(float v, float lo, float hi) { return v < lo ? lo : (v > hi ? hi : v); }
inline uint16_t pack_unorm_16(float x) { return uint16_t(x * 65535.0f); } // reference Core.h:62
inline uint32_t f2u(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
}
inline float u2f(uint32_t u) {
    float f;
    memcpy(&f, &u, 4);
    return f;
}

// light_t bit-field word (reference Core.h:194-201)
inline uint32_t light_bits(int type, bool doublesided, bool cast_shadow, bool visible, bool sky_portal, uint32_t ray_vis) {
    return uint32_t(type & 7) | (uint32_t(doublesided) << 3) | (uint32_t(cast_shadow) << 4) | (uint32_t(visible) << 5) |
           (uint32_t(sky_portal) << 6) | ((ray_vis & 0xffu) << 7);
}
inline int l_type(const rt::Light &l) { return int(l.bits & 7u); }
inline bool l_doublesided(const rt::Light &l) { return (l.bits >> 3) & 1u; }
inline bool l_visible(const rt::Light &l) { return (l.bits >> 5) & 1u; }
inline uint32_t l_ray_vis(const rt::Light &l) { return (l.bits >> 7) & 0xffu; }

inline uint32_t common_ray_vis(const rs_light_common &c) {
    return (uint32_t(c.diffuse_visibility != 0) << rt::RAY_DIFFUSE) | (uint32_t(c.specular_visibility != 0) << rt::RAY_SPECULAR) |
           (uint32_t(c.refraction_visibility != 0) << rt::RAY_REFR);
}

inline void xform_dir(const float *m, const float v[3], float out[3]) {
    out[0] = m[0] * v[0] + m[4] * v[1] + m[8] * v[2];
    out[1] = m[1] * v[0] + m[5] * v[1] + m[9] * v[2];
    out[2] = m[2] * v[0] + m[6] * v[1] + m[10] * v[2];
}
inline void xform_point(const float *m, const float v[3], float out[3]) {
    out[0] = m[0] * v[0] + m[4] * v[1] + m[8] * v[2] + m[12];
    out[1] = m[1] * v[0] + m[5] * v[1] + m[9] * v[2] + m[13];
    out[2] = m[2] * v[0] + m[6] * v[1] + m[10] * v[2] + m[14];
}
inline void cross3(const float a[3], const float b[3], float out[3]) {
    out[0] = a[1] * b[2] - a[2] * b[1];
    out[1] = a[2] * b[0] - a[0] * b[2];
    out[2] = a[0] * b[1] - a[1] * b[0];
}
inline float dot3(const float a[3], const float b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
inline float len3(const float a[3]) { return sqrtf(dot3(a, a)); }

// Plane-form triangle data, formulas of Ray::PreprocessTri (reference internal/Core.cpp:212-258): same operations in
// the same order (this TU is built with -ffp-contract=off), so an identical triangle yields identical planes and the
// kernels report the same (t,u,v) for it as on reference-built data.
bool make_tri_planes(const float p0[3], const float p1[3], const float p2[3], float n_plane[4], float u_plane[4],
                     float v_plane[4]) {
    const float e0[3] = {p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2]}, e1[3] = {p2[0] - p0[0], p2[1] - p0[1], p2[2] - p0[2]};
    float n[3] = {e0[1] * e1[2] - e0[2] * e1[1], e0[2] * e1[0] - e0[0] * e1[2], e0[0] * e1[1] - e0[1] * e1[0]};
    const float n_len_sqr = n[0] * n[0] + n[1] * n[1] + n[2] * n[2];
    if (n_len_sqr == 0.0f) {
        return false; // degenerate
    }
    const float u[3] = {(e1[1] * n[2] - e1[2] * n[1]) / n_len_sqr, (e1[2] * n[0] - e1[0] * n[2]) / n_len_sqr,
                        (e1[0] * n[1] - e1[1] * n[0]) / n_len_sqr};
    u_plane[0] = u[0];
    u_plane[1] = u[1];
    u_plane[2] = u[2];
    u_plane[3] = -(u[0] * p0[0] + u[1] * p0[1] + u[2] * p0[2]);
    const float v[3] = {(n[1] * e0[2] - n[2] * e0[1]) / n_len_sqr, (n[2] * e0[0] - n[0] * e0[2]) / n_len_sqr,
                        (n[0] * e0[1] - n[1] * e0[0]) / n_len_sqr};
    v_plane[0] = v[0];
    v_plane[1] = v[1];
    v_plane[2] = v[2];
    v_plane[3] = -(v[0] * p0[0] + v[1] * p0[1] + v[2] * p0[2]);
    const float l = sqrtf(n_len_sqr);
    n[0] /= l;
    n[1] /= l;
    n[2] /= l;
    n_plane[0] = n[0];
    n_plane[1] = n[1];
    n_plane[2] = n[2];
    n_plane[3] = n[0] * p0[0] + n[1] * p0[1] + n[2] * p0[2];
    return true;
}

// TransformBoundingBox (reference internal/Core.cpp:1368-1388)
void transform_box(const Aabb &b, const float *xform, Aabb &out) {
    for (int j = 0; j < 3; ++j) {
        out.mn[j] = out.mx[j] = xform[12 + j];
    }
    for (int j = 0; j < 3; ++j) {
        for (int i = 0; i < 3; ++i) {
            const float a = xform[i * 4 + j] * b.mn[i];
            const float c = xform[i * 4 + j] * b.mx[i];
            if (a < c) {
                out.mn[j] += a;
                out.mx[j] += c;
            } else {
                out.mn[j] += c;
                out.mx[j] += a;
            }
        }
    }
}

uint16_t encode_snorm_u16(float f) { return uint16_t(std::round(clampf((f + 1) / 2.0f, 0.0f, 1.0f) * 65535.0f)); }

// octahedral direction code decoded by the kernels' decode_oct_dir (rt_lights.cuh); reference Core.cpp:145-156
uint32_t encode_oct_dir(const float d[3]) {
    const float denom = fabsf(d[0]) + fabsf(d[1]) + fabsf(d[2]);
    const float v[3] = {d[0] / denom, d[1] / denom, d[2] / denom};
    if (v[2] < 0.0f) {
        const uint16_t x = encode_snorm_u16((1.0f - fabsf(v[1])) * copysignf(1.0f, v[0]));
        const uint16_t y = encode_snorm_u16((1.0f - fabsf(v[0])) * copysignf(1.0f, v[1]));
        return (uint32_t(x) << 16) | y;
    }
    return (uint32_t(encode_snorm_u16(v[0])) << 16) | encode_snorm_u16(v[1]);
}

uint32_t encode_cosines(float cos_a, float cos_b) { // reference Core.cpp:95-100
    const uint32_t a = uint32_t(std::floor(65534.0f * ((cos_a + 1.0f) / 2.0f)));
    const uint32_t b = uint32_t(std::floor(65534.0f * ((cos_b + 1.0f) / 2.0f)));
    return (a << 16) | b;
}

float quantize(float v, float mn, float mx) {
    if (mn == mx) {
        return 0.0f;
    }
    return clampf(255.0f * (v - mn) / (mx - mn), 0.0f, 255.0f);
}

struct LightNode {
    Aabb box;
    bool infinite = false;
    float flux = 0.0f, axis[3] = {0, 0, 0}, omega_n = 0.0f, omega_e = 0.0f;
    uint32_t left = 0, right = 0;
    bool leaf = false;
    uint32_t light_index = 0;
};

} // namespace

void InverseMatrix4(const float m[16], float out[16]) {
    // Gauss-Jordan in double; the reference uses a closed-form float cofactor expansion (Core.cpp:1390-1431)
    double a[4][8];
    for (int r = 0; r < 4; ++r) {
        for (int c = 0; c < 4; ++c) {
            a[r][c] = m[c * 4 + r]; // column-major input
            a[r][4 + c] = (r == c) ? 1.0 : 0.0;
        }
    }
    for (int col = 0; col < 4; ++col) {
        int piv = col;
        for (int r = col + 1; r < 4; ++r) {
            if (std::fabs(a[r][col]) > std::fabs(a[piv][col])) {
                piv = r;
            }
        }
        if (piv != col) {
            for (int c = 0; c < 8; ++c) {
                std::swap(a[piv][c], a[col][c]);
            }
        }
        const double d = a[col][col];
        if (d == 0.0) {
            continue; // singular: leave garbage-free but meaningless
        }
        for (int c = 0; c < 8; ++c) {
            a[col][c] /= d;
        }
        for (int r = 0; r < 4; ++r) {
            if (r != col) {
                const double f = a[r][col];
                for (int c = 0; c < 8; ++c) {
                    a[r][c] -= f * a[col][c];
                }
            }
        }
    }
    for (int r = 0; r < 4; ++r) {
        for (int c = 0; c < 4; ++c) {
            out[c * 4 + r] = float(a[r][4 + c]);
        }
    }
}

Scene::Scene(ILog *log, rc_ctx *build_ctx) {
    log_ = log;
    build_ctx_ = build_ctx;
    SetEnvironment(environment_desc_t{{0, 0, 0}, {0, 0, 0}, 1, RS_INVALID, RS_INVALID, 0.0f, 0.0f});
}
Scene::~Scene() {
    for (PinnedMirror &m : pinned_) {
        rc_host_free(m.ptr);
    }
}

// the rc_texture table FillView hands out; rebuilt under the unique lock (AddTexture / Finalize) so concurrent
// renderers preparing the same scene under the shared lock only read it
void Scene::RebuildTexViews_nolock() {
    tex_views_.clear();
    for (const TexImage &img : textures_) {
        rc_texture t = {};
        t.handle = img.handle;
        t.channels = img.channels;
        for (int lod = 0; lod < RC_TEX_MIP_LEVELS; ++lod) { // no mips: every level aliases level 0
            t.res[lod][0] = uint16_t(img.w);
            t.res[lod][1] = uint16_t(img.h);
            t.pixels[lod] = img.pixels.data();
        }
        tex_views_.push_back(t);
    }
}

void Scene::RefreshPinnedMirrors_nolock() {
    if (getenv("RAY_HOST_NO_PINNED")) { // A/B switch for measurements
        pinned_revision_ = 0;
        return;
    }
    const void *src[PM_COUNT] = {wnodes_.data(),      mtris_.data(),       vertices_.data(),
                                 vtx_indices_.data(), tri_indices_.data(), tri_materials_.data()};
    const size_t bytes[PM_COUNT] = {wnodes_.size() * sizeof(rt::WNode),   mtris_.size() * sizeof(rt::MTri),
                                    vertices_.size() * sizeof(rt::Vertex), vtx_indices_.size() * 4,
                                    tri_indices_.size() * 4,               tri_materials_.size() * sizeof(rt::TriMat)};
    bool ok = true;
    for (int i = 0; i < PM_COUNT; ++i) {
        PinnedMirror &m = pinned_[i];
        if (bytes[i] > m.capacity) {
            rc_host_free(m.ptr);
            m.capacity = bytes[i] + bytes[i] / 8;
            m.ptr = rc_host_alloc(m.capacity); // nullptr without a CUDA device: FillView then hands over the vectors
            if (!m.ptr) {
                m.capacity = 0;
            }
        }
        m.bytes = 0;
        if (m.ptr && bytes[i] != 0) {
            memcpy(m.ptr, src[i], bytes[i]);
            m.bytes = bytes[i];
        } else if (bytes[i] != 0) {
            ok = false;
        }
    }
    pinned_revision_ = ok ? revision_ : 0;
}

void Scene::GetEnvironment(environment_desc_t &env) {
    std::shared_lock<std::shared_timed_mutex> lock(mtx_);
    env = env_;
}
void Scene::SetEnvironment(const environment_desc_t &env) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    structure_dirty_ = true;
    env_ = env;
}

// reference SceneCPU.cpp:61-205 with texture compression off: RGBA -> storage 0, RGB -> 1, RG and every normal map -> 2
// (x, y kept, y inverted for the DX convention, z reconstructed when the map's z is not a constant 1), R -> 3.
// The uncompressed storages never build mips (TextureStorageCPU.cpp:232), so generate_mipmaps is accepted and ignored.
TextureHandle Scene::AddTexture(const tex_desc_t &t) {
    if (!t.data || t.w <= 0 || t.h <= 0 || t.w > 65535 || t.h > 65535) {
        log_->Error("Ray(CUDA): AddTexture: bad texture description");
        return TextureHandle{};
    }
    const size_t n = size_t(t.w) * t.h;
    bool reconstruct_z = t.reconstruct_z != 0;
    const bool invert_y = (t.convention == 1);
    TexImage img;
    img.w = t.w;
    img.h = t.h;
    int storage = -1;
    if (t.format == RS_TEX_RGBA8888 || t.format == RS_TEX_RGB888) {
        const int c = (t.format == RS_TEX_RGBA8888) ? 4 : 3;
        if (!t.is_normalmap) {
            storage = (c == 4) ? 0 : 1;
            img.channels = uint32_t(c);
            img.pixels.assign(t.data, t.data + n * c);
        } else {
            storage = 2;
            img.channels = 2;
            img.pixels.resize(n * 2);
            for (size_t i = 0; i < n; ++i) {
                img.pixels[i * 2 + 0] = t.data[i * c + 0];
                img.pixels[i * 2 + 1] = invert_y ? uint8_t(255 - t.data[i * c + 1]) : t.data[i * c + 1];
                reconstruct_z |= (t.data[i * c + 2] < 250);
            }
        }
    } else if (t.format == RS_TEX_RG88) {
        storage = 2;
        img.channels = 2;
        img.pixels.assign(t.data, t.data + n * 2);
        if (t.is_normalmap && invert_y) {
            for (size_t i = 0; i < n; ++i) {
                img.pixels[i * 2 + 1] = uint8_t(255 - img.pixels[i * 2 + 1]);
            }
        }
        reconstruct_z = t.is_normalmap != 0;
    } else if (t.format == RS_TEX_R8) {
        storage = 3;
        img.channels = 1;
        img.pixels.assign(t.data, t.data + n);
    } else {
        log_->Error("Ray(CUDA): AddTexture: format %u is not supported (uncompressed RGBA/RGB/RG/R only)", t.format);
        return TextureHandle{};
    }
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    structure_dirty_ = true;
    const uint32_t index = tex_storage_counts_[storage]++;
    img.handle = (uint32_t(storage) << 28) | index;
    uint32_t ret = img.handle;
    if (t.is_srgb) {
        ret |= rt::kTexSrgbBitHost;
    }
    if (reconstruct_z) {
        ret |= rt::kTexReconstructZBitHost;
    }
    textures_.push_back(std::move(img));
    RebuildTexViews_nolock();
    revision_ = NextRevision();
    return TextureHandle{ret, 0};
}

// reference SceneCPU.cpp:208-250
MaterialHandle Scene::AddMaterial_nolock(const shading_node_desc_t &m) {
    rt::Material mat;
    memset(&mat, 0, sizeof(mat));
    mat.type = m.type;
    mat.textures[rt::kTexBase] = m.base_texture;
    mat.roughness_unorm = pack_unorm_16(clampf(m.roughness, 0.0f, 1.0f));
    mat.textures[rt::kTexRough] = m.roughness_texture;
    memcpy(mat.base_color, m.base_color, 3 * sizeof(float));
    mat.ior = m.ior;
    mat.tangent_rotation_or_strength = 0.0f;
    mat.flags = 0;
    if (m.type == rt::NODE_DIFFUSE) {
        mat.sheen_unorm = pack_unorm_16(clampf(0.5f * m.sheen, 0.0f, 1.0f));
        mat.sheen_tint_unorm = pack_unorm_16(clampf(m.tint, 0.0f, 1.0f));
        mat.textures[rt::kTexMetallic] = m.metallic_texture;
    } else if (m.type == rt::NODE_GLOSSY) {
        mat.tangent_rotation_or_strength = 2.0f * PI * m.anisotropic_rotation;
        mat.textures[rt::kTexMetallic] = m.metallic_texture;
        mat.tint_unorm = pack_unorm_16(clampf(m.tint, 0.0f, 1.0f));
    } else if (m.type == rt::NODE_EMISSIVE) {
        mat.tangent_rotation_or_strength = m.strength;
        if (m.importance_sample) {
            mat.flags |= rt::kMatFlagImpSample;
        }
    } else if (m.type == rt::NODE_MIX) {
        mat.tangent_rotation_or_strength = m.strength;
        mat.textures[rt::kMixMat1] = m.mix_materials[0];
        mat.textures[rt::kMixMat2] = m.mix_materials[1];
        if (m.mix_add) {
            mat.flags |= rt::kMatFlagMixAdd;
        }
    }
    mat.textures[rt::kTexNormals] = m.normal_map;
    mat.normal_map_strength_unorm = pack_unorm_16(clampf(m.normal_map_intensity, 0.0f, 1.0f));
    materials_.push_back(mat);
    return MaterialHandle{uint32_t(materials_.size() - 1), 0};
}

MaterialHandle Scene::AddMaterial(const shading_node_desc_t &m) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    structure_dirty_ = true;
    return AddMaterial_nolock(m);
}

// reference SceneCPU.cpp:252-340: principled root (+ emissive via additive mix, + transparent via alpha mix)
MaterialHandle Scene::AddMaterial(const principled_mat_desc_t &m) {
    rt::Material mm;
    memset(&mm, 0, sizeof(mm));
    mm.type = rt::NODE_PRINCIPLED;
    mm.textures[rt::kTexBase] = m.base_texture;
    mm.textures[rt::kTexRough] = m.roughness_texture;
    mm.textures[rt::kTexMetallic] = m.metallic_texture;
    mm.textures[rt::kTexNormals] = m.normal_map;
    mm.textures[rt::kTexSpecular] = m.specular_texture;
    memcpy(mm.base_color, m.base_color, 3 * sizeof(float));
    mm.sheen_unorm = pack_unorm_16(clampf(0.5f * m.sheen, 0.0f, 1.0f));
    mm.sheen_tint_unorm = pack_unorm_16(clampf(m.sheen_tint, 0.0f, 1.0f));
    mm.roughness_unorm = pack_unorm_16(clampf(m.roughness, 0.0f, 1.0f));
    mm.tangent_rotation_or_strength = 2.0f * PI * clampf(m.anisotropic_rotation, 0.0f, 1.0f);
    mm.metallic_unorm = pack_unorm_16(clampf(m.metallic, 0.0f, 1.0f));
    mm.ior = m.ior;
    mm.flags = 0;
    mm.transmission_unorm = pack_unorm_16(clampf(m.transmission, 0.0f, 1.0f));
    mm.transmission_roughness_unorm = pack_unorm_16(clampf(m.transmission_roughness, 0.0f, 1.0f));
    mm.normal_map_strength_unorm = pack_unorm_16(clampf(m.normal_map_intensity, 0.0f, 1.0f));
    mm.anisotropic_unorm = pack_unorm_16(clampf(m.anisotropic, 0.0f, 1.0f));
    mm.specular_unorm = pack_unorm_16(clampf(m.specular, 0.0f, 1.0f));
    mm.specular_tint_unorm = pack_unorm_16(clampf(m.specular_tint, 0.0f, 1.0f));
    mm.clearcoat_unorm = pack_unorm_16(clampf(m.clearcoat, 0.0f, 1.0f));
    mm.clearcoat_roughness_unorm = pack_unorm_16(clampf(m.clearcoat_roughness, 0.0f, 1.0f));

    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    structure_dirty_ = true;
    materials_.push_back(mm);
    MaterialHandle root{uint32_t(materials_.size() - 1), 0};
    MaterialHandle emissive, transparent;

    if (m.emission_strength > 0.0f && (m.emission_color[0] > 0.0f || m.emission_color[1] > 0.0f || m.emission_color[2] > 0.0f)) {
        shading_node_desc_t e;
        rs_shading_node_defaults(&e);
        e.type = rt::NODE_EMISSIVE;
        memcpy(e.base_color, m.emission_color, 3 * sizeof(float));
        e.base_texture = m.emission_texture;
        e.strength = m.emission_strength;
        e.importance_sample = m.importance_sample;
        emissive = AddMaterial_nolock(e);
    }
    if (m.alpha != 1.0f || m.alpha_texture != RS_INVALID) {
        shading_node_desc_t t;
        rs_shading_node_defaults(&t);
        t.type = rt::NODE_TRANSPARENT;
        transparent = AddMaterial_nolock(t);
    }
    if (emissive._index != 0xffffffffu) {
        shading_node_desc_t mix;
        rs_shading_node_defaults(&mix);
        mix.type = rt::NODE_MIX;
        mix.strength = 0.5f;
        mix.ior = 0.0f;
        mix.mix_add = 1;
        mix.mix_materials[0] = root._index;
        mix.mix_materials[1] = emissive._index;
        root = AddMaterial_nolock(mix);
    }
    if (transparent._index != 0xffffffffu) {
        if (m.alpha == 0.0f) {
            root = transparent;
        } else {
            shading_node_desc_t mix;
            rs_shading_node_defaults(&mix);
            mix.type = rt::NODE_MIX;
            mix.base_texture = m.alpha_texture;
            mix.strength = m.alpha;
            mix.ior = 0.0f;
            mix.mix_materials[0] = transparent._index;
            mix.mix_materials[1] = root._index;
            root = AddMaterial_nolock(mix);
        }
    }
    return root;
}

uint64_t Scene::NextRevision() {
    static std::atomic<uint64_t> counter{1};
    return counter.fetch_add(1);
}

// Tangent frame of a mesh that came without binormals: per triangle the uv-aligned tangent / binormal, accumulated at
// the vertices; a vertex whose triangles disagree on the orientation of either is duplicated (up to three twins), the
// triangle re-pointed to the twin.  Finally b = normalize(cross(n, accumulated tangent)).
// Reference: Ray::ComputeTangentBasis, internal/TextureUtils.cpp:1603-1739 (same arithmetic, restated over plain arrays).
static void ComputeTangentBasis(std::vector<rt::Vertex> &verts, std::vector<uint32_t> &idx) {
    const float FLT_EPS_ = 0.0000001f;
    const size_t n0 = verts.size();
    std::vector<std::array<uint32_t, 3>> twins(n0, std::array<uint32_t, 3>{0, 0, 0});
    std::vector<std::array<float, 3>> bin(n0, std::array<float, 3>{0.0f, 0.0f, 0.0f});
    auto dot = [](const float a[3], const float b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; };
    for (size_t i = 0; i + 2 < idx.size(); i += 3) {
        const uint32_t id[3] = {idx[i], idx[i + 1], idx[i + 2]};
        float dp1[3], dp2[3];
        for (int a = 0; a < 3; ++a) {
            dp1[a] = verts[id[1]].p[a] - verts[id[0]].p[a];
            dp2[a] = verts[id[2]].p[a] - verts[id[0]].p[a];
        }
        const float dt1[2] = {verts[id[1]].t[0] - verts[id[0]].t[0], verts[id[1]].t[1] - verts[id[0]].t[1]};
        const float dt2[2] = {verts[id[2]].t[0] - verts[id[0]].t[0], verts[id[2]].t[1] - verts[id[0]].t[1]};
        float tangent[3], binormal[3];
        const float det = fabsf(dt1[0] * dt2[1] - dt1[1] * dt2[0]);
        if (det > FLT_EPS_) {
            const float inv_det = 1.0f / det;
            for (int a = 0; a < 3; ++a) {
                tangent[a] = (dp1[a] * dt2[1] - dp2[a] * dt1[1]) * inv_det;
                binormal[a] = (dp2[a] * dt1[0] - dp1[a] * dt2[0]) * inv_det;
            }
        } else {
            float plane_n[3];
            cross3(dp1, dp2, plane_n);
            int w = 2;
            tangent[0] = 0.0f, tangent[1] = 1.0f, tangent[2] = 0.0f;
            if (fabsf(plane_n[0]) <= fabsf(plane_n[1]) && fabsf(plane_n[0]) <= fabsf(plane_n[2])) {
                tangent[0] = 1.0f, tangent[1] = 0.0f, tangent[2] = 0.0f;
                w = 1;
            } else if (fabsf(plane_n[2]) <= fabsf(plane_n[0]) && fabsf(plane_n[2]) <= fabsf(plane_n[1])) {
                tangent[0] = 0.0f, tangent[1] = 0.0f, tangent[2] = 1.0f;
                w = 0;
            }
            if (fabsf(plane_n[w]) > FLT_EPS_) {
                cross3(plane_n, tangent, binormal);
                float l = len3(binormal);
                for (int a = 0; a < 3; ++a) {
                    binormal[a] /= l;
                }
                cross3(plane_n, binormal, tangent);
                l = len3(tangent);
                for (int a = 0; a < 3; ++a) {
                    tangent[a] /= l;
                }
            } else {
                for (int a = 0; a < 3; ++a) {
                    binormal[a] = tangent[a] = 0.0f;
                }
            }
        }
        for (int c = 0; c < 3; ++c) {
            const uint32_t vi = id[c];
            const int i1 = dot(verts[vi].b, tangent) < 0.0f ? 1 : 0;
            const int i2 = dot(bin[vi].data(), binormal) < 0.0f ? 2 : 0;
            uint32_t target = vi;
            if (i1 || i2) {
                uint32_t &twin = twins[vi][i1 + i2 - 1];
                if (twin == 0) {
                    twin = uint32_t(verts.size());
                    rt::Vertex copy = verts[vi];
                    copy.b[0] = copy.b[1] = copy.b[2] = 0.0f;
                    verts.push_back(copy);
                }
                target = twin;
                idx[i + c] = target;
            } else {
                bin[vi] = {binormal[0], binormal[1], binormal[2]};
            }
            for (int a = 0; a < 3; ++a) {
                verts[target].b[a] += tangent[a];
            }
        }
    }
    for (rt::Vertex &v : verts) {
        if (fabsf(v.b[0]) > FLT_EPS_ || fabsf(v.b[1]) > FLT_EPS_ || fabsf(v.b[2]) > FLT_EPS_) {
            float b[3];
            cross3(v.n, v.b, b);
            const float l = len3(b);
            if (l > FLT_EPS_) {
                v.b[0] = b[0] / l, v.b[1] = b[1] / l, v.b[2] = b[2] / l;
            }
        }
    }
}

// reference SceneCPU.cpp:342-546 + Core.cpp:260-328
MeshHandle Scene::AddMesh(const mesh_desc_t &m) {
    const rs_vtx_attribute &P = m.vtx_positions;
    if (!P.data || P.stride <= 0 || !m.vtx_indices || m.vtx_indices_count % 3 != 0 || m.vtx_indices_count == 0) {
        log_->Error("Ray(CUDA): AddMesh: bad mesh description");
        return MeshHandle{};
    }
    const uint32_t n_verts = uint32_t(P.count / uint64_t(P.stride));
    const uint32_t n_tris = uint32_t(m.vtx_indices_count / 3);

    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    structure_dirty_ = true;
    if (tlas_root_ != 0xffffffffu) { // drop the TLAS appended by a previous Finalize
        wnodes_.resize(blas_nodes_end_);
        tlas_root_ = 0xffffffffu;
    }
    const uint32_t vtx_base = uint32_t(vertices_.size());
    const uint32_t tri_base = uint32_t(tri_materials_.size());

    // vertices; without explicit binormals the tangent frame is derived from the uv mapping, which may split vertices
    // whose triangles disagree on handedness (reference SceneCPU.cpp:503-526, ComputeTangentBasis TextureUtils.cpp:1603)
    std::vector<rt::Vertex> nv(n_verts);
    for (uint32_t i = 0; i < n_verts; ++i) {
        rt::Vertex &v = nv[i];
        memset(&v, 0, sizeof(v));
        memcpy(v.p, &P.data[P.offset + size_t(i) * P.stride], 3 * sizeof(float));
        if (m.vtx_normals.data) {
            memcpy(v.n, &m.vtx_normals.data[m.vtx_normals.offset + size_t(i) * m.vtx_normals.stride], 3 * sizeof(float));
        } else {
            v.n[0] = 0.0f, v.n[1] = 1.0f, v.n[2] = 0.0f;
        }
        if (m.vtx_uvs.data) {
            memcpy(v.t, &m.vtx_uvs.data[m.vtx_uvs.offset + size_t(i) * m.vtx_uvs.stride], 2 * sizeof(float));
        }
        if (m.vtx_binormals.data) {
            memcpy(v.b, &m.vtx_binormals.data[m.vtx_binormals.offset + size_t(i) * m.vtx_binormals.stride], 3 * sizeof(float));
        }
    }
    std::vector<uint32_t> ni(m.vtx_indices_count);
    for (uint64_t i = 0; i < m.vtx_indices_count; ++i) {
        ni[i] = m.vtx_indices[i] + uint32_t(m.base_vertex);
        if (ni[i] >= n_verts) {
            log_->Error("Ray(CUDA): AddMesh: vertex index %u out of range (%u vertices)", ni[i], n_verts);
            return MeshHandle{};
        }
    }
    if (!m.vtx_binormals.data) {
        ComputeTangentBasis(nv, ni);
    }
    vertices_.insert(vertices_.end(), nv.begin(), nv.end());
    vtx_indices_.resize(size_t(tri_base) * 3 + m.vtx_indices_count);
    for (uint64_t i = 0; i < m.vtx_indices_count; ++i) {
        vtx_indices_[size_t(tri_base) * 3 + i] = vtx_base + ni[i];
    }
    tri_materials_.resize(tri_base + n_tris, rt::TriMat{0xffff, 0xffff});

    // plane-form triangles + primitive boxes
    struct TriRec {
        float n[4], u[4], v[4];
        uint32_t tri; // local triangle index
    };
    std::vector<TriRec> tris;
    std::vector<Aabb> boxes;
    tris.reserve(n_tris);
    boxes.reserve(n_tris);
    for (uint32_t t = 0; t < n_tris; ++t) {
        const float *p0 = vertices_[vtx_indices_[size_t(tri_base + t) * 3 + 0]].p;
        const float *p1 = vertices_[vtx_indices_[size_t(tri_base + t) * 3 + 1]].p;
        const float *p2 = vertices_[vtx_indices_[size_t(tri_base + t) * 3 + 2]].p;
        TriRec r;
        if (!make_tri_planes(p0, p1, p2, r.n, r.u, r.v)) {
            continue;
        }
        r.tri = t;
        tris.push_back(r);
        Aabb b;
        b.reset();
        b.grow(p0);
        b.grow(p1);
        b.grow(p2);
        boxes.push_back(b);
    }
    if (tris.empty()) {
        log_->Error("Ray(CUDA): AddMesh: mesh has no non-degenerate triangles");
        return MeshHandle{};
    }

    // binary SAH tree down to single triangles, then the SAH-optimal 8-wide collapse (BvhBuilder.h); RAY_HOST_BVH=greedy
    // keeps the earlier build (binary leaves of <= 8 triangles, widest-area-first collapse) for A/B measurements
    static const bool greedy = getenv("RAY_HOST_BVH") && !strcmp(getenv("RAY_HOST_BVH"), "greedy");
    std::vector<BinaryNode> bnodes;
    std::vector<uint32_t> order;
    bool built = false;
    if (m.use_fast_bvh_build && !greedy && build_ctx_ && boxes.size() >= 2) {
        // fast build (reference: PreprocessPrims_HLBVH, Core.cpp:574-720): Morton-order radix tree built on the device
        built = BuildBinaryLBVH(build_ctx_, boxes, bnodes, order);
        if (!built) {
            log_->Error("Ray(CUDA): AddMesh: device BVH build failed: %s", rc_last_error(build_ctx_));
            return MeshHandle{};
        }
    }
    if (!built) {
        BuildBinaryBVH(boxes, greedy ? 8 : 1, bnodes, order);
    }

    // every leaf owns one 8-triangle block; lanes past the leaf's count repeat its last triangle (Core.cpp:533-535)
    std::vector<rt::WNode> wide;
    wide.reserve(bnodes.size() / 4 + 8);
    const uint32_t node_base = uint32_t(wnodes_.size());
    auto leaf_range = [&](uint32_t first, uint32_t count) -> uint32_t {
        const uint32_t slot0 = uint32_t(tri_indices_.size());
        mtris_.emplace_back();
        rt::MTri &blk = mtris_.back();
        for (uint32_t k = 0; k < 8; ++k) {
            const uint32_t src = order[first + std::min(k, count - 1)];
            const TriRec &r = tris[src];
            tri_indices_.push_back(tri_base + r.tri);
            for (int c = 0; c < 4; ++c) {
                blk.n_plane[c][k] = r.n[c];
                blk.u_plane[c][k] = r.u[c];
                blk.v_plane[c][k] = r.v[c];
            }
        }
        return slot0;
    };
    auto leaf_payload = [&](const BinaryNode &leaf) -> uint32_t { return leaf_range(leaf.first, leaf.count); };
    float c_node = 1.0f, c_leaf = 1.6f;
    if (const char *e = getenv("RAY_HOST_BVH_COST")) {
        sscanf(e, "%f,%f", &c_node, &c_leaf);
    }
    const uint32_t root = greedy ? CollapseToWide(bnodes, 0, wide, node_base, leaf_payload)
                                 : CollapseToWideSAH(bnodes, wide, node_base, c_node, c_leaf, leaf_range);
    (void)root;
    wnodes_.insert(wnodes_.end(), wide.begin(), wide.end());
    blas_nodes_end_ = uint32_t(wnodes_.size());

    // triangle materials: SOLID bit = no Transparent node reachable through the mix graph (SceneCPU.cpp:444-500)
    auto is_solid = [&](uint32_t root_mat) {
        uint32_t stack[64];
        int sp = 0;
        stack[sp++] = root_mat;
        while (sp) {
            const rt::Material &mat = materials_[stack[--sp]];
            if (mat.type == rt::NODE_MIX) {
                if (sp + 2 <= 64) {
                    stack[sp++] = mat.textures[rt::kMixMat1];
                    stack[sp++] = mat.textures[rt::kMixMat2];
                }
            } else if (mat.type == rt::NODE_TRANSPARENT) {
                return false;
            }
        }
        return true;
    };
    for (uint32_t g = 0; g < m.groups_count; ++g) {
        const rs_mat_group_desc &grp = m.groups[g];
        if (grp.front_mat >= materials_.size() || (grp.back_mat != RS_INVALID && grp.back_mat >= materials_.size())) {
            log_->Error("Ray(CUDA): AddMesh: group %u references an unknown material", g);
            continue;
        }
        const bool front_solid = is_solid(grp.front_mat);
        const bool back_solid = (grp.back_mat == RS_INVALID) ? true : (grp.back_mat == grp.front_mat ? front_solid : is_solid(grp.back_mat));
        for (uint64_t i = grp.vtx_start; i < grp.vtx_start + grp.vtx_count; i += 3) {
            if (i / 3 >= n_tris) {
                break;
            }
            rt::TriMat &tm = tri_materials_[tri_base + uint32_t(i / 3)];
            tm.front_mi = uint16_t(grp.front_mat) | (front_solid ? uint16_t(rt::kMatSolidBit) : uint16_t(0));
            if (grp.back_mat != RS_INVALID) {
                tm.back_mi = uint16_t(grp.back_mat) | (back_solid ? uint16_t(rt::kMatSolidBit) : uint16_t(0));
            }
        }
    }

    MeshRec rec;
    rec.box = bnodes[0].box;
    rec.node_index = root;
    rec.tri_first = tri_base;
    rec.tri_count = n_tris;
    rec.alive = true;
    meshes_.push_back(rec);
    return MeshHandle{uint32_t(meshes_.size() - 1), 0};
}

void Scene::RemoveMesh(MeshHandle m) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    structure_dirty_ = true;
    if (m._index < meshes_.size()) {
        meshes_[m._index].alive = false;
        for (size_t i = 0; i < mesh_instances_.size(); ++i) {
            if (mesh_instances_[i].mesh_index == m._index) {
                RemoveMeshInstance_nolock(uint32_t(i));
            }
        }
    }
}

uint32_t Scene::AddLight_nolock(const rt::Light &l) {
    lights_.push_back(l);
    light_alive_.push_back(1);
    return uint32_t(lights_.size() - 1);
}

// reference SceneCPU.cpp:586-616
LightHandle Scene::AddLight(const directional_light_desc_t &d) {
    rt::Light l;
    memset(&l, 0, sizeof(l));
    l.bits = light_bits(rt::LIGHT_DIR, false, d.c.cast_shadow != 0, d.c.multiple_importance != 0, false, common_ray_vis(d.c));
    memcpy(l.col, d.c.color, 3 * sizeof(float));
    l.p[0] = -d.direction[0];
    l.p[1] = -d.direction[1];
    l.p[2] = -d.direction[2];
    const float angle = d.angle * PI / 360.0f;
    l.p[5] = angle;
    l.p[3] = cosf(angle);
    l.p[4] = tanf(angle);
    if (l.p[4] > 0.0f) {
        const float radius = l.p[4];
        const float mul = 1.0f / (PI * radius * radius);
        l.col[0] *= mul;
        l.col[1] *= mul;
        l.col[2] *= mul;
    }
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    return LightHandle{AddLight_nolock(l), 0};
}

// reference SceneCPU.cpp:618-640
LightHandle Scene::AddLight(const sphere_light_desc_t &d) {
    rt::Light l;
    memset(&l, 0, sizeof(l));
    l.bits = light_bits(rt::LIGHT_SPHERE, false, d.c.cast_shadow != 0, d.c.multiple_importance != 0 && (d.radius > 0.0f), false,
                        common_ray_vis(d.c));
    memcpy(l.col, d.c.color, 3 * sizeof(float));
    memcpy(&l.p[0], d.position, 3 * sizeof(float));
    l.p[3] = 4.0f * PI * d.radius * d.radius;
    l.p[7] = d.radius;
    l.p[8] = l.p[9] = -1.0f;
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    return LightHandle{AddLight_nolock(l), 0};
}

// reference SceneCPU.cpp:642-666
LightHandle Scene::AddLight(const spot_light_desc_t &d) {
    rt::Light l;
    memset(&l, 0, sizeof(l));
    l.bits = light_bits(rt::LIGHT_SPHERE, false, d.c.cast_shadow != 0, d.c.multiple_importance != 0 && (d.radius > 0.0f), false,
                        common_ray_vis(d.c));
    memcpy(l.col, d.c.color, 3 * sizeof(float));
    memcpy(&l.p[0], d.position, 3 * sizeof(float));
    memcpy(&l.p[4], d.direction, 3 * sizeof(float));
    l.p[3] = 4.0f * PI * d.radius * d.radius;
    l.p[7] = d.radius;
    l.p[8] = 0.5f * PI * d.spot_size / 180.0f;
    l.p[9] = d.spot_blend * d.spot_blend;
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    return LightHandle{AddLight_nolock(l), 0};
}

// reference SceneCPU.cpp:668-702
LightHandle Scene::AddLight(const rect_light_desc_t &d) {
    rt::Light l;
    memset(&l, 0, sizeof(l));
    uint32_t vis = common_ray_vis(d.c);
    if (d.sky_portal) {
        vis |= (1u << rt::RAY_SHADOW);
    }
    l.bits = light_bits(rt::LIGHT_RECT, d.doublesided != 0, d.c.cast_shadow != 0, d.c.multiple_importance != 0, d.sky_portal != 0, vis);
    memcpy(l.col, d.c.color, 3 * sizeof(float));
    l.p[0] = d.xform[12], l.p[1] = d.xform[13], l.p[2] = d.xform[14];
    l.p[3] = d.width * d.height;
    const float ex[3] = {1, 0, 0}, ez[3] = {0, 0, 1};
    float u[3], v[3];
    xform_dir(d.xform, ex, u);
    xform_dir(d.xform, ez, v);
    for (int i = 0; i < 3; ++i) {
        l.p[4 + i] = d.width * u[i];
        l.p[8 + i] = d.height * v[i];
    }
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    return LightHandle{AddLight_nolock(l), 0};
}

// reference SceneCPU.cpp:704-738
LightHandle Scene::AddLight(const disk_light_desc_t &d) {
    rt::Light l;
    memset(&l, 0, sizeof(l));
    uint32_t vis = common_ray_vis(d.c);
    if (d.sky_portal) {
        vis |= (1u << rt::RAY_SHADOW);
    }
    l.bits = light_bits(rt::LIGHT_DISK, d.doublesided != 0, d.c.cast_shadow != 0, d.c.multiple_importance != 0, d.sky_portal != 0, vis);
    memcpy(l.col, d.c.color, 3 * sizeof(float));
    l.p[0] = d.xform[12], l.p[1] = d.xform[13], l.p[2] = d.xform[14];
    l.p[3] = 0.25f * PI * d.size_x * d.size_y;
    const float ex[3] = {1, 0, 0}, ez[3] = {0, 0, 1};
    float u[3], v[3];
    xform_dir(d.xform, ex, u);
    xform_dir(d.xform, ez, v);
    for (int i = 0; i < 3; ++i) {
        l.p[4 + i] = d.size_x * u[i];
        l.p[8 + i] = d.size_y * v[i];
    }
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    return LightHandle{AddLight_nolock(l), 0};
}

// reference SceneCPU.cpp:740-768
LightHandle Scene::AddLight(const line_light_desc_t &d) {
    rt::Light l;
    memset(&l, 0, sizeof(l));
    l.bits = light_bits(rt::LIGHT_LINE, false, d.c.cast_shadow != 0, d.c.multiple_importance != 0, d.sky_portal != 0, common_ray_vis(d.c));
    memcpy(l.col, d.c.color, 3 * sizeof(float));
    l.p[0] = d.xform[12], l.p[1] = d.xform[13], l.p[2] = d.xform[14];
    l.p[3] = 2.0f * PI * d.radius * d.height;
    const float ex[3] = {1, 0, 0}, ey[3] = {0, 1, 0};
    float u[3], v[3];
    xform_dir(d.xform, ex, u);
    xform_dir(d.xform, ey, v);
    memcpy(&l.p[4], u, 3 * sizeof(float));
    l.p[7] = d.radius;
    memcpy(&l.p[8], v, 3 * sizeof(float));
    l.p[11] = d.height;
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    return LightHandle{AddLight_nolock(l), 0};
}

void Scene::RemoveLight(LightHandle l) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    if (l._index < light_alive_.size()) {
        light_alive_[l._index] = 0;
    }
}

// reference SceneCPU.cpp:770-863
MeshInstanceHandle Scene::AddMeshInstance(const mesh_instance_desc_t &d) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    structure_dirty_ = true;
    if (d.mesh >= meshes_.size() || !meshes_[d.mesh].alive) {
        log_->Error("Ray(CUDA): AddMeshInstance: unknown mesh %u", d.mesh);
        return MeshInstanceHandle{};
    }
    const MeshRec &m = meshes_[d.mesh];
    rt::MeshInstance mi;
    memset(&mi, 0, sizeof(mi));
    mi.mesh_index = d.mesh;
    mi.node_index = m.node_index;
    mi.lights_index = 0xffffffffu;
    mi.ray_visibility = (uint32_t(d.camera_visibility != 0) << rt::RAY_CAMERA) | (uint32_t(d.diffuse_visibility != 0) << rt::RAY_DIFFUSE) |
                        (uint32_t(d.specular_visibility != 0) << rt::RAY_SPECULAR) | (uint32_t(d.refraction_visibility != 0) << rt::RAY_REFR) |
                        (uint32_t(d.shadow_visibility != 0) << rt::RAY_SHADOW);
    memcpy(mi.xform, d.xform, 16 * sizeof(float));
    InverseMatrix4(mi.xform, mi.inv_xform);
    const uint32_t mi_index = uint32_t(mesh_instances_.size());

    // emissive triangles flagged for importance sampling become LIGHT_TYPE_TRI lights
    auto find_emissive = [&](uint16_t packed) -> uint32_t {
        if (packed == 0xffff) {
            return 0xffffffffu;
        }
        uint32_t q[64];
        int n = 0;
        q[n++] = packed & rt::kMatIndexBits;
        for (int i = 0; i < n; ++i) {
            const rt::Material &mat = materials_[q[i]];
            if (mat.type == rt::NODE_EMISSIVE && (mat.flags & rt::kMatFlagImpSample)) {
                return q[i];
            } else if (mat.type == rt::NODE_MIX && n + 2 <= 64) {
                q[n++] = mat.textures[rt::kMixMat1];
                q[n++] = mat.textures[rt::kMixMat2];
            }
        }
        return 0xffffffffu;
    };
    for (uint32_t tri = m.tri_first; tri < m.tri_first + m.tri_count; ++tri) {
        const rt::TriMat &tm = tri_materials_[tri];
        if (tm.front_mi == 0xffff) {
            continue;
        }
        const uint32_t fe = find_emissive(tm.front_mi), be = find_emissive(tm.back_mi);
        if (fe != 0xffffffffu) {
            const rt::Material &mat = materials_[fe];
            rt::Light l;
            memset(&l, 0, sizeof(l));
            uint32_t vis = mi.ray_visibility & 0xffu;
            vis &= ~(1u << rt::RAY_CAMERA);
            vis &= ~(1u << rt::RAY_SHADOW);
            l.bits = light_bits(rt::LIGHT_TRI, be != 0xffffffffu, true, false, false, vis);
            l.p[0] = u2f(tri);
            l.p[1] = u2f(mi_index);
            l.p[2] = u2f(mat.textures[rt::kTexBase]); // tri.tex_index (SceneCPU.cpp:840)
            l.col[0] = mat.base_color[0] * mat.tangent_rotation_or_strength;
            l.col[1] = mat.base_color[1] * mat.tangent_rotation_or_strength;
            l.col[2] = mat.base_color[2] * mat.tangent_rotation_or_strength;
            const uint32_t li = AddLight_nolock(l);
            if (mi.lights_index == 0xffffffffu) {
                mi.lights_index = li;
            }
        }
    }
    mesh_instances_.push_back(mi);
    instance_alive_.push_back(1);
    return MeshInstanceHandle{mi_index, 0};
}

void Scene::SetMeshInstanceTransform(MeshInstanceHandle h, const float *xform) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    if (h._index < mesh_instances_.size()) {
        memcpy(mesh_instances_[h._index].xform, xform, 16 * sizeof(float));
        InverseMatrix4(mesh_instances_[h._index].xform, mesh_instances_[h._index].inv_xform);
    }
}

// reference SceneCPU.cpp RemoveMeshInstance_nolock: the instance's emissive-triangle lights go with it
void Scene::RemoveMeshInstance_nolock(uint32_t index) {
    if (index < mesh_instances_.size()) {
        instance_alive_[index] = 0;
        for (size_t i = 0; i < lights_.size(); ++i) {
            if (l_type(lights_[i]) == rt::LIGHT_TRI && f2u(lights_[i].p[1]) == index) {
                light_alive_[i] = 0;
            }
        }
    }
}

void Scene::RemoveMeshInstance(MeshInstanceHandle h) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    structure_dirty_ = true;
    RemoveMeshInstance_nolock(h._index);
}

// reference SceneCommon.cpp:121-170 + Core.cpp:1321-1366 (ConstructCamera)
static void make_camera(const camera_desc_t &c, camera_t &cam, ILog *log) {
    cam.desc = c;
    rc_camera &r = cam.rc;
    memset(&r, 0, sizeof(r));
    if (c.type != RS_CAM_PERSP && c.type != RS_CAM_GEO) {
        log->Error("Ray(CUDA): only perspective and Geo cameras are supported by the CUDA backend");
    }
    if (c.type == RS_CAM_GEO && c.uv_index != 0) {
        log->Error("Ray(CUDA): Geo camera uv_index %u: meshes carry one uv set", c.uv_index);
    }
    // the pass-flag bools and mi_index stay in cam.desc: the renderer resolves them at render time
    // AgX / Filmic view transforms need their table (Cuda::Renderer::SetViewTransformLUT): checked at render time
    float o[3] = {c.origin[0], c.origin[1], c.origin[2]}, f[3] = {c.fwd[0], c.fwd[1], c.fwd[2]},
          u[3] = {c.up[0], c.up[1], c.up[2]};
    if ((0.0f + u[0] * u[0]) + u[1] * u[1] + u[2] * u[2] < 0.0000001f) {
        if (fabsf(f[1]) >= 0.999f) {
            u[0] = 1.0f, u[1] = 0.0f, u[2] = 0.0f;
        } else {
            u[0] = 0.0f, u[1] = 1.0f, u[2] = 0.0f;
        }
    }
    float s[3];
    cross3(f, u, s);
    const float sl = sqrtf(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]);
    s[0] /= sl, s[1] /= sl, s[2] /= sl;
    cross3(s, f, u);
    r.type = c.type;
    r.filter = c.filter;
    r.view_transform = c.view_transform;
    r.fov = c.fov;
    r.exposure = c.exposure;
    r.gamma = c.gamma;
    r.sensor_height = c.sensor_height;
    r.focus_distance = fmaxf(c.focus_distance, 0.0f);
    r.focal_length = 0.5f * c.sensor_height / tanf(0.5f * c.fov * PI / 180.0f);
    r.fstop = c.fstop;
    r.lens_rotation = c.lens_rotation;
    r.lens_ratio = c.lens_ratio;
    r.lens_blades = c.lens_blades;
    r.clip_start = c.clip_start;
    r.clip_end = c.clip_end;
    memcpy(r.origin, o, sizeof(o));
    memcpy(r.fwd, f, sizeof(f));
    memcpy(r.side, s, sizeof(s));
    memcpy(r.up, u, sizeof(u));
    memcpy(r.shift, c.shift, sizeof(r.shift));
    r.max_diff_depth = c.max_diff_depth;
    r.max_spec_depth = c.max_spec_depth;
    r.max_refr_depth = c.max_refr_depth;
    r.max_transp_depth = c.max_transp_depth;
    r.max_total_depth = c.max_total_depth;
    r.min_total_depth = c.min_total_depth;
    r.min_transp_depth = c.min_transp_depth;
    r.clamp_direct = c.clamp_direct;
    r.clamp_indirect = c.clamp_indirect;
    r.min_samples = c.min_samples;
    r.variance_threshold = c.variance_threshold;
    r.regularize_alpha = c.regularize_alpha;
}

CameraHandle Scene::AddCamera(const camera_desc_t &c) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    cams_.emplace_back();
    make_camera(c, cams_.back(), log_);
    const CameraHandle h{uint32_t(cams_.size() - 1), 0};
    if (current_cam_._index == 0xffffffffu) {
        current_cam_ = h;
    }
    return h;
}
void Scene::GetCamera(CameraHandle i, camera_desc_t &c) const {
    std::shared_lock<std::shared_timed_mutex> lock(mtx_);
    if (i._index < cams_.size()) {
        c = cams_[i._index].desc;
    }
}
void Scene::SetCamera(CameraHandle i, const camera_desc_t &c) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    if (i._index < cams_.size()) {
        make_camera(c, cams_[i._index], log_);
    }
}

// reference SceneCPU.cpp:882-926
void Scene::Finalize(const ParallelFor &) {
    std::unique_lock<std::shared_timed_mutex> lock(mtx_);
    if (env_light_index_ != 0xffffffffu) {
        light_alive_[env_light_index_] = 0;
        env_light_index_ = 0xffffffffu;
    }
    env_qtree_mips_.clear();
    if (env_.importance_sample && env_.env_col[0] > 0.0f && env_.env_col[1] > 0.0f && env_.env_col[2] > 0.0f) {
        if (env_.env_map != RS_INVALID) {
            PrepareEnvMapQTree_nolock();
        }
        rt::Light l;
        memset(&l, 0, sizeof(l));
        l.bits = light_bits(rt::LIGHT_ENV, false, true, true, false,
                            (1u << rt::RAY_DIFFUSE) | (1u << rt::RAY_SPECULAR) | (1u << rt::RAY_REFR));
        l.col[0] = l.col[1] = l.col[2] = 1.0f;
        env_light_index_ = AddLight_nolock(l);
    }
    RebuildTLAS_nolock();
    RebuildLightTree_nolock();
    GetBounds(bounds_min_, bounds_max_);
    revision_ = NextRevision();
    if (structure_dirty_) { // anything but instance transforms / analytic lights changed: the renderer uploads everything
        structure_revision_ = revision_;
        structure_dirty_ = false;
    }
    RebuildTexViews_nolock();
    RefreshPinnedMirrors_nolock();
}

const Scene::TexImage *Scene::FindTexture(uint32_t handle) const {
    for (const TexImage &t : textures_) {
        if (t.handle == (handle & 0xf0ffffffu)) {
            return &t;
        }
    }
    return nullptr;
}

namespace {
// Core.cpp:110-128 / Core.h:410-417 / CoreRef.h:234-237 on the host (same libm as the reference)
void canonical_to_dir(const float p[2], float y_rotation, float out_d[3]) {
    const float cos_theta = 2 * p[0] - 1;
    float phi = 2 * PI * p[1] + y_rotation;
    if (phi < 0) {
        phi += 2 * PI;
    }
    if (phi > 2 * PI) {
        phi -= 2 * PI;
    }
    const float sin_theta = sqrtf(1 - cos_theta * cos_theta);
    const float sin_phi = sinf(phi);
    const float cos_phi = cosf(phi);
    out_d[0] = sin_theta * cos_phi;
    out_d[1] = cos_theta;
    out_d[2] = -sin_theta * sin_phi;
}
float to_norm_float(uint8_t v) {
    const uint32_t val = 0x3f800000u + v * 0x8080u + (v + 1u) / 2u;
    float f;
    memcpy(&f, &val, 4);
    return f - 1.0f;
}
float fractf_(float v) { return v - floorf(v); }
} // namespace

// reference SceneCPU.cpp:1058-1211
void Scene::PrepareEnvMapQTree_nolock() {
    const TexImage *img = FindTexture(env_.env_map);
    if (!img || img->channels != 4) {
        log_->Error("Ray(CUDA): the environment map must be an RGBA8888 (RGBE) texture of this scene");
        return;
    }
    const int size[2] = {img->w, img->h};
    const int lowest_dim = std::min(size[0], size[1]);
    int res = 1;
    while (2 * res < lowest_dim) {
        res *= 2;
    }
    int cur_res = res;
    float total_lum = 0.0f;
    std::vector<std::vector<float>> mips;
    { // the first quad-tree level: 5x5 Gaussian footprint around every cell centre, looked up through the lat-long mapping
        mips.emplace_back(size_t(cur_res) * cur_res / 4 * 4, 0.0f);
        static const float FilterWeights[][5] = {{1 / 273.0f, 4 / 273.0f, 7 / 273.0f, 4 / 273.0f, 1 / 273.0f},
                                                 {4 / 273.0f, 16 / 273.0f, 26 / 273.0f, 16 / 273.0f, 4 / 273.0f},
                                                 {7 / 273.0f, 26 / 273.0f, 41 / 273.0f, 26 / 273.0f, 7 / 273.0f},
                                                 {4 / 273.0f, 16 / 273.0f, 26 / 273.0f, 16 / 273.0f, 4 / 273.0f},
                                                 {1 / 273.0f, 4 / 273.0f, 7 / 273.0f, 4 / 273.0f, 1 / 273.0f}};
        static const float FilterSize = 0.5f;
        for (int qy = 0; qy < cur_res; ++qy) {
            for (int qx = 0; qx < cur_res; ++qx) {
                for (int jj = -2; jj <= 2; ++jj) {
                    for (int ii = -2; ii <= 2; ++ii) {
                        const float q[2] = {fractf_(1.0f + (float(qx) + 0.5f + ii * FilterSize) / cur_res),
                                            fractf_(1.0f + (float(qy) + 0.5f + jj * FilterSize) / cur_res)};
                        float dir[3];
                        canonical_to_dir(q, 0.0f, dir);
                        const float theta = acosf(std::min(std::max(dir[1], -1.0f), 1.0f)) / PI;
                        float phi = atan2f(dir[2], dir[0]);
                        if (phi < 0) {
                            phi += 2 * PI;
                        }
                        if (phi > 2 * PI) {
                            phi -= 2 * PI;
                        }
                        const float u = fractf_(0.5f * phi / PI);
                        const float uvs[2] = {u * float(size[0]), theta * float(size[1])};
                        const int ix = std::min(std::max(int(uvs[0]), 0), size[0] - 1);
                        const int iy = std::min(std::max(int(uvs[1]), 0), size[1] - 1);
                        const uint8_t *px = &img->pixels[(size_t(iy) * size[0] + ix) * 4];
                        const float f = exp2f(float(px[3]) - 128.0f);
                        const float cur_lum = (to_norm_float(px[0]) * f + to_norm_float(px[1]) * f + to_norm_float(px[2]) * f);
                        const int index = (qx & 1) | ((qy & 1) << 1);
                        float &qv = mips[0][(size_t(qy / 2) * cur_res / 2 + (qx / 2)) * 4 + index];
                        qv = qv + cur_lum * FilterWeights[ii + 2][jj + 2];
                    }
                }
            }
        }
        for (size_t i = 0; i < mips[0].size(); i += 4) {
            const float *v = &mips[0][i];
            total_lum += ((v[0] + v[1]) + v[2]) + v[3]; // fvec4::hsum (SSE2 build of the reference)
        }
        cur_res /= 2;
    }
    while (cur_res > 1) {
        mips.emplace_back(size_t(cur_res) * cur_res / 4 * 4, 0.0f);
        const std::vector<float> &prev = mips[mips.size() - 2];
        for (int y = 0; y < cur_res; ++y) {
            for (int x = 0; x < cur_res; ++x) {
                const float *pv = &prev[(size_t(y) * cur_res + x) * 4];
                const float res_lum = pv[0] + pv[1] + pv[2] + pv[3];
                const int index = (x & 1) | ((y & 1) << 1);
                mips.back()[(size_t(y / 2) * cur_res / 2 + (x / 2)) * 4 + index] = res_lum;
            }
        }
        cur_res /= 2;
    }
    // how many levels are actually required
    static const float LumFractThreshold = 0.005f;
    cur_res = 2;
    int the_last_required_lod = 0;
    for (int lod = int(mips.size()) - 1; lod >= 0; --lod) {
        the_last_required_lod = lod;
        const std::vector<float> &cur = mips[lod];
        bool subdivision_required = false;
        for (int y = 0; y < (cur_res / 2) && !subdivision_required; ++y) {
            for (int x = 0; x < (cur_res / 2) && !subdivision_required; ++x) {
                const float *v = &cur[(size_t(y) * cur_res / 2 + x) * 4];
                const float thr = LumFractThreshold * total_lum;
                subdivision_required |= (v[0] > thr) || (v[1] > thr) || (v[2] > thr) || (v[3] > thr);
            }
        }
        if (!subdivision_required) {
            break;
        }
        cur_res *= 2;
    }
    if (the_last_required_lod > 0) {
        mips.erase(mips.begin(), mips.begin() + the_last_required_lod);
    }
    if (mips.size() > 16) {
        log_->Error("Ray(CUDA): environment quad-tree deeper than 16 levels");
        return;
    }
    env_qtree_mips_ = std::move(mips);
}

// reference SceneCPU.cpp:928-1015
void Scene::RebuildTLAS_nolock() {
    wnodes_.resize(blas_nodes_end_);
    tlas_root_ = 0xffffffffu;
    std::vector<Aabb> boxes;
    std::vector<uint32_t> ids;
    for (uint32_t i = 0; i < mesh_instances_.size(); ++i) {
        if (!instance_alive_[i]) {
            continue;
        }
        Aabb b;
        transform_box(meshes_[mesh_instances_[i].mesh_index].box, mesh_instances_[i].xform, b);
        boxes.push_back(b);
        ids.push_back(i);
    }
    if (boxes.empty()) {
        return;
    }
    std::vector<BinaryNode> bnodes;
    std::vector<uint32_t> order;
    BuildBinaryBVH(boxes, 1, bnodes, order);
    std::vector<rt::WNode> wide;
    const uint32_t base = uint32_t(wnodes_.size());
    auto payload = [&](const BinaryNode &leaf) -> uint32_t { return ids[order[leaf.first]]; };
    tlas_root_ = CollapseToWide(bnodes, 0, wide, base, payload);
    wnodes_.insert(wnodes_.end(), wide.begin(), wide.end());
}

// reference SceneCPU.cpp:1214-1521 (per-light bounds/cones :1240-1383, hierarchy propagation :1410-1456,
// 8-wide quantised flatten Core.cpp:1009-1186, leaf-level collapse SceneCPU.cpp:1469-1518)
void Scene::RebuildLightTree_nolock() {
    li_indices_.clear();
    light_cwnodes_.clear();
    visible_lights_count_ = blocker_lights_count_ = 0;

    std::vector<LightNode> leaves;
    for (uint32_t i = 0; i < lights_.size(); ++i) {
        if (!light_alive_[i]) {
            continue;
        }
        const rt::Light &l = lights_[i];
        LightNode n;
        n.leaf = true;
        n.light_index = i;
        n.box.reset();
        float axis[3] = {0.0f, 1.0f, 0.0f};
        float area = 1.0f, omega_n = 0.0f, omega_e = 0.0f;
        float lum = l.col[0] + l.col[1] + l.col[2];
        li_indices_.push_back(i);
        if (l_visible(l)) {
            ++visible_lights_count_;
        }
        if (l_ray_vis(l) & (1u << rt::RAY_SHADOW)) {
            ++blocker_lights_count_;
        }
        auto corner_box = [&](const float pos[3], const float a[3], const float b[3], const float c[3]) {
            for (int sa = -1; sa <= 1; sa += 2) {
                for (int sb = -1; sb <= 1; sb += 2) {
                    for (int sc = -1; sc <= 1; sc += 2) {
                        const float p[3] = {pos[0] + sa * a[0] + sb * b[0] + sc * c[0], pos[1] + sa * a[1] + sb * b[1] + sc * c[1],
                                            pos[2] + sa * a[2] + sb * b[2] + sc * c[2]};
                        n.box.grow(p);
                    }
                }
            }
        };
        const float zero[3] = {0, 0, 0};
        switch (l_type(l)) {
        case rt::LIGHT_SPHERE: {
            const float r = l.p[7];
            const float lo[3] = {l.p[0] - r, l.p[1] - r, l.p[2] - r}, hi[3] = {l.p[0] + r, l.p[1] + r, l.p[2] + r};
            n.box.grow(lo);
            n.box.grow(hi);
            if (l.p[3] != 0.0f) {
                area = l.p[3];
            }
            omega_n = PI;
            omega_e = PI / 2.0f;
        } break;
        case rt::LIGHT_DIR: {
            n.infinite = true;
            axis[0] = l.p[0], axis[1] = l.p[1], axis[2] = l.p[2];
            omega_n = 0.0f;
            omega_e = l.p[5];
            if (l.p[4] != 0.0f) {
                area = PI * l.p[4] * l.p[4];
            }
        } break;
        case rt::LIGHT_LINE: {
            float lv[3];
            cross3(&l.p[4], &l.p[8], lv);
            const float r = l.p[7], hh = 0.5f * l.p[11];
            const float a[3] = {l.p[4] * r, l.p[5] * r, l.p[6] * r}, b[3] = {lv[0] * r, lv[1] * r, lv[2] * r},
                        c[3] = {l.p[8] * hh, l.p[9] * hh, l.p[10] * hh};
            corner_box(&l.p[0], a, b, c);
            area = l.p[3];
            omega_n = PI;
            omega_e = PI / 2.0f;
        } break;
        case rt::LIGHT_RECT:
        case rt::LIGHT_DISK: {
            const float a[3] = {0.5f * l.p[4], 0.5f * l.p[5], 0.5f * l.p[6]}, b[3] = {0.5f * l.p[8], 0.5f * l.p[9], 0.5f * l.p[10]};
            corner_box(&l.p[0], a, b, zero);
            area = l.p[3];
            float nn[3];
            cross3(a, b, nn);
            const float nl = len3(nn);
            if (nl > 0) {
                axis[0] = nn[0] / nl, axis[1] = nn[1] / nl, axis[2] = nn[2] / nl;
            }
            omega_n = l_doublesided(l) ? PI : 0.0f;
            omega_e = PI / 2.0f;
        } break;
        case rt::LIGHT_TRI: {
            const uint32_t tri = f2u(l.p[0]);
            const rt::MeshInstance &lmi = mesh_instances_[f2u(l.p[1])];
            float p1[3], p2[3], p3[3];
            xform_point(lmi.xform, vertices_[vtx_indices_[size_t(tri) * 3 + 0]].p, p1);
            xform_point(lmi.xform, vertices_[vtx_indices_[size_t(tri) * 3 + 1]].p, p2);
            xform_point(lmi.xform, vertices_[vtx_indices_[size_t(tri) * 3 + 2]].p, p3);
            n.box.grow(p1);
            n.box.grow(p2);
            n.box.grow(p3);
            const float e1[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]}, e2[3] = {p3[0] - p1[0], p3[1] - p1[1], p3[2] - p1[2]};
            float nn[3];
            cross3(e1, e2, nn);
            const float nl = len3(nn);
            area = 0.5f * nl;
            if (nl > 0) {
                axis[0] = nn[0] / nl, axis[1] = nn[1] / nl, axis[2] = nn[2] / nl;
            }
            omega_n = l_doublesided(l) ? PI : 0.0f;
            omega_e = PI / 2.0f;
        } break;
        case rt::LIGHT_ENV: {
            // without an environment map the reference's env_map_qtree_.medium_lum is 0, i.e. the constant environment
            // gets zero flux in the tree (SceneCPU.cpp:1367) and is reached through BSDF sampling only
            lum = (lum / 3.0f) * 0.0f;
            n.infinite = true;
            omega_n = PI;
            omega_e = PI / 2.0f;
        } break;
        default:
            continue;
        }
        n.flux = lum * area;
        memcpy(n.axis, axis, sizeof(axis));
        n.omega_n = omega_n;
        n.omega_e = omega_e;
        leaves.push_back(n);
    }
    if (leaves.empty()) {
        return;
    }

    // binary hierarchy over the light boxes (infinite lights sit at the centre of the finite ones)
    Aabb finite;
    finite.reset();
    bool any_finite = false;
    for (const LightNode &n : leaves) {
        if (!n.infinite) {
            finite.grow(n.box);
            any_finite = true;
        }
    }
    std::vector<Aabb> boxes(leaves.size());
    for (size_t i = 0; i < leaves.size(); ++i) {
        if (leaves[i].infinite) {
            Aabb b;
            for (int a = 0; a < 3; ++a) {
                b.mn[a] = b.mx[a] = any_finite ? 0.5f * (finite.mn[a] + finite.mx[a]) : 0.0f;
            }
            boxes[i] = b;
        } else {
            boxes[i] = leaves[i].box;
        }
    }
    std::vector<BinaryNode> bnodes;
    std::vector<uint32_t> order;
    BuildBinaryBVH(boxes, 1, bnodes, order);

    std::vector<LightNode> ln(bnodes.size());
    // children always have larger indices than their parent in BuildBinaryBVH's output: walk backwards = bottom-up
    for (int i = int(bnodes.size()) - 1; i >= 0; --i) {
        const BinaryNode &b = bnodes[i];
        if (b.count != 0) {
            ln[i] = leaves[order[b.first]];
            continue;
        }
        LightNode &p = ln[i];
        const LightNode &c0 = ln[b.left], &c1 = ln[b.right];
        p.leaf = false;
        p.left = b.left;
        p.right = b.right;
        p.infinite = c0.infinite && c1.infinite;
        p.box.reset();
        if (!c0.infinite) {
            p.box.grow(c0.box);
        }
        if (!c1.infinite) {
            p.box.grow(c1.box);
        }
        p.flux = c0.flux + c1.flux;
        // cone union as the reference propagates it (SceneCPU.cpp:1424-1453)
        memcpy(p.axis, c0.axis, sizeof(p.axis));
        p.omega_n = c0.omega_n;
        {
            const float d = clampf(dot3(p.axis, c1.axis), -1.0f, 1.0f);
            const float angle_between = acosf(d);
            float ax[3] = {p.axis[0] + c1.axis[0], p.axis[1] + c1.axis[1], p.axis[2] + c1.axis[2]};
            const float al = len3(ax);
            if (al != 0.0f) {
                ax[0] /= al, ax[1] /= al, ax[2] /= al;
            } else {
                ax[0] = 0.0f, ax[1] = 1.0f, ax[2] = 0.0f;
            }
            memcpy(p.axis, ax, sizeof(ax));
            p.omega_n = fminf(0.5f * (p.omega_n + fmaxf(p.omega_n, angle_between + c1.omega_n)), PI);
            // make sure the merged cone covers both children
            p.omega_n = fminf(fmaxf(p.omega_n, 0.5f * angle_between + fmaxf(c0.omega_n, c1.omega_n)), PI);
        }
        p.omega_e = fmaxf(c0.omega_e, c1.omega_e);
    }

    // 8-wide flatten with the leaf level folded into the parents
    struct Emit {
        std::vector<rt::LightCWNode> &out;
        const std::vector<LightNode> &ln;
        uint32_t run(uint32_t node) {
            const uint32_t my = uint32_t(out.size());
            out.emplace_back();
            memset(&out[my], 0, sizeof(rt::LightCWNode));
            uint32_t kids[8];
            int nk = 0;
            if (ln[node].leaf) {
                kids[nk++] = node;
            } else {
                kids[nk++] = ln[node].left;
                kids[nk++] = ln[node].right;
                while (nk < 8) {
                    int best = -1;
                    float best_flux = -1.0f;
                    for (int i = 0; i < nk; ++i) {
                        if (!ln[kids[i]].leaf && ln[kids[i]].flux > best_flux) {
                            best_flux = ln[kids[i]].flux;
                            best = i;
                        }
                    }
                    if (best < 0) {
                        break;
                    }
                    const LightNode &c = ln[kids[best]];
                    kids[best] = c.left;
                    kids[nk++] = c.right;
                }
            }
            Aabb all;
            all.reset();
            for (int i = 0; i < nk; ++i) {
                if (!ln[kids[i]].infinite) {
                    all.grow(ln[kids[i]].box);
                }
            }
            uint32_t ids[8];
            for (int i = 0; i < 8; ++i) {
                if (i >= nk) {
                    ids[i] = rt::kEmptyChild;
                } else if (ln[kids[i]].leaf) {
                    ids[i] = rt::kLeafBit | ln[kids[i]].light_index;
                } else {
                    ids[i] = run(kids[i]);
                }
            }
            rt::LightCWNode &w = out[my];
            memcpy(w.bbox_min, all.mn, sizeof(all.mn));
            memcpy(w.bbox_max, all.mx, sizeof(all.mx));
            for (int i = 0; i < 8; ++i) {
                w.child[i] = ids[i];
                if (i >= nk) {
                    for (int a = 0; a < 3; ++a) {
                        w.ch_bbox_min[a][i] = 0xff;
                        w.ch_bbox_max[a][i] = 0xff;
                    }
                    continue;
                }
                const LightNode &c = ln[kids[i]];
                if (!c.infinite) {
                    for (int a = 0; a < 3; ++a) {
                        w.ch_bbox_min[a][i] = uint8_t(floorf(quantize(c.box.mn[a], all.mn[a], all.mx[a])));
                        w.ch_bbox_max[a][i] = uint8_t(ceilf(quantize(c.box.mx[a], all.mn[a], all.mx[a])));
                    }
                } else {
                    for (int a = 0; a < 3; ++a) {
                        w.ch_bbox_min[a][i] = 0xff;
                        w.ch_bbox_max[a][i] = 0;
                    }
                }
                w.flux[i] = c.flux;
                w.axis[i] = encode_oct_dir(c.axis);
                w.cos_omega_ne[i] = encode_cosines(cosf(c.omega_n), fmaxf(cosf(c.omega_e), 0.0f));
            }
            return my;
        }
    } emit{light_cwnodes_, ln};
    emit.run(0);
}

// reference SceneCPU.cpp:1523-1580
void Scene::GetBounds(float bbox_min[3], float bbox_max[3]) const {
    bbox_min[0] = bbox_min[1] = bbox_min[2] = MAX_DIST;
    bbox_max[0] = bbox_max[1] = bbox_max[2] = -MAX_DIST;
    if (tlas_root_ != 0xffffffffu) {
        const rt::WNode &root = wnodes_[tlas_root_];
        if (root.child[0] & rt::kLeafBit) {
            for (int i = 0; i < 3; ++i) {
                bbox_min[i] = root.bbox_min[i][0];
                bbox_max[i] = root.bbox_max[i][0];
            }
        } else {
            for (int j = 0; j < 8; ++j) {
                if (root.child[j] == rt::kEmptyChild) {
                    continue;
                }
                for (int i = 0; i < 3; ++i) {
                    bbox_min[i] = fminf(bbox_min[i], root.bbox_min[i][j]);
                    bbox_max[i] = fmaxf(bbox_max[i], root.bbox_max[i][j]);
                }
            }
        }
    }
    if (!light_cwnodes_.empty() && light_cwnodes_[0].bbox_min[0] <= light_cwnodes_[0].bbox_max[0]) {
        for (int i = 0; i < 3; ++i) {
            bbox_min[i] = fminf(bbox_min[i], light_cwnodes_[0].bbox_min[i]);
            bbox_max[i] = fmaxf(bbox_max[i], light_cwnodes_[0].bbox_max[i]);
        }
    }
}

bool Scene::GetDeviceCamera(rc_camera &out) const {
    std::shared_lock<std::shared_timed_mutex> lock(mtx_);
    if (current_cam_._index >= cams_.size()) {
        return false;
    }
    out = cams_[current_cam_._index].rc;
    return true;
}

void Scene::FillView(rc_scene_view &v) const {
    memset(&v, 0, sizeof(v));
    v.wnodes = {wnodes_.data(), uint32_t(wnodes_.size()), uint32_t(sizeof(rt::WNode))};
    v.mtris = {mtris_.data(), uint32_t(mtris_.size()), uint32_t(sizeof(rt::MTri))};
    v.tri_indices = {tri_indices_.data(), uint32_t(tri_indices_.size()), 4u};
    v.tri_materials = {tri_materials_.data(), uint32_t(tri_materials_.size()), uint32_t(sizeof(rt::TriMat))};
    v.materials = {materials_.data(), uint32_t(materials_.size()), uint32_t(sizeof(rt::Material))};
    v.mesh_instances = {mesh_instances_.data(), uint32_t(mesh_instances_.size()), uint32_t(sizeof(rt::MeshInstance))};
    v.vertices = {vertices_.data(), uint32_t(vertices_.size()), uint32_t(sizeof(rt::Vertex))};
    v.vtx_indices = {vtx_indices_.data(), uint32_t(vtx_indices_.size()), 4u};
    v.lights = {lights_.data(), uint32_t(lights_.size()), uint32_t(sizeof(rt::Light))};
    v.li_indices = {li_indices_.data(), uint32_t(li_indices_.size()), 4u};
    v.light_cwnodes = {light_cwnodes_.data(), uint32_t(light_cwnodes_.size()), uint32_t(sizeof(rt::LightCWNode))};
    v.tlas_root = tlas_root_;
    v.visible_lights_count = visible_lights_count_;
    v.blocker_lights_count = blocker_lights_count_;
    memcpy(v.env_col, env_.env_col, sizeof(v.env_col));
    v.env_map = env_.env_map;
    memcpy(v.back_col, env_.back_col, sizeof(v.back_col));
    v.back_map = env_.back_map;
    v.env_map_rotation = env_.env_map_rotation;
    v.back_map_rotation = env_.back_map_rotation;
    v.qtree_levels = int(env_qtree_mips_.size());
    for (int i = 0; i < v.qtree_levels; ++i) {
        v.qtree_mips[i] = env_qtree_mips_[i].data();
    }
    v.env_light_index = env_light_index_;
    v.sky_map_spread_angle = 0.0f;
    memcpy(v.bounds_min, bounds_min_, sizeof(v.bounds_min));
    memcpy(v.bounds_max, bounds_max_, sizeof(v.bounds_max));
    if (pinned_revision_ == revision_) { // same bytes, page-locked
        const rc_array *dst[PM_COUNT] = {&v.wnodes, &v.mtris, &v.vertices, &v.vtx_indices, &v.tri_indices, &v.tri_materials};
        for (int i = 0; i < PM_COUNT; ++i) {
            if (pinned_[i].bytes == size_t(dst[i]->count) * dst[i]->stride && pinned_[i].bytes != 0) {
                const_cast<rc_array *>(dst[i])->ptr = pinned_[i].ptr;
            }
        }
    }
    v.textures = tex_views_.empty() ? nullptr : tex_views_.data();
    v.texture_count = uint32_t(tex_views_.size());
}

} // namespace Cuda
} // namespace RayB200
