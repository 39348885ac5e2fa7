// rt_shade.cuh -- BSDF evaluation/sampling and the surface shader (ShadeSurface) for one ray/hit pair.
//
// Behavioural spec: reference internal/ShadeRef.cpp
//   calc_alpha :12-19            get_lobe_weights :32-52        fresnel_dielectric_cos :54-70
//   VNDF sampling (spherical cap, bounded) :118-179             GGX_VNDF_Reflection_Bounded_PDF :181-193
//   G1 :196-203   D_GTR1 :211-218   D_GGX :226-235              ensure_valid_reflection :238-333 (normal maps only)
//   IOR stack :355-381           BRDF_PrincipledDiffuse :383-401
//   Oren diffuse :403-440        principled diffuse+sheen :442-488    GGX specular :490-532
//   GGX refraction :534-595      clearcoat :597-643                   node wrappers :645-809
//   Evaluate/Sample_PrincipledNode :811-1028    Evaluate_EnvColor :1030-1066   Evaluate_LightColor :1068-1172
//   ShadeSurface :1174-1652
// Out of scope here (rc_upload_scene rejects such scenes): textures (base/rough/metal/spec/normal maps, textured tri
// lights), env maps + env quad-tree, spatial radiance cache, deferred procedural sky.
#pragma once

#include "rt_lights.cuh"

namespace rt {

struct PassSettings { // pass_settings_t, reference Types.h:92-100 (the pass flags travel in KParams::flags)
    int max_diff_depth, max_spec_depth, max_refr_depth, max_transp_depth, max_total_depth;
    int min_total_depth, min_transp_depth;
    float clamp_direct, clamp_indirect;
    float regularize_alpha;
};

struct RayD { // Ref::ray_data_t in registers
    v3 o, d;
    float pdf;
    v3 c;
    float ior[4];
    float cone_width, cone_spread;
    uint32_t xy, depth;
};

struct ShadowRayD { // Ref::shadow_ray_t in registers
    v3 o;
    uint32_t depth;
    v3 d;
    float dist;
    v3 c;
    uint32_t xy;
};


struct Surface {
    v3 P, T, B, N, plane_N;
    v2 uvs;
};

RT_FN v2 calc_alpha(float roughness, float anisotropy, float regularize_alpha) {
    const float roughness2 = sqr(roughness);
    const float aspect = sqrtf(1.0f - 0.9f * anisotropy);
    v2 alpha = v2{roughness2 / aspect, roughness2 * aspect};
    // where(alpha < reg, alpha) = clamp(2 * alpha, 0.25 * reg, reg); generic fvec<2>: min(max(v, lo), hi) with std::
    const float lo = 0.25f * regularize_alpha;
    if (alpha.x < regularize_alpha) {
        alpha.x = std_min(std_max(2 * alpha.x, lo), regularize_alpha);
    }
    if (alpha.y < regularize_alpha) {
        alpha.y = std_min(std_max(2 * alpha.y, lo), regularize_alpha);
    }
    return alpha;
}

RT_DEV float pow5(float v) { return (v * v) * (v * v) * v; }
RT_DEV float schlick_weight(float u) { return pow5(saturatef(1.0f - u)); }
RT_DEV v3 reflect(v3 I, v3 N, float dot_N_I) { return I - 2 * dot_N_I * N; }

struct LobeWeights {
    float diffuse, specular, clearcoat, refraction;
};

RT_FN LobeWeights get_lobe_weights(float base_color_lum, float spec_color_lum, float specular, float metallic,
                                    float transmission, float clearcoat) {
    LobeWeights w;
    w.diffuse = base_color_lum * (1.0f - metallic) * (1.0f - transmission);
    const float final_transmission = transmission * (1.0f - metallic);
    w.specular = (specular != 0.0f || metallic != 0.0f) ? spec_color_lum * (1.0f - final_transmission) : 0.0f;
    w.clearcoat = 0.25f * clearcoat * (1.0f - metallic);
    w.refraction = final_transmission * base_color_lum;
    const float total_weight = w.diffuse + w.specular + w.clearcoat + w.refraction;
    if (total_weight != 0.0f) {
        w.diffuse /= total_weight;
        w.specular /= total_weight;
        w.clearcoat /= total_weight;
        w.refraction /= total_weight;
    }
    return w;
}

RT_FN float fresnel_dielectric_cos(float cosi, float eta) {
    const float c = fabsf(cosi);
    float g = eta * eta - 1 + c * c;
    float result;
    if (g > 0) {
        g = sqrtf(g);
        const float A = (g - c) / (g + c);
        const float B = (c * (g + c) - 1) / (c * (g - c) + 1);
        result = 0.5f * A * A * (1 + B * B);
    } else {
        result = 1.0f;
    }
    return result;
}

RT_DEV v3 sample_vndf_sphcap(v3 Vh, v2 rand) {
    const float phi = 2.0f * kPi * rand.x;
    const float z = __fmaf_rn(1.0f - rand.y, 1.0f + Vh.z, -Vh.z);
    const float sin_theta = sqrtf(saturatef(1.0f - z * z));
    const v2 sc = portable_sincos(phi);
    const float x = sin_theta * sc.y;
    const float y = sin_theta * sc.x;
    return v3{x, y, z} + Vh;
}

RT_DEV v3 sample_vndf_sphcap_bounded(v3 Ve, v3 Vh, v2 alpha, v2 rand) {
    const float phi = 2.0f * kPi * rand.x;
    const float a = saturatef(fminf(alpha.x, alpha.y));
    const float s = 1.0f + length(v2{Ve.x, Ve.y});
    const float a2 = a * a, s2 = s * s;
    const float k = (1.0f - a2) * s2 / (s2 + a2 * Ve.z * Ve.z);
    const float b = (Ve.z > 0.0f) ? k * Vh.z : Vh.z;
    const float z = __fmaf_rn(1.0f - rand.y, 1.0f + b, -b);
    const float sin_theta = sqrtf(saturatef(1.0f - z * z));
    const v2 sc = portable_sincos(phi);
    const float x = sin_theta * sc.y;
    const float y = sin_theta * sc.x;
    return v3{x, y, z} + Vh;
}

RT_FN v3 sample_ggx_vndf(v3 Ve, v2 alpha, v2 rand) {
    const v3 Vh = normalize(v3{alpha.x * Ve.x, alpha.y * Ve.y, Ve.z});
    const v3 Nh = sample_vndf_sphcap(Vh, rand);
    return normalize(v3{alpha.x * Nh.x, alpha.y * Nh.y, fmaxf(0.0f, Nh.z)});
}

RT_FN v3 sample_ggx_vndf_bounded(v3 Ve, v2 alpha, v2 rand) {
    const v3 Vh = normalize(v3{alpha.x * Ve.x, alpha.y * Ve.y, Ve.z});
    const v3 Nh = sample_vndf_sphcap_bounded(Ve, Vh, alpha, rand);
    return normalize(v3{alpha.x * Nh.x, alpha.y * Nh.y, fmaxf(0.0f, Nh.z)});
}

RT_FN float ggx_vndf_reflection_bounded_pdf(float D, v3 view_dir_ts, v2 alpha) {
    const v2 ai = alpha * v2{view_dir_ts.x, view_dir_ts.y};
    const float len2 = dot(ai, ai);
    const float t = sqrtf(len2 + view_dir_ts.z * view_dir_ts.z);
    if (view_dir_ts.z >= 0.0f) {
        const float a = saturatef(fminf(alpha.x, alpha.y));
        const float s = 1.0f + length(v2{view_dir_ts.x, view_dir_ts.y});
        const float a2 = a * a, s2 = s * s;
        const float k = (1.0f - a2) * s2 / (s2 + a2 * view_dir_ts.z * view_dir_ts.z);
        return D / (2.0f * (k * view_dir_ts.z + t));
    }
    return D * (t - view_dir_ts.z) / (2.0f * len2);
}

RT_FN float G1(v3 Ve, v2 alpha) {
    alpha = alpha * alpha;
    const float delta =
        (-1.0f + sqrtf(1.0f + safe_div_pos(alpha.x * sqr(Ve.x) + alpha.y * sqr(Ve.y), sqr(Ve.z)))) / 2.0f;
    return 1.0f / (1.0f + delta);
}

RT_DEV float D_GTR1(float NDotH, float a) {
    if (a >= 1.0f) {
        return 1.0f / kPi;
    }
    const float a2 = sqr(a);
    const float t = 1.0f + (a2 - 1.0f) * NDotH * NDotH;
    // NOTE: the reference calls libm logf here; CUDA's logf may differ from glibc's by 1 ulp (clearcoat lobe only)
    return (a2 - 1.0f) / (kPi * libm_logf(a2) * t);
}

RT_FN float D_GGX(v3 H, v2 alpha) {
    if (H.z == 0.0f) {
        return 0.0f;
    }
    const float sx = -H.x / (H.z * alpha.x);
    const float sy = -H.y / (H.z * alpha.y);
    const float s1 = 1.0f + sx * sx + sy * sy;
    const float cos_theta_h4 = sqr(sqr(H.z));
    return 1.0f / (sqr(s1) * kPi * alpha.x * alpha.y * cos_theta_h4);
}

RT_DEV void push_ior_stack(float stack[4], float val) {
    if (stack[0] < 0.0f) {
        stack[0] = val;
        return;
    }
    if (stack[1] < 0.0f) {
        stack[1] = val;
        return;
    }
    if (stack[2] < 0.0f) {
        stack[2] = val;
        return;
    }
    stack[3] = val;
}

RT_DEV void pop_ior_stack(float stack[4]) {
#pragma unroll
    for (int i = 3; i >= 0; --i) {
        if (stack[i] > 0.0f) {
            stack[i] = -1.0f;
            return;
        }
    }
}

RT_DEV float peek_ior_stack(const float stack[4], bool skip_first) {
#pragma unroll
    for (int i = 3; i >= 0; --i) {
        if (stack[i] > 0.0f) {
            if (!skip_first) {
                return stack[i];
            }
            skip_first = false;
        }
    }
    return 1.0f;
}

RT_DEV float brdf_principled_diffuse(v3 V, v3 N, v3 L, v3 H, float roughness) {
    const float N_dot_L = dot(N, L);
    const float N_dot_V = dot(N, V);
    if (N_dot_L <= 0.0f) {
        return 0.0f;
    }
    const float FL = schlick_weight(N_dot_L);
    const float FV = schlick_weight(N_dot_V);
    const float L_dot_H = dot(L, H);
    const float Fd90 = 0.5f + 2.0f * L_dot_H * L_dot_H * roughness;
    return mixf(1.0f, Fd90, FL) * mixf(1.0f, Fd90, FV);
}

RT_FN c4 eval_oren_diffuse(v3 V, v3 N, v3 L, float roughness, v3 base_color) {
    const float sigma = roughness;
    const float div = 1.0f / (kPi + ((3.0f * kPi - 4.0f) / 6.0f) * sigma);
    const float a = 1.0f * div;
    const float b = sigma * div;
    const float nl = fmaxf(dot(N, L), 0.0f);
    const float nv = fmaxf(dot(N, V), 0.0f);
    float t = dot(L, V) - nl * nv;
    if (t > 0.0f) {
        t /= fmaxf(nl, nv) + kFltMin;
    }
    const float is = nl * (a + b * t);
    return c4{is * base_color.x, is * base_color.y, is * base_color.z, 0.5f / kPi};
}

RT_FN c4 sample_oren_diffuse(v3 T, v3 B, v3 N, v3 I, float roughness, v3 base_color, v2 rand, v3 &out_V) {
    const float phi = 2 * kPi * rand.y;
    const v2 sc = portable_sincos(phi);
    const float cos_phi = sc.y, sin_phi = sc.x;
    // Appendix C.1 of SURVEY.md: Ref uses rand.x * rand.y here (not rand.x^2); reproduced on purpose.
    const float dir = sqrtf(1.0f - rand.x * rand.y);
    const v3 V = v3{dir * cos_phi, dir * sin_phi, rand.x};
    out_V = world_from_tangent(T, B, N, V);
    return eval_oren_diffuse(-I, N, out_V, roughness, base_color);
}

RT_FN c4 eval_principled_diffuse(v3 V, v3 N, v3 L, float roughness, v3 base_color, v3 sheen_color) {
    const float weight = 1.0f;
    const float pdf = dot(N, L) / kPi;
    v3 H = normalize(L + V);
    if (dot(V, H) < 0.0f) {
        H = -H;
    }
    v3 diff_col = base_color * (weight * brdf_principled_diffuse(V, N, L, H, roughness));
    const float FH = kPi * schlick_weight(dot(L, H));
    diff_col += FH * sheen_color;
    return c4{diff_col.x, diff_col.y, diff_col.z, pdf};
}

RT_FN c4 sample_principled_diffuse(v3 T, v3 B, v3 N, v3 I, float roughness, v3 base_color, v3 sheen_color, v2 rand,
                                    v3 &out_V) {
    const float phi = 2 * kPi * rand.y;
    const v2 sc = portable_sincos(phi);
    const float cos_phi = sc.y, sin_phi = sc.x;
    const float dir = sqrtf(rand.x);
    const float k = sqrtf(1.0f - rand.x);
    const v3 V = v3{dir * cos_phi, dir * sin_phi, k};
    out_V = world_from_tangent(T, B, N, V);
    return eval_principled_diffuse(-I, N, out_V, roughness, base_color, sheen_color);
}

RT_FN c4 eval_ggx_specular(v3 view_dir_ts, v3 sampled_normal_ts, v3 reflected_dir_ts, v2 alpha, float spec_ior,
                            float spec_F0, v3 spec_col, v3 spec_col_90) {
    const float D = D_GGX(sampled_normal_ts, alpha);
    const float G = G1(view_dir_ts, alpha) * G1(reflected_dir_ts, alpha);
    const float FH =
        (fresnel_dielectric_cos(dot(view_dir_ts, sampled_normal_ts), spec_ior) - spec_F0) / (1.0f - spec_F0);
    v3 F = mix3(spec_col, spec_col_90, FH);
    const float denom = 4.0f * fabsf(view_dir_ts.z * reflected_dir_ts.z);
    F *= (denom != 0.0f) ? (D * G / denom) : 0.0f;
    F *= fmaxf(reflected_dir_ts.z, 0.0f);
    const float pdf = ggx_vndf_reflection_bounded_pdf(D, view_dir_ts, alpha);
    return c4{F.x, F.y, F.z, pdf};
}

RT_FN c4 sample_ggx_specular(v3 T, v3 B, v3 N, v3 I, v2 alpha, float spec_ior, float spec_F0, v3 spec_col,
                              v3 spec_col_90, v2 rand, v3 &out_V) {
    if (alpha.x * alpha.y < 1e-7f) {
        const v3 V = reflect(I, N, dot(N, I));
        const float FH = (fresnel_dielectric_cos(dot(V, N), spec_ior) - spec_F0) / (1.0f - spec_F0);
        const v3 F = mix3(spec_col, spec_col_90, FH);
        out_V = V;
        return c4{F.x * 1e6f, F.y * 1e6f, F.z * 1e6f, 1e6f};
    }
    const v3 view_dir_ts = normalize(tangent_from_world(T, B, N, -I));
    const v3 sampled_normal_ts = sample_ggx_vndf_bounded(view_dir_ts, alpha, rand);
    const float dot_N_V = -dot(sampled_normal_ts, view_dir_ts);
    const v3 reflected_dir_ts = normalize(reflect(-view_dir_ts, sampled_normal_ts, dot_N_V));
    out_V = world_from_tangent(T, B, N, reflected_dir_ts);
    return eval_ggx_specular(view_dir_ts, sampled_normal_ts, reflected_dir_ts, alpha, spec_ior, spec_F0, spec_col,
                             spec_col_90);
}

RT_FN c4 eval_ggx_refraction(v3 view_dir_ts, v3 sampled_normal_ts, v3 refr_dir_ts, v2 alpha, float eta, v3 refr_col) {
    if (refr_dir_ts.z >= 0.0f || view_dir_ts.z <= 0.0f || alpha.x * alpha.y < 1e-7f) {
        return c4{0.0f, 0.0f, 0.0f, 0.0f};
    }
    const float D = D_GGX(sampled_normal_ts, alpha);
    const float G1o = G1(refr_dir_ts, alpha), G1i = G1(view_dir_ts, alpha);
    const float denom = dot(refr_dir_ts, sampled_normal_ts) + dot(view_dir_ts, sampled_normal_ts) * eta;
    const float jacobian = safe_div_pos(fmaxf(-dot(refr_dir_ts, sampled_normal_ts), 0.0f), denom * denom);
    const float F = D * G1i * G1o * fmaxf(dot(view_dir_ts, sampled_normal_ts), 0.0f) * jacobian / (view_dir_ts.z);
    const float pdf = D * G1o * fmaxf(dot(view_dir_ts, sampled_normal_ts), 0.0f) * jacobian / view_dir_ts.z;
    return c4{F * refr_col.x, F * refr_col.y, F * refr_col.z, pdf};
}

// out_V.w of the reference (the `m` term) is never read by the callers on this path; only xyz is returned.
RT_FN c4 sample_ggx_refraction(v3 T, v3 B, v3 N, v3 I, v2 alpha, float eta, v3 refr_col, v2 rand, v3 &out_V) {
    if (alpha.x * alpha.y < 1e-7f) {
        const float cosi = -dot(I, N);
        const float cost2 = 1.0f - eta * eta * (1.0f - cosi * cosi);
        if (cost2 < 0) {
            return c4{0.0f, 0.0f, 0.0f, 0.0f};
        }
        const float m = eta * cosi - sqrtf(cost2);
        out_V = normalize(eta * I + m * N);
        return c4{refr_col.x * 1e6f, refr_col.y * 1e6f, refr_col.z * 1e6f, 1e6f};
    }
    const v3 view_dir_ts = normalize(tangent_from_world(T, B, N, -I));
    const v3 sampled_normal_ts = sample_ggx_vndf(view_dir_ts, alpha, rand);
    const float cosi = dot(view_dir_ts, sampled_normal_ts);
    const float cost2 = 1.0f - eta * eta * (1.0f - cosi * cosi);
    if (cost2 < 0) {
        return c4{0.0f, 0.0f, 0.0f, 0.0f};
    }
    const float m = eta * cosi - sqrtf(cost2);
    const v3 refr_dir_ts = normalize(-eta * view_dir_ts + m * sampled_normal_ts);
    const c4 F = eval_ggx_refraction(view_dir_ts, sampled_normal_ts, refr_dir_ts, alpha, eta, refr_col);
    out_V = world_from_tangent(T, B, N, refr_dir_ts);
    return F;
}

RT_FN c4 eval_clearcoat(v3 view_dir_ts, v3 sampled_normal_ts, v3 reflected_dir_ts, float clearcoat_roughness2,
                         float clearcoat_ior, float clearcoat_F0) {
    const float D = D_GTR1(sampled_normal_ts.z, clearcoat_roughness2);
    const v2 clearcoat_alpha = v2{0.25f * 0.25f, 0.25f * 0.25f};
    const float G = G1(view_dir_ts, clearcoat_alpha) * G1(reflected_dir_ts, clearcoat_alpha);
    const float FH = (fresnel_dielectric_cos(dot(reflected_dir_ts, sampled_normal_ts), clearcoat_ior) - clearcoat_F0) /
                     (1.0f - clearcoat_F0);
    float F = mixf(0.04f, 1.0f, FH);
    const float denom = 4.0f * fabsf(view_dir_ts.z) * fabsf(reflected_dir_ts.z);
    F *= (denom != 0.0f) ? D * G / denom : 0.0f;
    F *= fmaxf(reflected_dir_ts.z, 0.0f);
    const float pdf = ggx_vndf_reflection_bounded_pdf(D, view_dir_ts, clearcoat_alpha);
    return c4{F, F, F, pdf};
}

RT_FN c4 sample_clearcoat(v3 T, v3 B, v3 N, v3 I, float clearcoat_roughness2, float clearcoat_ior, float clearcoat_F0,
                           v2 rand, v3 &out_V) {
    if (sqr(clearcoat_roughness2) < 1e-7f) {
        const v3 V = reflect(I, N, dot(N, I));
        const float FH = (fresnel_dielectric_cos(dot(V, N), clearcoat_ior) - clearcoat_F0) / (1.0f - clearcoat_F0);
        const float F = mixf(0.04f, 1.0f, FH);
        out_V = V;
        return c4{F * 1e6f, F * 1e6f, F * 1e6f, 1e6f};
    }
    const v3 view_dir_ts = normalize(tangent_from_world(T, B, N, -I));
    // fvec2 constructed from one float: both lanes = clearcoat_roughness2
    const v3 sampled_normal_ts =
        sample_ggx_vndf_bounded(view_dir_ts, v2{clearcoat_roughness2, clearcoat_roughness2}, rand);
    const float dot_N_V = -dot(sampled_normal_ts, view_dir_ts);
    const v3 reflected_dir_ts = normalize(reflect(-view_dir_ts, sampled_normal_ts, dot_N_V));
    out_V = world_from_tangent(T, B, N, reflected_dir_ts);
    return eval_clearcoat(view_dir_ts, sampled_normal_ts, reflected_dir_ts, clearcoat_roughness2, clearcoat_ior,
                          clearcoat_F0);
}

struct SpecParams {
    v3 tmp_col;
    float roughness, ior, F0, anisotropy;
};
struct CoatParams {
    float roughness, ior, F0;
};
struct TransParams {
    float roughness, int_ior, eta, fresnel;
    bool backfacing;
};

RT_DEV float unorm16(uint16_t v) { return float(v) / 65535.0f; }

struct ShadeScene {
    SceneGeo geo;
    SceneSurf surf;
    SceneLights lights;
    SceneTex tex;
    const uint32_t *__restrict__ rand_seq;
    uint32_t li_count; // li_indices.size()
};

struct ShadeOut {
    c4 col;            // colour returned by ShadeSurface (alpha in w)
    bool has_secondary;
    bool has_shadow;
    RayD new_ray;
    ShadowRayD sh_r;
    v3 base_color;     // primary-only AOVs
    v3 aov_normal;
    float aov_depth;
    bool wrote_aov;
};

// ensure_valid_reflection (ShadeRef.cpp:237-333, "taken from Cycles"): only normal-mapped surfaces reach it
RT_FN v3 ensure_valid_reflection(v3 Ng, v3 I, v3 N) {
    const v3 R = (2.0f * dot(N, I)) * N - I;
    const float threshold = fminf(0.9f * dot(Ng, I), 0.01f);
    if (dot(Ng, R) >= threshold) {
        return N;
    }
    const float NdotNg = dot(N, Ng);
    const v3 X = normalize(N - NdotNg * Ng);
    const float Ix = dot(I, X), Iz = dot(I, Ng);
    const float Ix2 = (Ix * Ix), Iz2 = (Iz * Iz);
    const float a = Ix2 + Iz2;
    const float b = safe_sqrt(Ix2 * (a - (threshold * threshold)));
    const float c = Iz * threshold + a;
    const float fac = 0.5f / a;
    const float N1_z2 = fac * (b + c), N2_z2 = fac * (-b + c);
    bool valid1 = (N1_z2 > 1e-5f) && (N1_z2 <= (1.0f + 1e-5f));
    bool valid2 = (N2_z2 > 1e-5f) && (N2_z2 <= (1.0f + 1e-5f));
    v2 N_new;
    if (valid1 && valid2) {
        const v2 N1 = v2{safe_sqrt(1.0f - N1_z2), safe_sqrt(N1_z2)};
        const v2 N2 = v2{safe_sqrt(1.0f - N2_z2), safe_sqrt(N2_z2)};
        const float R1 = 2 * (N1.x * Ix + N1.y * Iz) * N1.y - Iz;
        const float R2 = 2 * (N2.x * Ix + N2.y * Iz) * N2.y - Iz;
        valid1 = (R1 >= 1e-5f);
        valid2 = (R2 >= 1e-5f);
        if (valid1 && valid2) {
            N_new = (R1 < R2) ? N1 : N2;
        } else {
            N_new = (R1 > R2) ? N1 : N2;
        }
    } else if (valid1 || valid2) {
        const float Nz2 = valid1 ? N1_z2 : N2_z2;
        N_new = v2{safe_sqrt(1.0f - Nz2), safe_sqrt(Nz2)};
    } else {
        return Ng;
    }
    return N_new.x * X + N_new.y * Ng;
}

// Everything a material-node branch of ShadeSurface reads or writes.  The branches are separate (non-inlined) functions
// so the kernel's hot instruction footprint is the branch actually taken, not all five (see RT_FN in rt_math.cuh).
struct MatCtx {
    const PassSettings *ps;
    const RayD *ray;
    const ShadeScene *sc;
    const Hit *inter;
    Surface surf;
    LightSample ls;
    const Material *mat;
    const MeshInstance *mi;
    const Vertex *vtx1, *vtx2, *vtx3;
    RayD *new_ray;
    ShadowRayD *sh_r;
    v3 col;
    v3 I, ro, base_color, tint_color;
    float N_dot_L, roughness, mix_weight, mix_rand, regularize_alpha, ext_ior, base_color_lum;
    v2 rand_bsdf;
    bool use_mis, is_backfacing;
    int diff_d, spec_d, refr_d, total_d;
    uint32_t tri_index;
    uint32_t *tl_stack;
    float *tl_factors;
    // carried between the phases of shade_surface_{a,l,b}
    uint32_t rand_dim, rand_hash;
    float term_rand_y, cone_width;
    int iteration;
    float lambda; // ray-cone texture LOD term (ShadeRef.cpp:1279-1284)
    v2 tex_rand;
};

RT_FN void shade_node_diffuse(MatCtx &c) {
    const PassSettings &ps = *c.ps;
    const RayD &ray = *c.ray;
    const ShadeScene &sc = *c.sc;
    const Hit &inter = *c.inter;
    const Surface &surf = c.surf;
    const LightSample &ls = c.ls;
    const Material *mat = c.mat;
    const MeshInstance *mi = c.mi;
    const Vertex &v1 = *c.vtx1, &v2_ = *c.vtx2, &v3_ = *c.vtx3;
    RayD &new_ray = *c.new_ray;
    ShadowRayD &sh_r = *c.sh_r;
    v3 &col = c.col;
    const v3 I = c.I, ro = c.ro, base_color = c.base_color, tint_color = c.tint_color;
    const float N_dot_L = c.N_dot_L, roughness = c.roughness, mix_weight = c.mix_weight, mix_rand = c.mix_rand,
                regularize_alpha = c.regularize_alpha, ext_ior = c.ext_ior, base_color_lum = c.base_color_lum;
    const v2 rand_bsdf = c.rand_bsdf;
    const bool use_mis = c.use_mis, is_backfacing = c.is_backfacing;
    const int diff_d = c.diff_d, spec_d = c.spec_d, refr_d = c.refr_d, total_d = c.total_d;
    const uint32_t tri_index = c.tri_index;
    uint32_t *tl_stack = c.tl_stack;
    float *tl_factors = c.tl_factors;
    (void)ps; (void)ray; (void)sc; (void)inter; (void)surf; (void)ls; (void)mat; (void)mi; (void)v1; (void)v2_; (void)v3_;
    (void)new_ray; (void)sh_r; (void)col; (void)I; (void)ro; (void)base_color; (void)tint_color; (void)N_dot_L;
    (void)roughness; (void)mix_weight; (void)mix_rand; (void)regularize_alpha; (void)ext_ior; (void)base_color_lum;
    (void)rand_bsdf; (void)use_mis; (void)is_backfacing; (void)diff_d; (void)spec_d; (void)refr_d; (void)total_d;
    (void)tri_index; (void)tl_stack; (void)tl_factors;
    if (ls.pdf > 0.0f && (ls.ray_flags & (1u << RAY_DIFFUSE)) != 0 && N_dot_L > 0.0f) {
        // Evaluate_DiffuseNode :645-672
        const c4 diff_col = eval_oren_diffuse(-I, surf.N, ls.L, roughness, base_color);
        const float bsdf_pdf = diff_col.w;
        float mis_weight = 1.0f;
        if (use_mis && ls.area > 0.0f) {
            mis_weight = power_heuristic(ls.pdf, bsdf_pdf);
        }
        const v3 lcol = ls.col * v3{diff_col.x, diff_col.y, diff_col.z} * (mix_weight * mis_weight / ls.pdf);
        if (!ls.cast_shadow) {
            col += lcol;
        } else {
            sh_r.o = offset_ray(surf.P, surf.plane_N);
            sh_r.c = lcol;
        }
    }
    if (diff_d < ps.max_diff_depth && total_d < ps.max_total_depth) {
        // Sample_DiffuseNode :674-692
        v3 V;
        const c4 F = sample_oren_diffuse(surf.T, surf.B, surf.N, I, roughness, base_color, rand_bsdf, V);
        new_ray.depth = (uint32_t(RAY_DIFFUSE) << 28) | ((ray.depth & 0x0fffffffu) + pack_depth(1, 0, 0, 0));
        new_ray.o = offset_ray(surf.P, surf.plane_N);
        new_ray.d = V;
        new_ray.c = v3{F.x * mix_weight / F.w, F.y * mix_weight / F.w, F.z * mix_weight / F.w};
        new_ray.pdf = F.w;
        new_ray.cone_spread += kMaxConeSpreadInc;
    }
}

RT_FN void shade_node_glossy(MatCtx &c) {
    const PassSettings &ps = *c.ps;
    const RayD &ray = *c.ray;
    const ShadeScene &sc = *c.sc;
    const Hit &inter = *c.inter;
    const Surface &surf = c.surf;
    const LightSample &ls = c.ls;
    const Material *mat = c.mat;
    const MeshInstance *mi = c.mi;
    const Vertex &v1 = *c.vtx1, &v2_ = *c.vtx2, &v3_ = *c.vtx3;
    RayD &new_ray = *c.new_ray;
    ShadowRayD &sh_r = *c.sh_r;
    v3 &col = c.col;
    const v3 I = c.I, ro = c.ro, base_color = c.base_color, tint_color = c.tint_color;
    const float N_dot_L = c.N_dot_L, roughness = c.roughness, mix_weight = c.mix_weight, mix_rand = c.mix_rand,
                regularize_alpha = c.regularize_alpha, ext_ior = c.ext_ior, base_color_lum = c.base_color_lum;
    const v2 rand_bsdf = c.rand_bsdf;
    const bool use_mis = c.use_mis, is_backfacing = c.is_backfacing;
    const int diff_d = c.diff_d, spec_d = c.spec_d, refr_d = c.refr_d, total_d = c.total_d;
    const uint32_t tri_index = c.tri_index;
    uint32_t *tl_stack = c.tl_stack;
    float *tl_factors = c.tl_factors;
    (void)ps; (void)ray; (void)sc; (void)inter; (void)surf; (void)ls; (void)mat; (void)mi; (void)v1; (void)v2_; (void)v3_;
    (void)new_ray; (void)sh_r; (void)col; (void)I; (void)ro; (void)base_color; (void)tint_color; (void)N_dot_L;
    (void)roughness; (void)mix_weight; (void)mix_rand; (void)regularize_alpha; (void)ext_ior; (void)base_color_lum;
    (void)rand_bsdf; (void)use_mis; (void)is_backfacing; (void)diff_d; (void)spec_d; (void)refr_d; (void)total_d;
    (void)tri_index; (void)tl_stack; (void)tl_factors;
    const float specular = 0.5f;
    const float spec_ior = (2.0f / (1.0f - sqrtf(0.08f * specular))) - 1.0f;
    const float spec_F0 = fresnel_dielectric_cos(1.0f, spec_ior);
    if (ls.pdf > 0.0f && (ls.ray_flags & (1u << RAY_SPECULAR)) != 0 && N_dot_L > 0.0f) {
        // Evaluate_GlossyNode :694-730
        const v3 H = normalize(ls.L - I);
        const v3 view_dir_ts = tangent_from_world(surf.T, surf.B, surf.N, -I);
        const v3 light_dir_ts = tangent_from_world(surf.T, surf.B, surf.N, ls.L);
        const v3 sampled_normal_ts = tangent_from_world(surf.T, surf.B, surf.N, H);
        const v2 alpha = calc_alpha(roughness, 0.0f, regularize_alpha);
        if (!(alpha.x * alpha.y < 1e-7f)) {
            const c4 spec_col = eval_ggx_specular(view_dir_ts, sampled_normal_ts, light_dir_ts, alpha, spec_ior,
                                                  spec_F0, base_color, base_color);
            const float bsdf_pdf = spec_col.w;
            float mis_weight = 1.0f;
            if (use_mis && ls.area > 0.0f) {
                mis_weight = power_heuristic(ls.pdf, bsdf_pdf);
            }
            const v3 lcol = ls.col * v3{spec_col.x, spec_col.y, spec_col.z} * (mix_weight * mis_weight / ls.pdf);
            if (!ls.cast_shadow) {
                col += lcol;
            } else {
                sh_r.o = offset_ray(surf.P, surf.plane_N);
                sh_r.c = lcol;
            }
        }
    }
    if (spec_d < ps.max_spec_depth && total_d < ps.max_total_depth) {
        // Sample_GlossyNode :732-752
        const v2 alpha = calc_alpha(roughness, 0.0f, regularize_alpha);
        v3 V;
        const c4 F = sample_ggx_specular(surf.T, surf.B, surf.N, I, alpha, spec_ior, spec_F0, base_color,
                                         base_color, rand_bsdf, V);
        new_ray.depth = (uint32_t(RAY_SPECULAR) << 28) | ((ray.depth & 0x0fffffffu) + pack_depth(0, 1, 0, 0));
        new_ray.o = offset_ray(surf.P, surf.plane_N);
        new_ray.d = V;
        const float k = safe_div_pos(mix_weight, F.w);
        new_ray.c = v3{F.x * k, F.y * k, F.z * k};
        new_ray.pdf = F.w;
        new_ray.cone_spread += kMaxConeSpreadInc * fminf(alpha.x, alpha.y);
    }
}

RT_FN void shade_node_refractive(MatCtx &c) {
    const PassSettings &ps = *c.ps;
    const RayD &ray = *c.ray;
    const ShadeScene &sc = *c.sc;
    const Hit &inter = *c.inter;
    const Surface &surf = c.surf;
    const LightSample &ls = c.ls;
    const Material *mat = c.mat;
    const MeshInstance *mi = c.mi;
    const Vertex &v1 = *c.vtx1, &v2_ = *c.vtx2, &v3_ = *c.vtx3;
    RayD &new_ray = *c.new_ray;
    ShadowRayD &sh_r = *c.sh_r;
    v3 &col = c.col;
    const v3 I = c.I, ro = c.ro, base_color = c.base_color, tint_color = c.tint_color;
    const float N_dot_L = c.N_dot_L, roughness = c.roughness, mix_weight = c.mix_weight, mix_rand = c.mix_rand,
                regularize_alpha = c.regularize_alpha, ext_ior = c.ext_ior, base_color_lum = c.base_color_lum;
    const v2 rand_bsdf = c.rand_bsdf;
    const bool use_mis = c.use_mis, is_backfacing = c.is_backfacing;
    const int diff_d = c.diff_d, spec_d = c.spec_d, refr_d = c.refr_d, total_d = c.total_d;
    const uint32_t tri_index = c.tri_index;
    uint32_t *tl_stack = c.tl_stack;
    float *tl_factors = c.tl_factors;
    (void)ps; (void)ray; (void)sc; (void)inter; (void)surf; (void)ls; (void)mat; (void)mi; (void)v1; (void)v2_; (void)v3_;
    (void)new_ray; (void)sh_r; (void)col; (void)I; (void)ro; (void)base_color; (void)tint_color; (void)N_dot_L;
    (void)roughness; (void)mix_weight; (void)mix_rand; (void)regularize_alpha; (void)ext_ior; (void)base_color_lum;
    (void)rand_bsdf; (void)use_mis; (void)is_backfacing; (void)diff_d; (void)spec_d; (void)refr_d; (void)total_d;
    (void)tri_index; (void)tl_stack; (void)tl_factors;
    if (ls.pdf > 0.0f && (ls.ray_flags & (1u << RAY_REFR)) != 0 && N_dot_L < 0.0f) {
        // Evaluate_RefractiveNode :754-786
        const float eta = is_backfacing ? (mat->ior / ext_ior) : (ext_ior / mat->ior);
        const v3 H = normalize(ls.L - I * eta);
        const v3 view_dir_ts = tangent_from_world(surf.T, surf.B, surf.N, -I);
        const v3 light_dir_ts = tangent_from_world(surf.T, surf.B, surf.N, ls.L);
        const v3 sampled_normal_ts = tangent_from_world(surf.T, surf.B, surf.N, H);
        const c4 refr_col = eval_ggx_refraction(view_dir_ts, sampled_normal_ts, light_dir_ts,
                                                calc_alpha(roughness, 0.0f, regularize_alpha), eta, base_color);
        const float bsdf_pdf = refr_col.w;
        float mis_weight = 1.0f;
        if (use_mis && ls.area > 0.0f) {
            mis_weight = power_heuristic(ls.pdf, bsdf_pdf);
        }
        const v3 lcol = ls.col * v3{refr_col.x, refr_col.y, refr_col.z} * (mix_weight * mis_weight / ls.pdf);
        if (!ls.cast_shadow) {
            col += lcol;
        } else {
            sh_r.o = offset_ray(surf.P, -surf.plane_N);
            sh_r.c = lcol;
        }
    }
    if (refr_d < ps.max_refr_depth && total_d < ps.max_total_depth) {
        // Sample_RefractiveNode :788-809
        const v2 alpha = calc_alpha(roughness, 0.0f, regularize_alpha);
        const float eta = is_backfacing ? (mat->ior / ext_ior) : (ext_ior / mat->ior);
        v3 V = v3{0.0f, 0.0f, 0.0f};
        const c4 F = sample_ggx_refraction(surf.T, surf.B, surf.N, I, alpha, eta, base_color, rand_bsdf, V);
        new_ray.depth = (uint32_t(RAY_REFR) << 28) | ((ray.depth & 0x0fffffffu) + pack_depth(0, 0, 1, 0));
        const float k = safe_div_pos(mix_weight, F.w);
        new_ray.c = v3{F.x * k, F.y * k, F.z * k};
        new_ray.pdf = F.w;
        if (!is_backfacing) {
            push_ior_stack(new_ray.ior, mat->ior);
        } else {
            pop_ior_stack(new_ray.ior);
        }
        new_ray.o = offset_ray(surf.P, -surf.plane_N);
        new_ray.d = V;
        new_ray.cone_spread += kMaxConeSpreadInc * fminf(alpha.x, alpha.y);
    }
}

RT_FN void shade_node_emissive(MatCtx &c) {
    const PassSettings &ps = *c.ps;
    const RayD &ray = *c.ray;
    const ShadeScene &sc = *c.sc;
    const Hit &inter = *c.inter;
    const Surface &surf = c.surf;
    const LightSample &ls = c.ls;
    const Material *mat = c.mat;
    const MeshInstance *mi = c.mi;
    const Vertex &v1 = *c.vtx1, &v2_ = *c.vtx2, &v3_ = *c.vtx3;
    RayD &new_ray = *c.new_ray;
    ShadowRayD &sh_r = *c.sh_r;
    v3 &col = c.col;
    const v3 I = c.I, ro = c.ro, base_color = c.base_color, tint_color = c.tint_color;
    const float N_dot_L = c.N_dot_L, roughness = c.roughness, mix_weight = c.mix_weight, mix_rand = c.mix_rand,
                regularize_alpha = c.regularize_alpha, ext_ior = c.ext_ior, base_color_lum = c.base_color_lum;
    const v2 rand_bsdf = c.rand_bsdf;
    const bool use_mis = c.use_mis, is_backfacing = c.is_backfacing;
    const int diff_d = c.diff_d, spec_d = c.spec_d, refr_d = c.refr_d, total_d = c.total_d;
    const uint32_t tri_index = c.tri_index;
    uint32_t *tl_stack = c.tl_stack;
    float *tl_factors = c.tl_factors;
    (void)ps; (void)ray; (void)sc; (void)inter; (void)surf; (void)ls; (void)mat; (void)mi; (void)v1; (void)v2_; (void)v3_;
    (void)new_ray; (void)sh_r; (void)col; (void)I; (void)ro; (void)base_color; (void)tint_color; (void)N_dot_L;
    (void)roughness; (void)mix_weight; (void)mix_rand; (void)regularize_alpha; (void)ext_ior; (void)base_color_lum;
    (void)rand_bsdf; (void)use_mis; (void)is_backfacing; (void)diff_d; (void)spec_d; (void)refr_d; (void)total_d;
    (void)tri_index; (void)tl_stack; (void)tl_factors;
    float mis_weight = 1.0f;
    if ((ray.depth & 0x00ffffffu) != 0 && (mat->flags & kMatFlagImpSample)) {
        const float pdf_factor = eval_tri_light_factor(sc.lights, surf.P, ro, tri_index, tl_stack, tl_factors);
        const v3 p1 = mk3(v1.p), p2 = mk3(v2_.p), p3 = mk3(v3_.p);
        float light_forward_len;
        const v3 light_forward =
            normalize_len(transform_direction(cross(p2 - p1, p3 - p1), mi->xform), light_forward_len);
        const float tri_area = 0.5f * light_forward_len;
        const float cos_theta = fabsf(dot(I, light_forward));
        if (cos_theta > 0.0f) {
            float light_pdf = 0.0f;
            {
                const v3 P = transform_point(ro, mi->inv_xform);
                light_pdf = sample_spherical_triangle(P, p1, p2, p3, v2{0.0f, 0.0f}, nullptr) / pdf_factor;
            }
            if (light_pdf == 0.0f) {
                light_pdf = (inter.t * inter.t) / (tri_area * cos_theta * pdf_factor);
            }
            mis_weight = power_heuristic(ray.pdf, light_pdf);
        }
    }
    col += mix_weight * mis_weight * mat->tangent_rotation_or_strength * base_color;
}

RT_FN void shade_node_principled(const bool tex_on, MatCtx &c) {
    const PassSettings &ps = *c.ps;
    const RayD &ray = *c.ray;
    const ShadeScene &sc = *c.sc;
    const Hit &inter = *c.inter;
    const Surface &surf = c.surf;
    const LightSample &ls = c.ls;
    const Material *mat = c.mat;
    const MeshInstance *mi = c.mi;
    const Vertex &v1 = *c.vtx1, &v2_ = *c.vtx2, &v3_ = *c.vtx3;
    RayD &new_ray = *c.new_ray;
    ShadowRayD &sh_r = *c.sh_r;
    v3 &col = c.col;
    const v3 I = c.I, ro = c.ro, base_color = c.base_color, tint_color = c.tint_color;
    const float N_dot_L = c.N_dot_L, roughness = c.roughness, mix_weight = c.mix_weight, mix_rand = c.mix_rand,
                regularize_alpha = c.regularize_alpha, ext_ior = c.ext_ior, base_color_lum = c.base_color_lum;
    const v2 rand_bsdf = c.rand_bsdf;
    const bool use_mis = c.use_mis, is_backfacing = c.is_backfacing;
    const int diff_d = c.diff_d, spec_d = c.spec_d, refr_d = c.refr_d, total_d = c.total_d;
    const uint32_t tri_index = c.tri_index;
    uint32_t *tl_stack = c.tl_stack;
    float *tl_factors = c.tl_factors;
    (void)ps; (void)ray; (void)sc; (void)inter; (void)surf; (void)ls; (void)mat; (void)mi; (void)v1; (void)v2_; (void)v3_;
    (void)new_ray; (void)sh_r; (void)col; (void)I; (void)ro; (void)base_color; (void)tint_color; (void)N_dot_L;
    (void)roughness; (void)mix_weight; (void)mix_rand; (void)regularize_alpha; (void)ext_ior; (void)base_color_lum;
    (void)rand_bsdf; (void)use_mis; (void)is_backfacing; (void)diff_d; (void)spec_d; (void)refr_d; (void)total_d;
    (void)tri_index; (void)tl_stack; (void)tl_factors;
    float metallic = unorm16(mat->metallic_unorm);
    if (tex_on && mat->textures[kTexMetallic] != kTexInvalid) { // ShadeRef.cpp:1540-1545 (no colour-space conversion)
        const uint32_t metallic_tex = mat->textures[kTexMetallic];
        metallic *= tex_unpack(tex_sample_bytes(sc.tex, metallic_tex, surf.uvs, tex_lod(sc.tex, metallic_tex, c.lambda), c.tex_rand)).x;
    }
    float specular = unorm16(mat->specular_unorm);
    if (tex_on && mat->textures[kTexSpecular] != kTexInvalid) { // ShadeRef.cpp:1547-1557
        const uint32_t specular_tex = mat->textures[kTexSpecular];
        specular *= tex_sample_color(sc.tex, specular_tex, surf.uvs, tex_lod(sc.tex, specular_tex, c.lambda), c.tex_rand).x;
    }
    const float specular_tint = unorm16(mat->specular_tint_unorm);
    const float transmission = unorm16(mat->transmission_unorm);
    const float clearcoat = unorm16(mat->clearcoat_unorm);
    const float clearcoat_roughness = unorm16(mat->clearcoat_roughness_unorm);
    const float sheen = 2.0f * unorm16(mat->sheen_unorm);
    const float sheen_tint = unorm16(mat->sheen_tint_unorm);

    const v3 one3 = v3{1.0f, 1.0f, 1.0f};
    const v3 diff_base_color = base_color;
    const v3 diff_sheen_color = sheen * mix3(one3, tint_color, sheen_tint);
    const float diff_roughness = roughness;

    SpecParams spec;
    spec.tmp_col = mix3(one3, tint_color, specular_tint);
    spec.tmp_col = mix3(specular * 0.08f * spec.tmp_col, base_color, metallic);
    spec.roughness = roughness;
    spec.ior = (2.0f / (1.0f - sqrtf(0.08f * specular))) - 1.0f;
    spec.F0 = fresnel_dielectric_cos(1.0f, spec.ior);
    spec.anisotropy = unorm16(mat->anisotropic_unorm);

    CoatParams coat;
    coat.roughness = clearcoat_roughness;
    coat.ior = (2.0f / (1.0f - sqrtf(0.08f * clearcoat))) - 1.0f;
    coat.F0 = fresnel_dielectric_cos(1.0f, coat.ior);

    TransParams trans;
    trans.roughness = 1.0f - (1.0f - roughness) * (1.0f - unorm16(mat->transmission_roughness_unorm));
    trans.int_ior = mat->ior;
    trans.eta = is_backfacing ? (mat->ior / ext_ior) : (ext_ior / mat->ior);
    trans.fresnel = fresnel_dielectric_cos(dot(I, surf.N), 1.0f / trans.eta);
    trans.backfacing = is_backfacing;

    const float FN = (fresnel_dielectric_cos(dot(I, surf.N), spec.ior) - spec.F0) / (1.0f - spec.F0);
    const v3 approx_spec_col = mix3(spec.tmp_col, one3, FN);
    const float spec_color_lum = lum(approx_spec_col);

    const LobeWeights lobe = get_lobe_weights(mixf(base_color_lum, 1.0f, sheen), spec_color_lum, specular, metallic,
                                              transmission, clearcoat);

    if (ls.pdf > 0.0f) {
        // Evaluate_PrincipledNode :811-903
        v3 lcol = v3{0.0f, 0.0f, 0.0f};
        float bsdf_pdf = 0.0f;
        if (lobe.diffuse > 0.0f && N_dot_L > 0.0f && (ls.ray_flags & (1u << RAY_DIFFUSE)) != 0) {
            const c4 dc = eval_principled_diffuse(-I, surf.N, ls.L, diff_roughness, diff_base_color, diff_sheen_color);
            bsdf_pdf += lobe.diffuse * dc.w;
            v3 diff_col = v3{dc.x, dc.y, dc.z};
            diff_col *= (1.0f - metallic) * (1.0f - transmission);
            lcol += ls.col * N_dot_L * diff_col / (kPi * ls.pdf);
        }
        v3 H;
        if (N_dot_L > 0.0f) {
            H = normalize(ls.L - I);
        } else {
            H = normalize(ls.L - I * trans.eta);
        }
        const v3 view_dir_ts = tangent_from_world(surf.T, surf.B, surf.N, -I);
        const v3 light_dir_ts = tangent_from_world(surf.T, surf.B, surf.N, ls.L);
        const v3 sampled_normal_ts = tangent_from_world(surf.T, surf.B, surf.N, H);

        const v2 spec_alpha = calc_alpha(spec.roughness, spec.anisotropy, regularize_alpha);
        if (lobe.specular > 0.0f && spec_alpha.x * spec_alpha.y >= 1e-7f && N_dot_L > 0.0f &&
            (ls.ray_flags & (1u << RAY_SPECULAR)) != 0) {
            const c4 sc4 = eval_ggx_specular(view_dir_ts, sampled_normal_ts, light_dir_ts, spec_alpha, spec.ior,
                                             spec.F0, spec.tmp_col, one3);
            bsdf_pdf += lobe.specular * sc4.w;
            lcol += ls.col * v3{sc4.x, sc4.y, sc4.z} / ls.pdf;
        }
        const v2 coat_alpha = calc_alpha(coat.roughness, 0.0f, regularize_alpha);
        if (lobe.clearcoat > 0.0f && coat_alpha.x * coat_alpha.y >= 1e-7f && N_dot_L > 0.0f &&
            (ls.ray_flags & (1u << RAY_SPECULAR)) != 0) {
            const c4 cc = eval_clearcoat(view_dir_ts, sampled_normal_ts, light_dir_ts, coat_alpha.x, coat.ior, coat.F0);
            bsdf_pdf += lobe.clearcoat * cc.w;
            lcol += 0.25f * ls.col * v3{cc.x, cc.y, cc.z} / ls.pdf;
        }
        if (lobe.refraction > 0.0f) {
            const v2 refr_spec_alpha = calc_alpha(spec.roughness, 0.0f, regularize_alpha);
            if (trans.fresnel != 0.0f && refr_spec_alpha.x * refr_spec_alpha.y >= 1e-7f && N_dot_L > 0.0f &&
                (ls.ray_flags & (1u << RAY_SPECULAR)) != 0) {
                const c4 sc4 = eval_ggx_specular(view_dir_ts, sampled_normal_ts, light_dir_ts, refr_spec_alpha,
                                                 1.0f, 0.0f, one3, one3);
                bsdf_pdf += lobe.refraction * trans.fresnel * sc4.w;
                lcol += ls.col * v3{sc4.x, sc4.y, sc4.z} * (trans.fresnel / ls.pdf);
            }
            const v2 refr_trans_alpha = calc_alpha(trans.roughness, 0.0f, regularize_alpha);
            if (trans.fresnel != 1.0f && refr_trans_alpha.x * refr_trans_alpha.y >= 1e-7f && N_dot_L < 0.0f &&
                (ls.ray_flags & (1u << RAY_REFR)) != 0) {
                const c4 rc = eval_ggx_refraction(view_dir_ts, sampled_normal_ts, light_dir_ts, refr_trans_alpha,
                                                  trans.eta, diff_base_color);
                bsdf_pdf += lobe.refraction * (1.0f - trans.fresnel) * rc.w;
                lcol += ls.col * v3{rc.x, rc.y, rc.z} * ((1.0f - trans.fresnel) / ls.pdf);
            }
        }
        float mis_weight = 1.0f;
        if (use_mis && ls.area > 0.0f) {
            mis_weight = power_heuristic(ls.pdf, bsdf_pdf);
        }
        lcol *= mix_weight * mis_weight;
        if (!ls.cast_shadow) {
            col += lcol;
        } else {
            sh_r.o = offset_ray(surf.P, N_dot_L < 0.0f ? -surf.plane_N : surf.plane_N);
            sh_r.c = lcol;
        }
    }

    { // Sample_PrincipledNode :905-1028
        const int ptotal = diff_d + spec_d + refr_d;
        if (mix_rand < lobe.diffuse) {
            if (diff_d < ps.max_diff_depth && ptotal < ps.max_total_depth) {
                v3 V;
                const c4 F4 = sample_principled_diffuse(surf.T, surf.B, surf.N, I, diff_roughness, diff_base_color,
                                                        diff_sheen_color, rand_bsdf, V);
                const float pdf = F4.w;
                v3 F = v3{F4.x, F4.y, F4.z};
                F *= (1.0f - metallic) * (1.0f - transmission);
                new_ray.depth = (uint32_t(RAY_DIFFUSE) << 28) | ((ray.depth & 0x0fffffffu) + pack_depth(1, 0, 0, 0));
                new_ray.o = offset_ray(surf.P, surf.plane_N);
                new_ray.d = V;
                const float k = safe_div_pos(mix_weight, lobe.diffuse);
                new_ray.c = v3{F.x * k, F.y * k, F.z * k};
                new_ray.pdf = pdf;
                new_ray.cone_spread += kMaxConeSpreadInc;
            }
        } else if (mix_rand < lobe.diffuse + lobe.specular) {
            if (spec_d < ps.max_spec_depth && ptotal < ps.max_total_depth) {
                const v2 alpha = calc_alpha(spec.roughness, spec.anisotropy, regularize_alpha);
                v3 V;
                const c4 F = sample_ggx_specular(surf.T, surf.B, surf.N, I, alpha, spec.ior, spec.F0, spec.tmp_col,
                                                 one3, rand_bsdf, V);
                const float pdf = F.w * lobe.specular;
                new_ray.depth = (uint32_t(RAY_SPECULAR) << 28) | ((ray.depth & 0x0fffffffu) + pack_depth(0, 1, 0, 0));
                const float k = safe_div_pos(mix_weight, pdf);
                new_ray.c = v3{F.x * k, F.y * k, F.z * k};
                new_ray.pdf = pdf;
                new_ray.o = offset_ray(surf.P, surf.plane_N);
                new_ray.d = V;
                new_ray.cone_spread += kMaxConeSpreadInc * fminf(alpha.x, alpha.y);
            }
        } else if (mix_rand < lobe.diffuse + lobe.specular + lobe.clearcoat) {
            if (spec_d < ps.max_spec_depth && ptotal < ps.max_total_depth) {
                const float alpha = calc_alpha(coat.roughness, 0.0f, regularize_alpha).x;
                v3 V;
                const c4 F = sample_clearcoat(surf.T, surf.B, surf.N, I, alpha, coat.ior, coat.F0, rand_bsdf, V);
                const float pdf = F.w * lobe.clearcoat;
                new_ray.depth = (uint32_t(RAY_SPECULAR) << 28) | ((ray.depth & 0x0fffffffu) + pack_depth(0, 1, 0, 0));
                const float k = safe_div_pos(mix_weight, pdf);
                new_ray.c = v3{0.25f * F.x * k, 0.25f * F.y * k, 0.25f * F.z * k};
                new_ray.pdf = pdf;
                new_ray.o = offset_ray(surf.P, surf.plane_N);
                new_ray.d = V;
                new_ray.cone_spread += kMaxConeSpreadInc * alpha;
            }
        } else {
            float mr = mix_rand;
            mr -= lobe.diffuse + lobe.specular + lobe.clearcoat;
            mr = safe_div_pos(mr, lobe.refraction);
            if (((mr >= trans.fresnel && refr_d < ps.max_refr_depth) || (mr < trans.fresnel && spec_d < ps.max_spec_depth)) &&
                ptotal < ps.max_total_depth) {
                c4 F;
                v3 V = v3{0.0f, 0.0f, 0.0f};
                if (mr < trans.fresnel) {
                    const v2 alpha = calc_alpha(spec.roughness, 0.0f, regularize_alpha);
                    F = sample_ggx_specular(surf.T, surf.B, surf.N, I, alpha, 1.0f, 0.0f, one3, one3, rand_bsdf, V);
                    new_ray.depth = (uint32_t(RAY_SPECULAR) << 28) | ((ray.depth & 0x0fffffffu) + pack_depth(0, 1, 0, 0));
                    new_ray.o = offset_ray(surf.P, surf.plane_N);
                    new_ray.cone_spread += kMaxConeSpreadInc * fminf(alpha.x, alpha.y);
                } else {
                    const v2 alpha = calc_alpha(trans.roughness, 0.0f, regularize_alpha);
                    F = sample_ggx_refraction(surf.T, surf.B, surf.N, I, alpha, trans.eta, diff_base_color, rand_bsdf, V);
                    new_ray.depth = (uint32_t(RAY_REFR) << 28) | ((ray.depth & 0x0fffffffu) + pack_depth(0, 0, 1, 0));
                    new_ray.o = offset_ray(surf.P, -surf.plane_N);
                    new_ray.cone_spread += kMaxConeSpreadInc * fminf(alpha.x, alpha.y);
                    if (!trans.backfacing) {
                        push_ior_stack(new_ray.ior, trans.int_ior);
                    } else {
                        pop_ior_stack(new_ray.ior);
                    }
                }
                const float pdf = F.w * lobe.refraction;
                const float k = safe_div_pos(mix_weight, pdf);
                new_ray.c = v3{F.x * k, F.y * k, F.z * k};
                new_ray.pdf = pdf;
                new_ray.d = V;
            }
        }
    }
}

// One invocation of Ref::ShadeSurface.  `limits` = {direct, indirect} clamp limits (FLT_MAX when clamping is off).
// ShadeSurface (ShadeRef.cpp:1173-1652) in three phases so that the kernel can keep the warps of a block in step between
// them (RT_SHADE_SYNC):  a = miss / light hit / surface frame + mix resolution,  l = light sampling (NEE),
// b = the material node + path continuation.  `c` carries everything from one phase to the next.
// Phase a returns false when the ray is finished (out.col is final).
// `tex_on` is a compile-time constant at every call site (k_shade<PRIMARY, TEX>): untextured scenes run kernels from
// which every texture branch has been folded away.
RT_DEV bool shade_surface_a(const bool tex_on, const PassSettings &ps, float limit0, const Hit &inter, const RayD &ray,
                            uint32_t rand_seed, int iteration, const ShadeScene &sc, uint32_t *tl_stack,
                            float *tl_factors, MatCtx &c, ShadeOut &out) {
    out.has_secondary = out.has_shadow = false;
    out.wrote_aov = false;
    out.base_color = v3{0.0f, 0.0f, 0.0f};
    out.aov_normal = v3{0.0f, 0.0f, 0.0f};
    out.aov_depth = 0.0f;

    const v3 I = ray.d;
    const v3 ro = ray.o;

    const uint32_t px_hash = hash_u32(ray.xy);
    const uint32_t rand_hash = hash_combine(px_hash, rand_seed);
    const uint32_t rand_dim = kRandDimBase + total_depth(ray.depth) * kRandDimBounce;

    if (inter.v < 0.0f) {
        // miss: environment (constant colour; Evaluate_EnvColor :1030-1066 without an env map / quad-tree)
        const float pdf_factor =
            (total_depth(ray.depth) < ps.max_total_depth) ? safe_div_pos(1.0f, inter.u) : -1.0f;
        c4 env_col = c4{1.0f, 1.0f, 1.0f, 1.0f};
        const SceneEnv &env = sc.lights.env;
        const uint32_t env_map = is_indirect(ray.depth) ? env.env_map : env.back_map;
        const float env_map_rotation = is_indirect(ray.depth) ? env.env_map_rotation : env.back_map_rotation;
        if (tex_on && env_map != kTexInvalid) {
            const v2 tex_rand = rand2d(rand_dim + kRandDimTex, rand_hash, iteration - 1, sc.rand_seq);
            const v3 m = sample_latlong_rgbe(sc.tex, env_map, I, env_map_rotation, tex_rand);
            env_col = c4{m.x, m.y, m.z, 1.0f};
        }
        if (sc.lights.env_light_index != 0xffffffffu && pdf_factor >= 0.0f && is_indirect(ray.depth)) {
            const float light_pdf = (tex_on && env.qtree_levels != 0)
                                        ? safe_div_pos(evaluate_env_qtree(env, env_map_rotation, I), pdf_factor)
                                        : safe_div_pos(0.5f, kPi * pdf_factor);
            const float bsdf_pdf = ray.pdf;
            const float mis_weight = power_heuristic(bsdf_pdf, light_pdf);
            env_col.x *= mis_weight;
            env_col.y *= mis_weight;
            env_col.z *= mis_weight;
            env_col.w *= mis_weight;
        }
        const float *ec = is_indirect(ray.depth) ? sc.lights.env_col : sc.lights.back_col;
        env_col.x *= ec[0];
        env_col.y *= ec[1];
        env_col.z *= ec[2];
        env_col.w = 1.0f;
        env_col.x *= ray.c.x;
        env_col.y *= ray.c.y;
        env_col.z *= ray.c.z;
        env_col.w *= 0.0f;
        const float sum = ((env_col.x + env_col.y) + env_col.z) + env_col.w;
        if (sum > limit0) {
            const float k = limit0 / sum;
            env_col.x *= k;
            env_col.y *= k;
            env_col.z *= k;
            env_col.w *= k;
        }
        out.col = env_col;
        return false;
    }

    Surface &surf = c.surf; // the surface and the light sample are built in place in the context the node functions read
    surf.P = ro + inter.t * I;

    if (inter.obj < 0) { // analytic light hit: Evaluate_LightColor :1068-1172
        const Light &l = sc.lights.lights[-inter.obj - 1];
        const float pdf_factor = 1.0f / inter.u;
        v3 lcol = mk3(l.col);
        if (l_sky_portal(l)) {
            v3 env_col = mk3(sc.lights.env_col);
            if (tex_on && sc.lights.env.env_map != kTexInvalid) {
                const v2 tex_rand = rand2d(rand_dim + kRandDimTex, rand_hash, iteration - 1, sc.rand_seq);
                env_col *= sample_latlong_rgbe(sc.tex, sc.lights.env.env_map, I, sc.lights.env.env_map_rotation, tex_rand);
            }
            lcol *= env_col;
        }
        const int type = l_type(l);
        if (type == LIGHT_SPHERE) {
            const v3 light_pos = mk3(&l.p[0]);
            const float radius = l.p[7];
            float d;
            const v3 disk_normal = normalize_len(light_pos - ro, d);
            if (d > radius) {
                const float temp = sqrtf(d * d - radius * radius);
                const float disk_radius = (temp * radius) / d;
                float disk_dist = dot(ro, disk_normal) - dot(light_pos, disk_normal);
                const float sampled_area = kPi * disk_radius * disk_radius;
                const float cos_theta = dot(I, disk_normal);
                disk_dist /= cos_theta;
                const float light_pdf = (disk_dist * disk_dist) / (sampled_area * cos_theta * pdf_factor);
                const float mis_weight = power_heuristic(ray.pdf, light_pdf);
                lcol *= mis_weight;
                const float spot = l.p[8], blend = l.p[9];
                if (spot > 0.0f && blend > 0.0f) {
                    const float _dot = -dot(I, mk3(&l.p[4]));
                    const float _angle = libm_acosf(saturatef(_dot));
                    lcol *= saturatef((spot - _angle) / blend);
                }
            }
        } else if (type == LIGHT_DIR) {
            const float radius = l.p[4];
            const float light_area = kPi * radius * radius;
            const float cos_theta = dot(I, mk3(&l.p[0]));
            const float light_pdf = 1.0f / (light_area * cos_theta * pdf_factor);
            lcol *= power_heuristic(ray.pdf, light_pdf);
        } else if (type == LIGHT_RECT) {
            const v3 light_pos = mk3(&l.p[0]);
            const v3 light_u = mk3(&l.p[4]), light_v = mk3(&l.p[8]);
            float light_pdf = sample_spherical_rectangle(ro, light_pos, light_u, light_v, v2{0.0f, 0.0f}, nullptr) / pdf_factor;
            if (light_pdf == 0.0f) {
                const v3 light_forward = normalize(cross(light_u, light_v));
                const float light_area = l.p[3];
                const float cos_theta = dot(I, light_forward);
                light_pdf = (inter.t * inter.t) / (light_area * cos_theta * pdf_factor);
            }
            lcol *= power_heuristic(ray.pdf, light_pdf);
        } else if (type == LIGHT_DISK) {
            const v3 light_u = mk3(&l.p[4]), light_v = mk3(&l.p[8]);
            const v3 light_forward = normalize(cross(light_u, light_v));
            const float light_area = l.p[3];
            const float cos_theta = dot(I, light_forward);
            const float light_pdf = (inter.t * inter.t) / (light_area * cos_theta * pdf_factor);
            lcol *= power_heuristic(ray.pdf, light_pdf);
        } else if (type == LIGHT_LINE) {
            const v3 light_dir = mk3(&l.p[8]);
            const float light_area = l.p[3];
            const float cos_theta = 1.0f - fabsf(dot(I, light_dir));
            const float light_pdf = (inter.t * inter.t) / (light_area * cos_theta * pdf_factor);
            lcol *= power_heuristic(ray.pdf, light_pdf);
        }
        lcol *= ray.c;
        const float sum = ((lcol.x + lcol.y) + lcol.z) + 0.0f;
        if (sum > limit0) {
            lcol *= (limit0 / sum);
        }
        out.col = c4{lcol.x, lcol.y, lcol.z, 1.0f};
        return false;
    }

    const bool is_backfacing = (inter.prim < 0);
    const uint32_t tri_index = is_backfacing ? uint32_t(-inter.prim - 1) : uint32_t(inter.prim);

    const TriMat tm = sc.geo.tri_materials[tri_index];
    const Material *mat = &sc.surf.materials[tm.front_mi & kMatIndexBits];
    const MeshInstance *mi = &sc.geo.instances[inter.obj];

    const Vertex &v1 = sc.surf.vertices[sc.surf.vtx_indices[tri_index * 3 + 0]];
    const Vertex &v2_ = sc.surf.vertices[sc.surf.vtx_indices[tri_index * 3 + 1]];
    const Vertex &v3_ = sc.surf.vertices[sc.surf.vtx_indices[tri_index * 3 + 2]];

    const float w = 1.0f - inter.u - inter.v;
    surf.N = normalize(mk3(v1.n) * w + mk3(v2_.n) * inter.u + mk3(v3_.n) * inter.v);
    surf.uvs = v2{v1.t[0] * w + v2_.t[0] * inter.u + v3_.t[0] * inter.v, v1.t[1] * w + v2_.t[1] * inter.u + v3_.t[1] * inter.v};

    float pa;
    // fvec4{v.p} loads 4 floats (p.xyz, n.x); the 4th lane of the cross product is set to 0 by cross()
    surf.plane_N = normalize_len(cross(mk3(v2_.p) - mk3(v1.p), mk3(v3_.p) - mk3(v1.p)), pa);

    surf.B = mk3(v1.b) * w + mk3(v2_.b) * inter.u + mk3(v3_.b) * inter.v;
    surf.T = cross(surf.B, surf.N);

    if (is_backfacing) {
        if (tm.back_mi == 0xffff) {
            out.col = c4{0.0f, 0.0f, 0.0f, 0.0f};
            return false;
        } else {
            mat = &sc.surf.materials[tm.back_mi & kMatIndexBits];
            surf.plane_N = -surf.plane_N;
            surf.N = -surf.N;
            surf.B = -surf.B;
            surf.T = -surf.T;
        }
    }

    surf.plane_N = transform_normal(surf.plane_N, mi->inv_xform);
    surf.N = transform_normal(surf.N, mi->inv_xform);
    surf.B = transform_normal(surf.B, mi->inv_xform);
    surf.T = transform_normal(surf.T, mi->inv_xform);

    surf.plane_N = safe_normalize(surf.plane_N);
    surf.N = safe_normalize(surf.N);
    surf.B = safe_normalize(surf.B);
    surf.T = safe_normalize(surf.T);

    const float cone_width = ray.cone_width + ray.cone_spread * inter.t;
    // texture LOD term and jitter: only consumed by texture fetches (pure functions of the inputs, so skipping them for
    // untextured scenes changes nothing)
    const bool has_tex = tex_on;
    float lambda = 0.0f;
    v2 tex_rand = v2{0.0f, 0.0f};
    if (has_tex) {
        const float ta = fabsf((v2_.t[0] - v1.t[0]) * (v3_.t[1] - v1.t[1]) - (v3_.t[0] - v1.t[0]) * (v2_.t[1] - v1.t[1]));
        lambda = 0.5f * fast_log2(ta / pa);
        lambda += fast_log2(cone_width);
        tex_rand = rand2d(rand_dim + kRandDimTex, rand_hash, iteration - 1, sc.rand_seq);
    }

    const float ext_ior = peek_ior_stack(ray.ior, is_backfacing);

    v3 col = v3{0.0f, 0.0f, 0.0f};

    const int diff_d = diff_depth(ray.depth), spec_d = spec_depth(ray.depth), refr_d = refr_depth(ray.depth);
    const int total_d = diff_d + spec_d + refr_d; // transparency depth is not accounted here

    const v2 mix_term_rand = rand2d(rand_dim + kRandDimBsdfPick, rand_hash, iteration - 1, sc.rand_seq);

    float mix_rand = mix_term_rand.x;
    float mix_weight = 1.0f;

    // resolve mix material
    while (mat->type == NODE_MIX) {
        float mix_val = mat->tangent_rotation_or_strength;
        const uint32_t mix_texture = mat->textures[kTexBase];
        if (tex_on && mix_texture != kTexInvalid) {
            mix_val *= tex_sample_color(sc.tex, mix_texture, surf.uvs, 0, tex_rand, true).x;
        }
        const float eta = is_backfacing ? safe_div_pos(ext_ior, mat->ior) : safe_div_pos(mat->ior, ext_ior);
        const float RR = mat->ior != 0.0f ? fresnel_dielectric_cos(dot(I, surf.N), eta) : 1.0f;
        mix_val *= saturatef(RR);
        if (mix_rand > mix_val) {
            mix_weight *= (mat->flags & kMatFlagMixAdd) ? 1.0f / (1.0f - mix_val) : 1.0f;
            mat = &sc.surf.materials[mat->textures[kMixMat1]];
            mix_rand = safe_div_pos(mix_rand - mix_val, 1.0f - mix_val);
        } else {
            mix_weight *= (mat->flags & kMatFlagMixAdd) ? 1.0f / mix_val : 1.0f;
            mat = &sc.surf.materials[mat->textures[kMixMat2]];
            mix_rand = safe_div_pos(mix_rand, mix_val);
        }
    }

    // apply normal map (ShadeRef.cpp:1335-1349)
    if (tex_on && mat->textures[kTexNormals] != kTexInvalid) {
        const uint32_t nh = mat->textures[kTexNormals];
        const c4 nc = tex_unpack(tex_sample_bytes(sc.tex, nh, surf.uvs, 0, tex_rand));
        const float nx = nc.x * 2.0f - 1.0f, ny = nc.y * 2.0f - 1.0f;
        float nz = 1.0f;
        if (nh & kTexReconstructZBit) {
            nz = safe_sqrt(1.0f - nx * nx - ny * ny);
        }
        const v3 in_normal = surf.N;
        surf.N = normalize(nx * surf.T + nz * surf.N + ny * surf.B);
        if (mat->normal_map_strength_unorm != 0xffff) {
            surf.N = normalize(in_normal + (surf.N - in_normal) * unorm16(mat->normal_map_strength_unorm));
        }
        surf.N = ensure_valid_reflection(surf.plane_N, -I, surf.N);
    }

    { // radial tangent in local space
        const v3 P_ls = mk3(v1.p) * w + mk3(v2_.p) * inter.u + mk3(v3_.p) * inter.v;
        v3 tangent = v3{-P_ls.z, 0.0f, P_ls.x};
        tangent = transform_normal(tangent, mi->inv_xform);
        if (length2(cross(tangent, surf.N)) == 0.0f) {
            tangent = transform_normal(P_ls, mi->inv_xform);
        }
        const float rot = mat->tangent_rotation_or_strength;
        if (rot != 0.0f) { // rotate_around_axis :335-353
            const v3 p = tangent, axis = surf.N;
            const v2 sc2 = portable_sincos(rot);
            const float costheta = sc2.y, sintheta = sc2.x;
            v3 r;
            r.x = ((costheta + (1.0f - costheta) * axis.x * axis.x) * p.x) +
                  (((1.0f - costheta) * axis.x * axis.y - axis.z * sintheta) * p.y) +
                  (((1.0f - costheta) * axis.x * axis.z + axis.y * sintheta) * p.z);
            r.y = (((1.0f - costheta) * axis.x * axis.y + axis.z * sintheta) * p.x) +
                  ((costheta + (1.0f - costheta) * axis.y * axis.y) * p.y) +
                  (((1.0f - costheta) * axis.y * axis.z - axis.x * sintheta) * p.z);
            r.z = (((1.0f - costheta) * axis.x * axis.z - axis.y * sintheta) * p.x) +
                  (((1.0f - costheta) * axis.y * axis.z + axis.x * sintheta) * p.y) +
                  ((costheta + (1.0f - costheta) * axis.z * axis.z) * p.z);
            tangent = r;
        }
        surf.B = safe_normalize(cross(tangent, surf.N));
        surf.T = cross(surf.N, surf.B);
    }

    c.ps = &ps;
    c.ray = &ray;
    c.sc = &sc;
    c.inter = &inter;
    c.mat = mat;
    c.mi = mi;
    c.vtx1 = &v1;
    c.vtx2 = &v2_;
    c.vtx3 = &v3_;
    c.col = col;
    c.I = I;
    c.ro = ro;
    c.mix_weight = mix_weight;
    c.mix_rand = mix_rand;
    c.ext_ior = ext_ior;
    c.is_backfacing = is_backfacing;
    c.diff_d = diff_d;
    c.spec_d = spec_d;
    c.refr_d = refr_d;
    c.total_d = total_d;
    c.tri_index = tri_index;
    c.tl_stack = tl_stack;
    c.tl_factors = tl_factors;
    c.rand_dim = rand_dim;
    c.rand_hash = rand_hash;
    c.term_rand_y = mix_term_rand.y;
    c.cone_width = cone_width;
    c.iteration = iteration;
    c.lambda = lambda;
    c.tex_rand = tex_rand;
    return true;
}

RT_DEV void shade_surface_l(const bool tex_on, MatCtx &c) {
    const ShadeScene &sc = *c.sc;
    const Surface &surf = c.surf;
    LightSample &ls = c.ls;
    ls.col = ls.L = ls.lp = v3{0.0f, 0.0f, 0.0f};
    ls.area = 0.0f;
    ls.dist_mul = 1.0f;
    ls.pdf = 0.0f;
    ls.cast_shadow = false;
    ls.from_env = false;
    ls.ray_flags = 0;
    if (sc.lights.nodes_count != 0 && c.mat->type != NODE_EMISSIVE) {
        const float rand_pick_light =
            rand2d(c.rand_dim + kRandDimLightPick, c.rand_hash, c.iteration - 1, sc.rand_seq).x;
        const v2 rand_light_uv = rand2d(c.rand_dim + kRandDimLight, c.rand_hash, c.iteration - 1, sc.rand_seq);
        sample_light_source(tex_on, surf.P, surf.T, surf.B, surf.N, sc.lights, sc.geo, sc.surf, sc.tex, rand_pick_light,
                            rand_light_uv, c.tex_rand, ls);
    }
}

// white_base: RC_RENDER_LIGHTING_ONLY at the first hit -- shade with a white base colour, record the real one as AOV
RT_DEV void shade_surface_b(const bool tex_on, MatCtx &c, float limit1, ShadeOut &out, const bool white_base) {
    const PassSettings &ps = *c.ps;
    const RayD &ray = *c.ray;
    const ShadeScene &sc = *c.sc;
    const Hit &inter = *c.inter;
    const Surface &surf = c.surf;
    const LightSample &ls = c.ls;
    const Material *mat = c.mat;
    const uint32_t rand_dim = c.rand_dim, rand_hash = c.rand_hash;
    const int iteration = c.iteration;
    const float cone_width = c.cone_width;
    const int total_d = c.total_d;
    v3 col = c.col;
    const float N_dot_L = dot(surf.N, ls.L);

    v3 base_color = mk3(mat->base_color);
    if (tex_on && mat->textures[kTexBase] != kTexInvalid) { // ShadeRef.cpp:1405-1419
        const uint32_t base_texture = mat->textures[kTexBase];
        const c4 tex_color = tex_sample_color(sc.tex, base_texture, surf.uvs, tex_lod(sc.tex, base_texture, c.lambda), c.tex_rand, true);
        base_color.x *= tex_color.x;
        base_color.y *= tex_color.y;
        base_color.z *= tex_color.z;
    }
    out.base_color = base_color;
    if (white_base) {
        base_color = v3{1.0f, 1.0f, 1.0f};
    }
    out.aov_normal = surf.N;
    out.aov_depth = inter.t;
    out.wrote_aov = true;

    v3 tint_color = v3{0.0f, 0.0f, 0.0f};
    const float base_color_lum = lum(base_color);
    if (base_color_lum > 0.0f) {
        tint_color = base_color / base_color_lum;
    }

    float roughness = unorm16(mat->roughness_unorm);
    if (tex_on && mat->textures[kTexRough] != kTexInvalid) { // ShadeRef.cpp:1440-1449
        const uint32_t roughness_tex = mat->textures[kTexRough];
        roughness *= tex_sample_color(sc.tex, roughness_tex, surf.uvs, tex_lod(sc.tex, roughness_tex, c.lambda), c.tex_rand).x;
    }

    const v2 rand_bsdf = rand2d(rand_dim + kRandDimBsdf, rand_hash, iteration - 1, sc.rand_seq);

    RayD &new_ray = out.new_ray;
    new_ray.o = new_ray.d = new_ray.c = v3{0.0f, 0.0f, 0.0f};
    new_ray.depth = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        new_ray.ior[i] = ray.ior[i];
    }
    new_ray.cone_width = cone_width;
    new_ray.cone_spread = ray.cone_spread;
    new_ray.xy = ray.xy;
    new_ray.pdf = 0.0f;

    ShadowRayD &sh_r = out.sh_r;
    sh_r.o = sh_r.d = v3{0.0f, 0.0f, 0.0f};
    sh_r.dist = 0.0f;
    sh_r.c = v3{0.0f, 0.0f, 0.0f};
    sh_r.depth = ray.depth;
    sh_r.xy = ray.xy;

    const float regularize_alpha = (diff_depth(ray.depth) > 0) ? ps.regularize_alpha : 0.0f;
    const bool use_mis = (total_d < ps.max_total_depth);

    {
        c.new_ray = &new_ray;
        c.sh_r = &sh_r;
        c.base_color = base_color;
        c.tint_color = tint_color;
        c.N_dot_L = N_dot_L;
        c.roughness = roughness;
        c.regularize_alpha = regularize_alpha;
        c.base_color_lum = base_color_lum;
        c.rand_bsdf = rand_bsdf;
        c.use_mis = use_mis;
        switch (mat->type) {
        case NODE_DIFFUSE: shade_node_diffuse(c); break;
        case NODE_GLOSSY: shade_node_glossy(c); break;
        case NODE_REFRACTIVE: shade_node_refractive(c); break;
        case NODE_EMISSIVE: shade_node_emissive(c); break;
        case NODE_PRINCIPLED: shade_node_principled(tex_on, c); break;
        default: break;
        }
        col = c.col;
    }

    const bool can_terminate_path = total_d > ps.min_total_depth;

    new_ray.c = new_ray.c * ray.c;
    const float lum_ = fmaxf(new_ray.c.x, fmaxf(new_ray.c.y, new_ray.c.z));
    const float p = c.term_rand_y;
    const float q = can_terminate_path ? fmaxf(0.05f, 1.0f - lum_) : 0.0f;
    if (p >= q && lum_ > 0.0f && new_ray.pdf > 0.0f) {
        new_ray.pdf = fminf(new_ray.pdf, 1e6f);
        new_ray.c.x /= (1.0f - q);
        new_ray.c.y /= (1.0f - q);
        new_ray.c.z /= (1.0f - q);
        out.has_secondary = true;
    }

    sh_r.c = sh_r.c * ray.c;
    const float sh_lum = fmaxf(sh_r.c.x, fmaxf(sh_r.c.y, sh_r.c.z));
    if (sh_lum > 0.0f) {
        float dist;
        const v3 to_light = normalize_len(ls.lp - sh_r.o, dist);
        sh_r.d = to_light;
        dist *= ls.dist_mul;
        if (ls.from_env) {
            dist = -dist;
        }
        sh_r.dist = dist;
        out.has_shadow = true;
    }

    col *= ray.c;
    const float sum = ((col.x + col.y) + col.z) + 0.0f;
    if (sum > limit1) {
        col *= (limit1 / sum);
    }
    out.col = c4{col.x, col.y, col.z, 1.0f};
}

} // namespace rt
