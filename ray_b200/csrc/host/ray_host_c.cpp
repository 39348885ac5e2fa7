// ray_host_c.cpp -- flat C wrapper (include/ray_host.h) over the C++ host layer.
#include "../../../include/ray_host.h"

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>

#include "RendererCuda.h"

using namespace RayB200;

namespace {
class CollectLog final : public ILog {
  public:
    std::mutex m;
    int errors = 0;
    std::string last;
    void Info(const char *, ...) override {}
    void Warning(const char *, ...) override {}
    void Error(const char *fmt, ...) override {
        char buf[1024];
        va_list vl;
        va_start(vl, fmt);
        vsnprintf(buf, sizeof(buf), fmt, vl);
        va_end(vl);
        std::lock_guard<std::mutex> _(m);
        ++errors;
        last = buf;
    }
};
struct RendererBox {
    std::unique_ptr<CollectLog> log;
    std::unique_ptr<RendererBase> r;
};
CollectLog g_standalone_log; // log of free-standing scenes (rh_create_scene(NULL))
inline RendererBox *B(rh_renderer *r) { return reinterpret_cast<RendererBox *>(r); }
inline Cuda::Renderer *R(rh_renderer *r) { return static_cast<Cuda::Renderer *>(B(r)->r.get()); }
inline Cuda::Scene *S(rh_scene *s) { return reinterpret_cast<Cuda::Scene *>(s); }
} // namespace

extern "C" {

static rh_renderer *create_renderer(int w, int h, const std::string &dev);

rh_renderer *rh_create_renderer(int w, int h, int device) { return create_renderer(w, h, std::to_string(device)); }

// devices: settings_t::preferred_device of the CUDA backend ("3", "0,1,2,3", "0-7", "all")
rh_renderer *rh_create_renderer_multi(int w, int h, const char *devices) { return create_renderer(w, h, devices ? devices : ""); }

static rh_renderer *create_renderer(int w, int h, const std::string &dev) {
    auto box = std::make_unique<RendererBox>();
    box->log = std::make_unique<CollectLog>();
    settings_t st;
    st.w = w;
    st.h = h;
    st.preferred_device = dev;
    RendererBase *r = CreateRenderer(st, box->log.get(), parallel_for_serial, 1u << uint32_t(eRendererType::CUDA));
    if (!r) {
        return nullptr;
    }
    box->r.reset(r);
    box->log->errors = 0;
    return reinterpret_cast<rh_renderer *>(box.release());
}
void rh_destroy_renderer(rh_renderer *r) { delete B(r); }
const char *rh_device_name(rh_renderer *r) {
    static thread_local std::string s;
    s = std::string(R(r)->device_name());
    return s.c_str();
}
int rh_error_count(rh_renderer *r) { return r ? B(r)->log->errors : g_standalone_log.errors; }
const char *rh_last_error(rh_renderer *r) { return r ? B(r)->log->last.c_str() : g_standalone_log.last.c_str(); }
void rh_resize(rh_renderer *r, int w, int h) { R(r)->Resize(w, h); }
void rh_clear(rh_renderer *r, const float rgba[4]) { R(r)->Clear(color_rgba_t{{rgba[0], rgba[1], rgba[2], rgba[3]}}); }

rh_scene *rh_create_scene(rh_renderer *r) {
    if (!r) {
        // scene building is pure host work: a NULL renderer gives a free-standing Cuda::Scene (CPU-side tests of the
        // builders); its errors go to a process-wide log readable through rh_error_count(NULL) / rh_last_error(NULL)
        return reinterpret_cast<rh_scene *>(static_cast<SceneBase *>(new Cuda::Scene(&g_standalone_log)));
    }
    return reinterpret_cast<rh_scene *>(R(r)->CreateScene());
}
void rh_destroy_scene(rh_scene *s) { delete static_cast<SceneBase *>(S(s)); }
void rh_set_environment(rh_scene *s, const rs_environment_desc *d) { S(s)->SetEnvironment(*d); }
uint32_t rh_add_texture(rh_scene *s, const rs_tex_desc *d) { return S(s)->AddTexture(*d)._index; }
uint32_t rh_add_material_node(rh_scene *s, const rs_shading_node_desc *d) { return S(s)->AddMaterial(*d)._index; }
uint32_t rh_add_material_principled(rh_scene *s, const rs_principled_mat_desc *d) { return S(s)->AddMaterial(*d)._index; }
uint32_t rh_add_mesh(rh_scene *s, const rs_mesh_desc *d) { return S(s)->AddMesh(*d)._index; }
uint32_t rh_add_mesh_instance(rh_scene *s, const rs_mesh_instance_desc *d) { return S(s)->AddMeshInstance(*d)._index; }
void rh_set_mesh_instance_transform(rh_scene *s, uint32_t instance, const float *xform) {
    MeshInstanceHandle h;
    h._index = instance;
    S(s)->SetMeshInstanceTransform(h, xform);
}
void rh_remove_mesh_instance(rh_scene *s, uint32_t instance) {
    MeshInstanceHandle h;
    h._index = instance;
    S(s)->RemoveMeshInstance(h);
}
uint32_t rh_add_light_directional(rh_scene *s, const rs_directional_light_desc *d) { return S(s)->AddLight(*d)._index; }
uint32_t rh_add_light_sphere(rh_scene *s, const rs_sphere_light_desc *d) { return S(s)->AddLight(*d)._index; }
uint32_t rh_add_light_spot(rh_scene *s, const rs_spot_light_desc *d) { return S(s)->AddLight(*d)._index; }
uint32_t rh_add_light_rect(rh_scene *s, const rs_rect_light_desc *d) { return S(s)->AddLight(*d)._index; }
uint32_t rh_add_light_disk(rh_scene *s, const rs_disk_light_desc *d) { return S(s)->AddLight(*d)._index; }
uint32_t rh_add_light_line(rh_scene *s, const rs_line_light_desc *d) { return S(s)->AddLight(*d)._index; }
uint32_t rh_add_camera(rh_scene *s, const rs_camera_desc *d) {
    const CameraHandle h = S(s)->AddCamera(*d);
    S(s)->set_current_cam(h);
    return h._index;
}
void rh_finalize(rh_scene *s) { S(s)->Finalize(); }
uint32_t rh_triangle_count(rh_scene *s) { return S(s)->triangle_count(); }
uint32_t rh_node_count(rh_scene *s) { return S(s)->node_count(); }
void rh_scene_view(rh_scene *s, rc_scene_view *out) { S(s)->FillView(*out); }
void rh_get_camera(rh_scene *s, rc_camera *out) {
    if (!S(s)->GetDeviceCamera(*out)) {
        memset(out, 0, sizeof(*out));
    }
}

void rh_render(rh_renderer *r, rh_scene *s, const rc_rect *rect, int *iteration, int count) {
    RegionContext region(rect_t{rect->x, rect->y, rect->w, rect->h});
    region.iteration = *iteration;
    if (count <= 1) {
        R(r)->RenderScene(*S(s), region);
    } else {
        R(r)->RenderSceneBatch(*S(s), region, count);
    }
    *iteration = region.iteration;
}
void rh_denoise(rh_renderer *r, const rc_rect *rect, int iteration) {
    RegionContext region(rect_t{rect->x, rect->y, rect->w, rect->h});
    region.iteration = iteration;
    R(r)->DenoiseImage(region);
}
const float *rh_get_pixels(rh_renderer *r, int which, int *pitch) {
    color_data_rgba_t d{nullptr, 0};
    switch (which) {
    case 0: d = R(r)->get_pixels_ref(); break;
    case 1: d = R(r)->get_raw_pixels_ref(); break;
    case 2: d = R(r)->get_aux_pixels_ref(eAUXBuffer::BaseColor); break;
    case 3: d = R(r)->get_aux_pixels_ref(eAUXBuffer::DepthNormals); break;
    default: break;
    }
    if (pitch) {
        *pitch = d.pitch;
    }
    return d.ptr ? d.ptr->v : nullptr;
}
const float *rh_get_sh_data(rh_renderer *r, int *pitch) {
    const shl1_data_t *d = R(r)->get_sh_data_ref();
    if (pitch) {
        *pitch = d ? R(r)->size().first : 0;
    }
    return d ? d->coeff_r : nullptr;
}
void rh_get_stats(rh_renderer *r, uint64_t us[11]) {
    RendererBase::stats_t st = {};
    R(r)->GetStats(st);
    const unsigned long long v[11] = {st.time_primary_ray_gen_us, st.time_primary_trace_us, st.time_primary_shade_us,
                                      st.time_primary_shadow_us,  st.time_secondary_sort_us, st.time_secondary_trace_us,
                                      st.time_secondary_shade_us, st.time_secondary_shadow_us, st.time_denoise_us,
                                      st.time_cache_update_us,    st.time_cache_resolve_us};
    for (int i = 0; i < 11; ++i) {
        us[i] = v[i];
    }
}
void rh_reset_stats(rh_renderer *r) { R(r)->ResetStats(); }
void rh_get_counters(rh_renderer *r, rc_counters *out) {
    if (R(r)->native_comm()) {
        rc_comm_get_counters(R(r)->native_comm(), out);
    } else {
        rc_get_counters(R(r)->native_context(), out);
    }
}
int rh_device_count(rh_renderer *r) { return R(r)->device_count(); }
// UNet denoiser: weights once, then InitUNetFilter + DenoiseImage(pass, region) for every pass (returns the pass count)
int rh_set_unet_weights(rh_renderer *r, const rc_unet_layer layers[16], uint32_t unet_flags) {
    R(r)->SetUNetFlags(unet_flags);
    return R(r)->SetUNetWeights(layers) ? 0 : 1;
}
int rh_set_view_lut(rh_renderer *r, uint32_t view_transform, const uint32_t *lut) {
    return R(r)->SetViewTransformLUT(view_transform, lut) ? 0 : 1;
}
int rh_denoise_unet(rh_renderer *r, const rc_rect *rect, int iteration) {
    const unet_filter_properties_t props = R(r)->InitUNetFilter(false, parallel_for_serial);
    RegionContext region(rect_t{rect->x, rect->y, rect->w, rect->h});
    region.iteration = iteration;
    for (int pass = 0; pass < props.pass_count; ++pass) {
        R(r)->DenoiseImage(pass, region);
    }
    return props.pass_count;
}
void rh_get_kernel_ms(rh_renderer *r, double ms[6], uint64_t launches[6]) { rc_get_kernel_ms(R(r)->native_context(), ms, launches); }
void rh_set_sampler_table(rh_renderer *r, const uint32_t *table) { R(r)->SetSamplerTable(table); }
void rh_set_render_flags(rh_renderer *r, uint32_t f) { R(r)->SetRenderFlags(f); }
void rh_invalidate_scene(rh_renderer *r) { R(r)->InvalidateScene(); }
void *rh_native_context(rh_renderer *r) { return R(r)->native_context(); }
void rh_builtin_sampler_table(uint32_t *out) {
    const std::vector<uint32_t> t = Cuda::GenerateSamplerTable();
    memcpy(out, t.data(), t.size() * sizeof(uint32_t));
}
void rh_builtin_filter_table(uint32_t filter, float filter_width, float *out) {
    const std::vector<float> t = Cuda::GenerateFilterTable(filter, filter_width);
    memcpy(out, t.data(), t.size() * sizeof(float));
}
int rh_abi_sizeof(int which) {
    switch (which) {
    case 0: return int(sizeof(rs_shading_node_desc));
    case 1: return int(sizeof(rs_principled_mat_desc));
    case 2: return int(sizeof(rs_mat_group_desc));
    case 3: return int(sizeof(rs_vtx_attribute));
    case 4: return int(sizeof(rs_mesh_desc));
    case 5: return int(sizeof(rs_mesh_instance_desc));
    case 6: return int(sizeof(rs_light_common));
    case 7: return int(sizeof(rs_directional_light_desc));
    case 8: return int(sizeof(rs_sphere_light_desc));
    case 9: return int(sizeof(rs_spot_light_desc));
    case 10: return int(sizeof(rs_rect_light_desc));
    case 11: return int(sizeof(rs_disk_light_desc));
    case 12: return int(sizeof(rs_line_light_desc));
    case 13: return int(sizeof(rs_camera_desc));
    case 14: return int(sizeof(rs_environment_desc));
    default: return -1;
    }
}

} // extern "C"
