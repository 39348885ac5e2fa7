// RendererCuda.cpp -- see RendererCuda.h.
#include "RendererCuda.h"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace RayB200 {

LogNull g_null_log;
LogStdout g_stdout_log;

static void vlog(const char *fmt, va_list vl) {
    vprintf(fmt, vl);
    putc('\n', stdout);
}
void LogStdout::Info(const char *fmt, ...) {
    va_list vl;
    va_start(vl, fmt);
    vlog(fmt, vl);
    va_end(vl);
}
void LogStdout::Warning(const char *fmt, ...) {
    va_list vl;
    va_start(vl, fmt);
    vlog(fmt, vl);
    va_end(vl);
}
void LogStdout::Error(const char *fmt, ...) {
    va_list vl;
    va_start(vl, fmt);
    vlog(fmt, vl);
    va_end(vl);
}

// reference RendererBase.cpp:6-48
std::string_view RendererTypeName(const eRendererType rt) {
    switch (rt) {
    case eRendererType::Reference: return "REF";
    case eRendererType::SIMD_SSE41: return "SSE41";
    case eRendererType::SIMD_AVX: return "AVX";
    case eRendererType::SIMD_AVX2: return "AVX2";
    case eRendererType::SIMD_AVX512: return "AVX512";
    case eRendererType::SIMD_NEON: return "NEON";
    case eRendererType::Vulkan: return "VK";
    case eRendererType::DirectX12: return "DX";
    case eRendererType::CUDA: return "CUDA";
    }
    return "";
}
eRendererType RendererTypeFromName(std::string_view name) {
    for (uint32_t i = 0; i <= uint32_t(eRendererType::CUDA); ++i) {
        if (RendererTypeName(eRendererType(i)) == name) {
            return eRendererType(i);
        }
    }
    return eRendererType::Reference;
}

const char *Version() { return "ray-b200 0.1 (hot path of sergcpp/Ray v0.4.0)"; }

// reference Ray.cpp:53-133: try the backend, log and fall through when its constructor throws
RendererBase *CreateRenderer(const settings_t &s, ILog *log, const ParallelFor &, const uint32_t enabled_types) {
    if (enabled_types & (1u << uint32_t(eRendererType::CUDA))) {
        log->Info("Ray: Creating CUDA renderer %ix%i", s.w, s.h);
        try {
            return new Cuda::Renderer(s, log);
        } catch (std::exception &e) {
            log->Info("Ray: Failed to create CUDA renderer, %s", e.what());
        }
    }
    log->Error("Ray: no enabled renderer type is available in this library (only CUDA exists here; no CPU fallback)");
    return nullptr;
}

namespace Cuda {

// settings_t::preferred_device: "" = device 0, "3" = device 3, "0,1,2,3" / "0-7" / "all" = several devices of this node
// (the frame is sharded over them in row bands, SURVEY.md section 8(e))
static std::vector<int> parse_devices(std::string_view spec) {
    std::vector<int> out;
    const std::string s(spec);
    if (s.empty()) {
        return {0};
    }
    if (s == "all") {
        for (int i = 0; i < rc_device_count(); ++i) {
            out.push_back(i);
        }
        return out;
    }
    size_t pos = 0;
    while (pos < s.size()) {
        size_t end = s.find(',', pos);
        if (end == std::string::npos) {
            end = s.size();
        }
        const std::string tok = s.substr(pos, end - pos);
        const size_t dash = tok.find('-');
        if (dash != std::string::npos && dash > 0) {
            for (int i = atoi(tok.substr(0, dash).c_str()); i <= atoi(tok.substr(dash + 1).c_str()); ++i) {
                out.push_back(i);
            }
        } else if (!tok.empty()) {
            out.push_back(atoi(tok.c_str()));
        }
        pos = end + 1;
    }
    return out;
}

Renderer::Renderer(const settings_t &s, ILog *log) : log_(log) {
    const std::vector<int> devices = parse_devices(s.preferred_device);
    if (devices.empty()) {
        throw std::runtime_error("no CUDA device selected by preferred_device");
    }
    for (const int device : devices) {
        rc_ctx *c = nullptr;
        const int rc = rc_create(device, &c);
        if (rc != 0 || !c) {
            for (rc_ctx *o : ctxs_) {
                rc_destroy(o);
            }
            ctxs_.clear();
            throw std::runtime_error("no usable sm_100 CUDA device " + std::to_string(device) + " (rc_create code " +
                                     std::to_string(rc) + ")");
        }
        ctxs_.push_back(c);
    }
    ctx_ = ctxs_[0];
    if (ctxs_.size() > 1 && rc_comm_init(ctxs_.data(), int(ctxs_.size()), &comm_) != 0) {
        for (rc_ctx *o : ctxs_) {
            rc_destroy(o);
        }
        throw std::runtime_error("rc_comm_init failed (one context per device is required)");
    }
    device_name_ = rc_device_name(ctx_);
    if (ctxs_.size() > 1) {
        device_name_ += " x" + std::to_string(ctxs_.size());
    }
    log_->Info("============================================================================");
    log_->Info("Device       is %s", device_name_.c_str());
    if (s.use_spatial_cache) {
        log_->Warning("SpatialCache is not supported by the CUDA backend (ignored)");
    }
    log_->Info("============================================================================");
    sampler_table_ = GenerateSamplerTable();
    Resize(s.w, s.h);
}

Renderer::~Renderer() {
    FreeMirrors();
    rc_comm_destroy(comm_);
    for (rc_ctx *c : ctxs_) {
        rc_destroy(c);
    }
}

void Renderer::FreeMirrors() {
    rc_host_free(final_buf_);
    rc_host_free(raw_buf_);
    rc_host_free(base_color_buf_);
    rc_host_free(depth_normals_buf_);
    rc_host_free(sh_buf_);
    rc_host_free(sh_stage_);
    final_buf_ = raw_buf_ = base_color_buf_ = depth_normals_buf_ = nullptr;
    sh_buf_ = nullptr;
    sh_stage_ = nullptr;
}

void Renderer::Resize(const int w, const int h) {
    if (w == w_ && h == h_) {
        return;
    }
    for (rc_ctx *c : ctxs_) { // every device holds full-size planes; only its band of rows is ever rendered there
        if (rc_resize(c, w, h) != 0) {
            log_->Error("Ray(CUDA): %s", rc_last_error(c));
            return;
        }
    }
    frame_on_dev0_ = false;
    w_ = w;
    h_ = h;
    const size_t n = size_t(w) * h;
    FreeMirrors();
    final_buf_ = static_cast<color_rgba_t *>(rc_host_alloc(n * sizeof(color_rgba_t)));
    raw_buf_ = static_cast<color_rgba_t *>(rc_host_alloc(n * sizeof(color_rgba_t)));
    base_color_buf_ = static_cast<color_rgba_t *>(rc_host_alloc(n * sizeof(color_rgba_t)));
    depth_normals_buf_ = static_cast<color_rgba_t *>(rc_host_alloc(n * sizeof(color_rgba_t)));
    if (!final_buf_ || !raw_buf_ || !base_color_buf_ || !depth_normals_buf_) {
        log_->Error("Ray(CUDA): failed to allocate the host pixel mirrors");
        return;
    }
    memset(final_buf_, 0, n * sizeof(color_rgba_t));
    memset(raw_buf_, 0, n * sizeof(color_rgba_t));
    memset(base_color_buf_, 0, n * sizeof(color_rgba_t));
    memset(depth_normals_buf_, 0, n * sizeof(color_rgba_t));
    final_dirty_ = raw_dirty_ = base_dirty_ = dn_dirty_ = sh_dirty_ = true;
    sh_used_ = false;
}

void Renderer::Clear(const color_rgba_t &c) {
    for (rc_ctx *x : ctxs_) {
        if (rc_clear(x, c.v) != 0) {
            log_->Error("Ray(CUDA): %s", rc_last_error(x));
        }
    }
    frame_on_dev0_ = false;
    final_dirty_ = raw_dirty_ = base_dirty_ = dn_dirty_ = sh_dirty_ = true;
}

SceneBase *Renderer::CreateScene() { return new Scene(log_, ctx_); }

void Renderer::SetSamplerTable(const uint32_t *table) {
    sampler_table_.assign(table, table + size_t(rt::kRandDims) * rt::kRandSamples * 2);
    tables_dirty_ = true;
}

bool Renderer::Prepare(const Scene &s, const camera_t &cam) {
    if (cam.rc.filter != filter_table_filter_ || cam.desc.filter_width != filter_table_width_) {
        filter_table_ = GenerateFilterTable(cam.rc.filter, cam.desc.filter_width);
        filter_table_filter_ = cam.rc.filter;
        filter_table_width_ = cam.desc.filter_width;
        tables_dirty_ = true;
    }
    if (tables_dirty_) {
        for (rc_ctx *c : ctxs_) {
            if (rc_upload_tables(c, sampler_table_.data(), rt::kRandDims, rt::kRandSamples, filter_table_.data(),
                                 int(filter_table_.size())) != 0) {
                log_->Error("Ray(CUDA): %s", rc_last_error(c));
                return false;
            }
        }
        tables_dirty_ = false;
    }
    if (uploaded_scene_ != &s || uploaded_revision_ != s.revision()) {
        rc_scene_view v;
        s.FillView(v);
        // only instance transforms / lights moved since the upload: refresh the top level, keep the geometry in HBM
        const bool top_level_only = uploaded_scene_ == &s && uploaded_structure_ == s.structure_revision();
        for (rc_ctx *c : ctxs_) { // replicated: every band needs the whole scene
            const int rc = top_level_only ? rc_update_instances(c, &v, s.first_tlas_node()) : rc_upload_scene(c, &v);
            if (rc != 0) {
                log_->Error("Ray(CUDA): %s", rc_last_error(c));
                uploaded_scene_ = nullptr;
                return false;
            }
        }
        uploaded_scene_ = &s;
        uploaded_revision_ = s.revision();
        uploaded_structure_ = s.structure_revision();
    }
    return true;
}

void Renderer::RenderScene(const SceneBase &scene, RegionContext &region) { RenderSceneBatch(scene, region, 1); }

void Renderer::RenderSceneBatch(const SceneBase &scene, RegionContext &region, const int count) {
    const auto *sp = dynamic_cast<const Scene *>(&scene);
    if (!sp) {
        log_->Error("Ray(CUDA): RenderScene needs a scene created by this renderer's CreateScene()");
        return;
    }
    const Scene &s = *sp;
    std::shared_lock<std::shared_timed_mutex> lock(s.mtx_);
    if (s.current_cam_._index >= s.cams_.size()) {
        log_->Error("Ray(CUDA): the scene has no current camera");
        return;
    }
    const camera_t &cam = s.cams_[s.current_cam_._index];
    rc_pass_desc p;
    memset(&p, 0, sizeof(p));
    if (cam.desc.type == RS_CAM_GEO) {
        // the baked instance is resolved against the scene as it is now: it must still exist
        const uint32_t mi = cam.desc.mi_index;
        if (cam.desc.uv_index != 0) {
            log_->Error("Ray(CUDA): Geo camera uv_index %u: meshes carry one uv set", cam.desc.uv_index);
            return;
        }
        if (mi >= s.mesh_instances_.size() || !s.instance_alive_[mi] ||
            s.mesh_instances_[mi].mesh_index >= s.meshes_.size() || !s.meshes_[s.mesh_instances_[mi].mesh_index].alive) {
            log_->Error("Ray(CUDA): Geo camera: mesh instance %u does not exist", mi);
            return;
        }
        const Scene::MeshRec &m = s.meshes_[s.mesh_instances_[mi].mesh_index];
        p.geo_instance = mi;
        p.geo_tri_first = m.tri_first;
        p.geo_tri_count = m.tri_count;
    }
    if (!Prepare(s, cam)) {
        return;
    }
    p.cam = cam.rc;
    p.rect = rc_rect{region.rect().x, region.rect().y, region.rect().w, region.rect().h};
    p.flags = render_flags_ | RC_RENDER_ASYNC;
    p.flags |= (cam.desc.skip_direct_lighting ? RC_RENDER_SKIP_DIRECT : 0u) |
               (cam.desc.skip_indirect_lighting ? RC_RENDER_SKIP_INDIRECT : 0u) |
               (cam.desc.lighting_only ? RC_RENDER_LIGHTING_ONLY : 0u) |
               (cam.desc.no_background ? RC_RENDER_NO_BACKGROUND : 0u) | (cam.desc.output_sh ? RC_RENDER_OUTPUT_SH : 0u);
    if (cam.desc.output_sh) {
        sh_used_ = true;
    }
    for (int i = 0; i < count; ++i) {
        ++region.iteration;
        p.iteration = region.iteration;
        if (comm_) {
            if (rc_comm_render(comm_, &p) != 0) {
                log_->Error("Ray(CUDA): %s", rc_comm_last_error(comm_));
                break;
            }
        } else if (rc_render(ctx_, &p) != 0) {
            log_->Error("Ray(CUDA): %s", rc_last_error(ctx_));
            break;
        }
    }
    if (comm_) {
        if (rc_comm_sync(comm_) != 0) {
            log_->Error("Ray(CUDA): %s", rc_comm_last_error(comm_));
        }
    } else if (rc_sync(ctx_) != 0) {
        log_->Error("Ray(CUDA): %s", rc_last_error(ctx_));
    }
    frame_on_dev0_ = false;
    final_dirty_ = raw_dirty_ = base_dirty_ = dn_dirty_ = sh_dirty_ = true;
}

void Renderer::Readback(const int which, color_rgba_t *dst) const {
    if (w_ == 0 || h_ == 0 || !dst) {
        return;
    }
    const rc_rect r{0, 0, w_, h_};
    if (comm_ && !frame_on_dev0_) {
        // every device copies its own band straight into the page-locked mirror: N PCIe links in parallel
        if (rc_gather(comm_, which, &r, &dst[0].v[0], w_) != 0) {
            log_->Error("Ray(CUDA): %s", rc_comm_last_error(comm_));
        }
        return;
    }
    if (rc_readback(ctx_, which, &r, &dst[0].v[0], w_) != 0) {
        log_->Error("Ray(CUDA): %s", rc_last_error(ctx_));
    }
}

color_data_rgba_t Renderer::get_pixels_ref() const {
    if (final_dirty_) {
        Readback(RC_BUF_FINAL, final_buf_);
        final_dirty_ = false;
    }
    return {final_buf_, w_};
}
color_data_rgba_t Renderer::get_raw_pixels_ref() const {
    if (raw_dirty_) {
        Readback(RC_BUF_RAW, raw_buf_);
        raw_dirty_ = false;
    }
    return {raw_buf_, w_};
}
const shl1_data_t *Renderer::get_sh_data_ref() const {
    if (!sh_used_ || w_ == 0 || h_ == 0) {
        return nullptr;
    }
    if (sh_dirty_) {
        const size_t n = size_t(w_) * h_;
        if (!sh_buf_) {
            sh_buf_ = static_cast<shl1_data_t *>(rc_host_alloc(n * sizeof(shl1_data_t)));
            sh_stage_ = static_cast<color_rgba_t *>(rc_host_alloc(n * sizeof(color_rgba_t)));
            if (!sh_buf_ || !sh_stage_) {
                log_->Error("Ray(CUDA): failed to allocate the host SH mirror");
                return nullptr;
            }
        }
        for (int ch = 0; ch < 3; ++ch) {
            // the SH planes stay where they were rendered (the denoisers do not gather them)
            const rc_rect r{0, 0, w_, h_};
            const int rc = comm_ ? rc_gather(comm_, RC_BUF_SH_R + ch, &r, &sh_stage_[0].v[0], w_)
                                 : rc_readback(ctx_, RC_BUF_SH_R + ch, &r, &sh_stage_[0].v[0], w_);
            if (rc != 0) {
                log_->Error("Ray(CUDA): %s", comm_ ? rc_comm_last_error(comm_) : rc_last_error(ctx_));
                return nullptr;
            }
            for (size_t i = 0; i < n; ++i) {
                float *dst = ch == 0 ? sh_buf_[i].coeff_r : (ch == 1 ? sh_buf_[i].coeff_g : sh_buf_[i].coeff_b);
                memcpy(dst, sh_stage_[i].v, 4 * sizeof(float));
            }
        }
        sh_dirty_ = false;
    }
    return sh_buf_;
}

color_data_rgba_t Renderer::get_aux_pixels_ref(const eAUXBuffer buf) const {
    if (buf == eAUXBuffer::BaseColor) {
        if (base_dirty_) {
            Readback(RC_BUF_BASE_COLOR, base_color_buf_);
            base_dirty_ = false;
        }
        return {base_color_buf_, w_};
    } else if (buf == eAUXBuffer::DepthNormals) {
        if (dn_dirty_) {
            Readback(RC_BUF_DEPTH_NORMALS, depth_normals_buf_);
            dn_dirty_ = false;
        }
        return {depth_normals_buf_, w_};
    }
    return {nullptr, 0};
}

// out of the hot-path scope (SURVEY.md section 8(b)): report through the log like any backend missing a feature
// reference internal/RendererCPU.h:661-787: joint NLM filter of the region (rt_denoise.cuh)
void Renderer::DenoiseImage(const RegionContext &region) {
    const rect_t &r = region.rect();
    const rc_rect rr = {r.x, r.y, r.w, r.h};
    if (comm_) {
        // the filter reads a neighbourhood across band borders: bring the planes it needs onto device 0 (NVLink peer
        // copies) and filter there; pixels are then read back from device 0 until the next RenderScene
        const rc_rect frame{0, 0, w_, h_};
        for (const int plane : {RC_BUF_FULL, RC_BUF_HALF, RC_BUF_RAW, RC_BUF_BASE_COLOR, RC_BUF_DEPTH_NORMALS, RC_BUF_TEMP}) {
            if (rc_gather_device(comm_, plane, &frame) != 0) {
                log_->Error("Ray(CUDA): %s", rc_comm_last_error(comm_));
                return;
            }
        }
        frame_on_dev0_ = true;
        base_dirty_ = dn_dirty_ = true;
    }
    if (rc_denoise_nlm(ctx_, &rr, region.iteration) != 0) {
        log_->Error("Ray(CUDA): %s", rc_last_error(ctx_));
        return;
    }
    final_dirty_ = raw_dirty_ = true;
}
// reference internal/RendererCPU.h:790-1007: one pass of the 16-pass UNet filter (rt_unet.cuh)
void Renderer::DenoiseImage(const int pass, const RegionContext &region) {
    if (comm_ && pass <= 0) {
        // the network runs on device 0 (its receptive field spans the whole frame): bring the planes the first pass
        // reads there over NVLink; the later passes work on device 0's tensors
        const rc_rect frame{0, 0, w_, h_};
        for (const int plane : {RC_BUF_FULL, RC_BUF_BASE_COLOR, RC_BUF_DEPTH_NORMALS}) {
            if (rc_gather_device(comm_, plane, &frame) != 0) {
                log_->Error("Ray(CUDA): %s", rc_comm_last_error(comm_));
                return;
            }
        }
        frame_on_dev0_ = true;
        base_dirty_ = dn_dirty_ = true;
    }
    const rect_t &r = region.rect();
    const rc_rect rr = {r.x, r.y, r.w, r.h};
    if (rc_denoise_unet(ctx_, pass, &rr, unet_flags_) != 0) {
        log_->Error("Ray(CUDA): %s", rc_last_error(ctx_));
        return;
    }
    final_dirty_ = raw_dirty_ = true;
}
void Renderer::UpdateSpatialCache(const SceneBase &, RegionContext &) { log_->Error("Ray(CUDA): the spatial cache is not implemented by the CUDA backend"); }
void Renderer::ResolveSpatialCache(const SceneBase &, const ParallelFor &) { log_->Error("Ray(CUDA): the spatial cache is not implemented by the CUDA backend"); }
void Renderer::ResetSpatialCache(const SceneBase &, const ParallelFor &) {}
// The stand-alone library does not carry OIDN's weight blob (inside the reference tree the binding passes the tree's
// own, oracle/cuda_binding/RendererCUDA.cpp): the application hands it over once with SetUNetWeights.
bool Renderer::SetUNetWeights(const rc_unet_layer layers[16]) {
    if (rc_unet_set_weights(ctx_, layers) != 0) {
        log_->Error("Ray(CUDA): %s", rc_last_error(ctx_));
        return false;
    }
    unet_weights_set_ = true;
    return true;
}

bool Renderer::SetViewTransformLUT(uint32_t view_transform, const uint32_t *lut) {
    for (rc_ctx *c : ctxs_) {
        if (rc_set_view_lut(c, view_transform, lut, 48) != 0) {
            log_->Error("Ray(CUDA): %s", rc_last_error(c));
            return false;
        }
    }
    return true;
}

unet_filter_properties_t Renderer::InitUNetFilter(bool, const ParallelFor &) {
    unet_filter_properties_t props = {};
    if (!unet_weights_set_) {
        log_->Error("Ray(CUDA): InitUNetFilter needs the network weights (Cuda::Renderer::SetUNetWeights)");
        return props;
    }
    props.pass_count = 16; // UNetFilterPasses
    for (int i = 0; i < 16; ++i) {
        for (int j = 0; j < 4; ++j) {
            props.alias_dependencies[i][j] = -1; // tensors are not aliased on the device
        }
    }
    return props;
}

void Renderer::GetStats(stats_t &st) {
    uint64_t us[11] = {};
    rc_get_stats(ctx_, us);
    st.time_primary_ray_gen_us = us[0];
    st.time_primary_trace_us = us[1];
    st.time_primary_shade_us = us[2];
    st.time_primary_shadow_us = us[3];
    st.time_secondary_sort_us = us[4];
    st.time_secondary_trace_us = us[5];
    st.time_secondary_shade_us = us[6];
    st.time_secondary_shadow_us = us[7];
    st.time_denoise_us = us[8];
    st.time_cache_update_us = us[9];
    st.time_cache_resolve_us = us[10];
}
void Renderer::ResetStats() { rc_reset_stats(ctx_); }

} // namespace Cuda
} // namespace RayB200
