// RendererCuda.h -- RayB200::Cuda::Renderer: the RendererBase implementation that drives libray_cuda.so.
//
// Role in the reference: the CUDA twin of Cpu::Renderer<SIMDPolicy> (internal/RendererCPU.h:193-320, RenderScene
// :374-659) / Vk::Renderer (internal/RendererVK.cpp:368-791).  All device work goes through the C-ABI of
// include/ray_cuda.h; this class only converts arguments, tracks scene revisions, and keeps host mirrors of the
// frame buffers for get_*_pixels_ref (lazy readback with dirty flags, like RendererVK.cpp:1698-1757).
#pragma once

#include <mutex>
#include <string>
#include <vector>

#include "../../../include/ray_cuda.h"
#include "RayB200.h"
#include "SceneCuda.h"

namespace RayB200 {
namespace Cuda {

class Renderer final : public RendererBase {
    ILog *log_;
    rc_ctx *ctx_ = nullptr;          // device 0 of this renderer (the only one unless several were asked for)
    std::vector<rc_ctx *> ctxs_;      // all devices; the frame is sharded over them in row bands (include/ray_cuda.h)
    rc_comm *comm_ = nullptr;         // non-null when ctxs_.size() > 1
    mutable bool frame_on_dev0_ = false; // a denoise pass gathered the frame onto device 0: read back from there
    int w_ = 0, h_ = 0;
    std::string device_name_;

    // host mirrors of the device planes, in pinned memory (rc_host_alloc) so a readback runs at full PCIe speed
    mutable color_rgba_t *final_buf_ = nullptr, *raw_buf_ = nullptr, *base_color_buf_ = nullptr, *depth_normals_buf_ = nullptr;
    mutable bool final_dirty_ = true, raw_dirty_ = true, base_dirty_ = true, dn_dirty_ = true;
    // L1 SH of the bake passes (camera_desc_t::output_sh): w*h shl1_data_t, filled from the three RC_BUF_SH_* planes
    mutable shl1_data_t *sh_buf_ = nullptr;
    mutable color_rgba_t *sh_stage_ = nullptr; // one plane, staging for the interleave
    mutable bool sh_dirty_ = true;
    bool sh_used_ = false; // a pass with output_sh ran since the last Resize

    const Scene *uploaded_scene_ = nullptr;
    uint64_t uploaded_revision_ = 0;
    uint64_t uploaded_structure_ = 0;
    uint32_t filter_table_filter_ = 0xffffffffu;
    float filter_table_width_ = 0.0f;
    std::vector<uint32_t> sampler_table_;
    bool tables_dirty_ = true;
    std::vector<float> filter_table_;
    uint32_t render_flags_ = 0;
    uint32_t unet_flags_ = RC_UNET_TENSOR_CORES;
    bool unet_weights_set_ = false;

    void Readback(int which, color_rgba_t *dst) const;
    void FreeMirrors();
    bool Prepare(const Scene &s, const camera_t &cam);

  public:
    Renderer(const settings_t &s, ILog *log); // throws std::runtime_error when no sm_100 device can be opened
    ~Renderer() override;

    eRendererType type() const override { return eRendererType::CUDA; }
    ILog *log() const override { return log_; }
    std::string_view device_name() const override { return device_name_; }
    std::pair<int, int> size() const override { return {w_, h_}; }
    color_data_rgba_t get_pixels_ref() const override;
    color_data_rgba_t get_raw_pixels_ref() const override;
    color_data_rgba_t get_aux_pixels_ref(eAUXBuffer buf) const override;
    const shl1_data_t *get_sh_data_ref() const override;
    void Resize(int w, int h) override;
    void Clear(const color_rgba_t &c) override;
    SceneBase *CreateScene() override;
    void RenderScene(const SceneBase &scene, RegionContext &region) override;
    void DenoiseImage(const RegionContext &region) override;
    void DenoiseImage(int pass, const RegionContext &region) override;
    void UpdateSpatialCache(const SceneBase &scene, RegionContext &region) override;
    void ResolveSpatialCache(const SceneBase &scene, const ParallelFor &parallel_for) override;
    void ResetSpatialCache(const SceneBase &scene, const ParallelFor &parallel_for) override;
    void GetStats(stats_t &st) override;
    void ResetStats() override;
    unet_filter_properties_t InitUNetFilter(bool alias_memory, const ParallelFor &parallel_for) override;

    // ---- CUDA-backend extras (not part of RendererBase) ----
    /// `count` consecutive RenderScene calls on the same region enqueued back to back with ONE synchronisation at the
    /// end (the per-call blocking semantic of RenderScene costs a host round trip per sample).
    void RenderSceneBatch(const SceneBase &scene, RegionContext &region, int count);
    /// Replace the built-in (0,2)-sequence sampler table with a caller-provided 32 x 4096 x 2 table -- inside the
    /// reference tree this is `__pmj02_samples`; parity tests pass that table so the sample sequences are identical.
    void SetSamplerTable(const uint32_t *table);
    void SetRenderFlags(uint32_t rc_render_flags) { render_flags_ = rc_render_flags; }
    /// The 16 convolutions of the UNet denoiser as fp16 OIHW weights + biases (include/ray_cuda.h rc_unet_layer).
    bool SetUNetWeights(const rc_unet_layer layers[16]);
    // 48^3 packed table of an AgX / Filmic view transform (Ray::transform_luts[view_transform] inside the reference
    // tree; the stand-alone library does not carry the tables)
    bool SetViewTransformLUT(uint32_t view_transform, const uint32_t *lut);
    void SetUNetFlags(uint32_t rc_unet_flags) { unet_flags_ = rc_unet_flags; }
    /// Forget the uploaded scene: the next RenderScene copies all scene arrays host->device again (dynamic scenes,
    /// end-to-end measurements).
    void InvalidateScene() { uploaded_scene_ = nullptr; }
    rc_ctx *native_context() const { return ctx_; }
    rc_comm *native_comm() const { return comm_; }
    int device_count() const { return int(ctxs_.size()); }
};

std::vector<uint32_t> GenerateSamplerTable();                                   // SamplerTable.cpp
std::vector<float> GenerateFilterTable(uint32_t filter, float filter_width);   // FilterTable.cpp

} // namespace Cuda
} // namespace RayB200
