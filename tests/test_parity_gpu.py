"""GPU parity: every stage of the CUDA hot path against the reference's own Ref:: functions (oracle/_ref), fed the
same inputs on byte-identical scene arrays, through the C-ABI stage entry points.  Bar: BIT-EXACT records.

Stages mirror the SIMDPolicy stage functions of the reference (internal/RendererCPU.h:39-189):
  GeneratePrimaryRays -> TraceRays -> ShadePrimary -> TraceShadowRays -> [TraceRays(lights) -> ShadeSecondary -> ...]

Without the oracle library (it is built from the reference's sources) every case runs on the scene built by the product's
host layer with the built-in tables, feeds each stage the CUDA path's own outputs of the previous stage, and checks every
output bitwise against the digests stored in tests/golden/cuda_digests.json (common.STORED).
"""
import numpy as np
import pytest

from ray_b200 import capi, scenes
from common import STORED, bits_equal, by_xy, field_mismatch, make_pair, maybe_oracle

pytestmark = pytest.mark.gpu

SCENES = {
    "cornell": lambda: scenes.cornell_box(96, 96),
    "zoo": lambda: scenes.material_zoo(),
    "zoo_env_dof": lambda: scenes.material_zoo(128, 96, lights=("rect", "sphere"), env=(0.4, 0.5, 0.7),
                                               filter=capi.FILTER_BLACKMAN_HARRIS, fstop=2.0),
    # hexagonal, rotated, anamorphic aperture + sensor shift + radiance clamps + exposure / gamma
    "zoo_lens_clamp": lambda: _lens_clamp_scene(),
    "instanced": lambda: scenes.instanced(36, 600, 128, 96),
    "hall_small": lambda: scenes.hall("principled", 160, 90, floor_res=48, n_columns=8, col_seg=12, col_rings=8,
                                      extra_lights=12),
    # SURVEY section 8(f) row 1: every texture fetch on the path (base / roughness / metallic / specular / normal maps,
    # texture-driven Mix, alpha cut-out through the transparency loops, textured emissive triangles)
    "textured": lambda: scenes.textured(96, 72),
    # SURVEY section 8(f) row 2: RGBE lat-long environment map: miss shading, quad-tree importance sampling + MIS,
    # a rotated background map for camera rays, a sky-portal rect light
    "envmap_zoo": lambda: scenes.envmap_zoo(96, 72),
    # the same textured scene built the way the reference does by default (settings_t::use_tex_compression = true):
    # BCn-coded blocks and YCoCg-coded base-colour maps (CoreRef.h:239-251, ShadeRef.cpp:1308,1411)
    "textured_compressed": lambda: scenes.textured(96, 72),
}


def _lens_clamp_scene():
    d = scenes.material_zoo(112, 80, lights=("spot", "disk", "line"), env=(0.2, 0.2, 0.25), filter=capi.FILTER_GAUSSIAN,
                            fstop=1.4)
    c = d.camera
    c.lens_blades, c.lens_rotation, c.lens_ratio = 6, 0.3, 1.3
    c.shift[0], c.shift[1] = 0.05, -0.03
    c.clamp_direct, c.clamp_indirect = 2.0, 1.0
    c.exposure, c.gamma = 0.5, 2.2
    c.filter_width = 2.0
    return d


@pytest.fixture(scope="module", params=list(SCENES))
def pair(request):
    p = make_pair(SCENES[request.param](), tex_compression=(request.param == "textured_compressed"))
    p.name = request.param
    yield p
    p.close()


def _assert_records(a, b, what):
    a, b = by_xy(a), by_xy(b)
    assert len(a) == len(b), f"{what}: {len(a)} records vs reference {len(b)}"
    if not bits_equal(a, b):
        raise AssertionError(f"{what}: records differ bitwise in fields {field_mismatch(a, b)} of {len(a)}")


@pytest.mark.parametrize("iteration", [1, 7])
def test_generate_primary_rays(pair, iteration):
    p = pair.make_pass(iteration)
    rays, hits = pair.ctx.stage_generate_primary_rays(p)
    assert len(rays) == pair.w * pair.h
    if pair.osc is None:
        order = np.argsort(rays["xy"], kind="stable")
        STORED.check(f"parity/{pair.name}/primary_rays/{iteration}", rays[order], hits[order])
        return
    ref_rays, ref_hits = pair.osc.generate_primary_rays(pair.w, pair.h, (0, 0, pair.w, pair.h), iteration)
    order, ref_order = np.argsort(rays["xy"], kind="stable"), np.argsort(ref_rays["xy"], kind="stable")
    assert bits_equal(rays[order], ref_rays[ref_order]), field_mismatch(rays[order], ref_rays[ref_order])
    assert bits_equal(hits[order], ref_hits[ref_order]), field_mismatch(hits[order], ref_hits[ref_order])


def test_trace_primary(pair):
    it = 3
    if pair.osc is None:
        rays, hits = pair.ctx.stage_generate_primary_rays(pair.make_pass(it))
        order = np.argsort(rays["xy"], kind="stable")  # pixel order, as the reference generates them
        rays, hits = rays[order], hits[order]
        g_rays, g_hits = pair.ctx.stage_trace_rays(pair.make_pass(it), rays, hits, False)
        assert (g_hits["v"] >= 0).any()
        STORED.check(f"parity/{pair.name}/trace_primary", g_rays, g_hits)
        return
    ref_rays, ref_hits = pair.osc.generate_primary_rays(pair.w, pair.h, (0, 0, pair.w, pair.h), it)
    o_rays, o_hits = pair.osc.trace_rays(it, ref_rays, ref_hits, False)
    g_rays, g_hits = pair.ctx.stage_trace_rays(pair.make_pass(it), ref_rays, ref_hits, False)
    # misses carry an unresolved prim_index by design (SURVEY appendix C.2) but it is the same garbage on both sides
    assert bits_equal(g_hits, o_hits), field_mismatch(g_hits, o_hits)
    assert bits_equal(g_rays, o_rays), field_mismatch(g_rays, o_rays)
    assert (o_hits["v"] >= 0).any()


def test_wavefront_stage_by_stage(pair):
    """Walk 1 sample through all bounces, feeding BOTH sides the reference's outputs of the previous stage, and compare
    every stage's outputs bitwise: secondary rays, shadow rays, the radiance (temp) buffer and the primary AOVs."""
    it = 2
    w, h = pair.w, pair.h
    cam = pair.cam
    p = pair.make_pass(it)
    if pair.osc is None:
        return _stage_by_stage_stored(pair, it)
    rays, hits = pair.osc.generate_primary_rays(w, h, (0, 0, w, h), it)
    rays, hits = pair.osc.trace_rays(it, rays, hits, False)

    temp = np.zeros((h, w, 4), np.float32)
    pair.ctx.fill_temp((0, 0, 0, 0))
    o_sec, o_sh, o_base, o_dn = pair.osc.shade(w, h, it, True, 0, rays, hits, temp)
    g_sec, g_sh = pair.ctx.stage_shade(p, True, 0, rays, hits)
    _assert_records(g_sec, o_sec, "primary shade: secondary rays")
    _assert_records(g_sh, o_sh, "primary shade: shadow rays")
    assert bits_equal(pair.ctx.readback(capi.RC_BUF_TEMP), temp), "primary shade: colour buffer"
    assert bits_equal(pair.ctx.readback(capi.RC_BUF_BASE_COLOR), o_base), "primary shade: base colour AOV"
    assert bits_equal(pair.ctx.readback(capi.RC_BUF_DEPTH_NORMALS), o_dn), "primary shade: depth-normal AOV"

    pair.osc.trace_shadow_rays(w, it, o_sh, cam.clamp_direct, temp)
    pair.ctx.stage_trace_shadow_rays(p, o_sh, cam.clamp_direct)
    assert bits_equal(pair.ctx.readback(capi.RC_BUF_TEMP), temp), "primary shadow: colour buffer"

    total = len(rays)
    sec = by_xy(o_sec)
    for bounce in range(1, cam.max_total_depth + 1):
        if len(sec) == 0:
            break
        hits0 = np.zeros(len(sec), dtype=hits.dtype)
        hits0["obj_index"] = -1
        hits0["prim_index"] = -1
        hits0["t"] = np.float32(3.402823466e+30)
        hits0["v"] = -1.0
        o_rays, o_hits = pair.osc.trace_rays(it, sec, hits0, True)
        g_rays, g_hits = pair.ctx.stage_trace_rays(p, sec, hits0, True)
        assert bits_equal(g_hits, o_hits), f"bounce {bounce} trace: hits {field_mismatch(g_hits, o_hits)}"
        assert bits_equal(g_rays, o_rays), f"bounce {bounce} trace: rays {field_mismatch(g_rays, o_rays)}"
        total += len(sec)

        o_sec, o_sh, _, _ = pair.osc.shade(w, h, it, False, bounce, o_rays, o_hits, temp)
        g_sec, g_sh = pair.ctx.stage_shade(p, False, bounce, o_rays, o_hits)
        _assert_records(g_sec, o_sec, f"bounce {bounce} shade: secondary rays")
        _assert_records(g_sh, o_sh, f"bounce {bounce} shade: shadow rays")
        assert bits_equal(pair.ctx.readback(capi.RC_BUF_TEMP), temp), f"bounce {bounce} shade: colour buffer"

        pair.osc.trace_shadow_rays(w, it, o_sh, cam.clamp_indirect, temp)
        pair.ctx.stage_trace_shadow_rays(p, o_sh, cam.clamp_indirect)
        assert bits_equal(pair.ctx.readback(capi.RC_BUF_TEMP), temp), f"bounce {bounce} shadow: colour buffer"
        sec = by_xy(o_sec)
    assert total > w * h, "no secondary rays were exercised"


def _stage_by_stage_stored(pair, it):
    """The stage walk above on the CUDA path alone, each stage fed the previous one's outputs (sorted by pixel, as the
    reference's are), every output checked against its stored digest."""
    w, h, cam, key = pair.w, pair.h, pair.cam, f"parity/{pair.name}/stages"
    p = pair.make_pass(it)
    rays, hits = pair.ctx.stage_generate_primary_rays(p)
    order = np.argsort(rays["xy"], kind="stable")
    rays, hits = pair.ctx.stage_trace_rays(p, rays[order], hits[order], False)
    pair.ctx.fill_temp((0, 0, 0, 0))
    sec, sh = pair.ctx.stage_shade(p, True, 0, rays, hits)
    sec, sh = by_xy(sec), by_xy(sh)
    STORED.check(f"{key}/primary_shade", sec, sh, pair.ctx.readback(capi.RC_BUF_TEMP),
                 pair.ctx.readback(capi.RC_BUF_BASE_COLOR), pair.ctx.readback(capi.RC_BUF_DEPTH_NORMALS))
    pair.ctx.stage_trace_shadow_rays(p, sh, cam.clamp_direct)
    STORED.check(f"{key}/primary_shadow", pair.ctx.readback(capi.RC_BUF_TEMP))
    total = len(rays)
    for bounce in range(1, cam.max_total_depth + 1):
        if len(sec) == 0:
            break
        hits0 = np.zeros(len(sec), dtype=hits.dtype)
        hits0["obj_index"] = -1
        hits0["prim_index"] = -1
        hits0["t"] = np.float32(3.402823466e+30)
        hits0["v"] = -1.0
        g_rays, g_hits = pair.ctx.stage_trace_rays(p, sec, hits0, True)
        total += len(sec)
        sec, sh = pair.ctx.stage_shade(p, False, bounce, g_rays, g_hits)
        sec, sh = by_xy(sec), by_xy(sh)
        pair.ctx.stage_trace_shadow_rays(p, sh, cam.clamp_indirect)
        STORED.check(f"{key}/bounce{bounce}", g_hits, sec, sh, pair.ctx.readback(capi.RC_BUF_TEMP))
    assert total > w * h, "no secondary rays were exercised"


@pytest.mark.parametrize("sort", [False, True])
def test_full_render_matches_reference_renderer(pair, sort):
    """rc_render (the whole RenderScene sequence, with and without the results-neutral ray sort) against the
    reference's own Ref renderer run on the SAME wide-BVH scene object: north_star bar is 1e-4 per-pixel L-inf on the
    linear image; this backend is expected to be bit-identical."""
    spp = 4
    if pair.osc is not None:
        ref = pair.oracle.Renderer(capi.RT_REFERENCE, pair.w, pair.h)
        it = 0
        for _ in range(spp):
            it = ref.render(pair.osc, (0, 0, pair.w, pair.h), it)
        ref_raw, ref_final = ref.pixels(1), ref.pixels(0)
        ref_base, ref_dn = ref.pixels(2), ref.pixels(3)
        ref.close()

    pair.ctx.resize(pair.w, pair.h)
    pair.ctx.clear((0, 0, 0, 0))
    pair.ctx.fill_temp((0, 0, 0, 0))
    # fresh AOV accumulation: Resize() is a no-op at unchanged size, so run on a context-local clean state instead
    flags = 0 if sort else capi.RC_RENDER_NO_SORT
    for i in range(1, spp + 1):
        pair.ctx.render(pair.make_pass(i, flags=flags))
    raw = pair.ctx.readback(capi.RC_BUF_RAW)
    final = pair.ctx.readback(capi.RC_BUF_FINAL)
    c = pair.ctx.counters()
    assert c["primary_rays"] >= spp * pair.w * pair.h
    if pair.osc is None:
        # one digest for both: the ray sort must not change a bit of the image
        STORED.check(f"parity/{pair.name}/full_render", raw, final)
        if sort:
            pair.ctx.resize(pair.w + 1, pair.h)
            pair.ctx.resize(pair.w, pair.h)
            for i in range(1, spp + 1):
                pair.ctx.render(pair.make_pass(i, flags=flags))
            STORED.check(f"parity/{pair.name}/full_render_aovs", pair.ctx.readback(capi.RC_BUF_BASE_COLOR),
                         pair.ctx.readback(capi.RC_BUF_DEPTH_NORMALS))
        return
    diff = np.abs(raw - ref_raw)
    n_bad = int((diff.max(axis=-1) > 1e-4).sum())
    assert n_bad == 0, f"{n_bad} pixels differ by more than 1e-4 (L-inf {diff.max()})"
    assert bits_equal(raw, ref_raw), f"linear image not bit-identical: L-inf {diff.max()}, {int((diff > 0).any(-1).sum())} px"
    # the display transform goes through powf: the device runs a restatement of the host libm's algorithm (rt_math.cuh
    # libm_powf, tests/test_libm.py), so the tonemapped plane is bit-identical too
    assert bits_equal(final, ref_final), f"tonemapped image: L-inf {np.abs(final - ref_final).max()}"
    if sort:
        # AOVs (running means of base colour and depth / normals, ShadeRef.cpp:1677-1698); the stage test above left
        # them dirty, so compare a run that starts from zeroed planes
        pair.ctx.resize(pair.w + 1, pair.h)
        pair.ctx.resize(pair.w, pair.h)
        for i in range(1, spp + 1):
            pair.ctx.render(pair.make_pass(i, flags=flags))
        assert bits_equal(pair.ctx.readback(capi.RC_BUF_BASE_COLOR), ref_base), "base colour AOV"
        assert bits_equal(pair.ctx.readback(capi.RC_BUF_DEPTH_NORMALS), ref_dn), "depth-normals AOV"


def _ref_render(o, pair, spp):
    """The reference's RendererRef, `spp` samples over the pair's scene (None without the oracle)."""
    if o is None:
        return None, 0
    ref = o.Renderer(capi.RT_REFERENCE, pair.w, pair.h)
    it = 0
    for _ in range(spp):
        it = ref.render(pair.osc, (0, 0, pair.w, pair.h), it)
    return ref, it


def _cuda_render(pair, spp):
    pair.ctx.clear((0, 0, 0, 0))
    for i in range(1, spp + 1):
        pair.ctx.render(pair.make_pass(i))
    return pair.ctx.readback(capi.RC_BUF_RAW), spp


def test_adaptive_sampling_matches_reference_renderer():
    """variance estimate + required_samples (RendererCPU.h:607-658): pixels whose two half-buffers agree stop being
    sampled after min_samples, raygen skips them (CoreRef.cpp:1446-1449).  Same image, bit for bit, as RendererRef."""
    o = maybe_oracle()
    desc = scenes.cornell_box(64, 64)
    desc.camera.min_samples = 4
    desc.camera.variance_threshold = 0.02
    pair = make_pair(desc)
    spp = 12
    ref, _ = _ref_render(o, pair, spp)
    raw, _ = _cuda_render(pair, spp)
    if ref is None:
        STORED.check("parity/adaptive", raw, pair.ctx.required_samples())
    else:
        ref_raw = ref.pixels(1)
        ref.close()
        assert bits_equal(raw, ref_raw)
    c = pair.ctx.counters()
    assert c["primary_rays"] < spp * pair.w * pair.h, "no pixel converged: the adaptive path was not exercised"
    pair.close()


def test_nlm_denoise_matches_reference_renderer():
    """RendererBase::DenoiseImage(region) (SURVEY 8(f)-3, NLM half): same 8 spp accumulated on both sides (bit-identical,
    see above), then the joint NLM filter.  The filtered LINEAR image must be bit-identical (the weights go through a
    restated libm expf); the tonemapped plane goes through powf (tolerance as for rc_render).  A sub-rect call checks
    the clamped fetches at region borders that are not image borders."""
    o = maybe_oracle()
    desc = scenes.cornell_box(96, 80)
    pair = make_pair(desc)
    spp = 8
    ref, it = _ref_render(o, pair, spp)
    raw, it = _cuda_render(pair, spp)
    if ref is None:
        STORED.check("parity/nlm/noisy", raw)
    else:
        assert bits_equal(raw, ref.pixels(1))
    for rect in ((0, 0, pair.w, pair.h), (17, 9, 40, 33)):
        pair.ctx.denoise_nlm(rect, it)
        raw, final = pair.ctx.readback(capi.RC_BUF_RAW), pair.ctx.readback(capi.RC_BUF_FINAL)
        x, y, w, h = rect
        sl = (slice(y, y + h), slice(x, x + w))
        assert np.isfinite(raw[sl]).all()
        if ref is None:
            STORED.check(f"parity/nlm/{rect}", raw[sl], final[sl])
            continue
        ref.denoise(rect, it)
        ref_raw, ref_final = ref.pixels(1), ref.pixels(0)
        d = np.abs(raw[sl] - ref_raw[sl])
        assert bits_equal(raw[sl], ref_raw[sl]), f"rect {rect}: filtered linear image L-inf {d.max()}, {int((d > 0).any(-1).sum())} px"
        assert bits_equal(final[sl], ref_final[sl]), f"rect {rect}: tonemapped L-inf {np.abs(final[sl] - ref_final[sl]).max()}"
    if ref is not None:
        ref.close()
    pair.close()


def _synthetic_view_lut(seed):
    """A 48^3 packed 10-10-10-2 table for the runs without the reference's own AgX / Filmic tables: a seeded monotone
    curve per channel, so the device's lookup and interpolation are exercised on a table that is not the identity."""
    g = np.linspace(0.0, 1.0, 48) ** (1.0 + 0.1 * seed)
    r, gg, b = np.meshgrid(g, g, g, indexing="ij")
    q = lambda x: np.round(np.clip(x, 0, 1) * 1023).astype(np.uint32)
    return (q(r) | (q(0.8 * gg + 0.1) << 10) | (q(b * b) << 20)).ravel(order="F").astype(np.uint32)


@pytest.mark.parametrize("view_transform", [1, 2, 6, 9])  # AgX, AgX_Punchy, Filmic_MediumContrast, Filmic_VeryHighContrast
def test_lut_view_transforms_match_reference_renderer(view_transform):
    """camera_desc_t::view_transform = AgX / Filmic (TonemapFilmic, TonemapRef.cpp:29-66): the 48^3 table comes from the
    reference through rc_set_view_lut; the tonemapped plane after rc_render and after the NLM denoiser is bit-identical,
    with a non-unit gamma on top.  Without the table the render call fails loudly.  (Without the oracle: a synthetic
    table, results checked against stored digests.)"""
    o = maybe_oracle()
    desc = scenes.cornell_box(80, 64)
    desc.camera.view_transform = view_transform
    desc.camera.gamma = 1.8
    desc.camera.exposure = 0.5
    pair = make_pair(desc)
    assert pair.cam.view_transform == view_transform
    with pytest.raises(Exception):
        pair.ctx.render(pair.make_pass(1))
    pair.ctx.set_view_lut(view_transform, o.view_lut(view_transform) if o else _synthetic_view_lut(view_transform))
    spp = 6
    ref, it = _ref_render(o, pair, spp)
    raw, it = _cuda_render(pair, spp)
    final = pair.ctx.readback(capi.RC_BUF_FINAL)
    assert final[..., :3].std() > 0.01
    rect = (0, 0, pair.w, pair.h)
    if ref is None:
        pair.ctx.denoise_nlm(rect, it)
        STORED.check(f"parity/lut/{view_transform}", raw, final, pair.ctx.readback(capi.RC_BUF_FINAL))
        pair.close()
        return
    assert bits_equal(raw, ref.pixels(1))
    ref_final = ref.pixels(0)
    assert bits_equal(final, ref_final), f"tonemapped plane: L-inf {np.abs(final - ref_final).max()}"
    ref.denoise(rect, it)
    pair.ctx.denoise_nlm(rect, it)
    assert bits_equal(pair.ctx.readback(capi.RC_BUF_FINAL), ref.pixels(0))
    ref.close()
    pair.close()


# (input channels, output channels) of the 16 convolutions (rt_unet.cuh unet_layer; skip tensors included)
UNET_SHAPES = [(9, 32), (32, 32), (32, 48), (48, 64), (64, 80), (80, 96), (96, 96), (160, 112), (112, 112), (160, 96),
               (96, 96), (128, 64), (64, 64), (73, 64), (64, 32), (32, 3)]


def unet_layers(o, seed=5):
    """The reference's weight set, or without the oracle a seeded one of the network's shapes."""
    if o is not None:
        return o.unet_layers()
    rng = np.random.default_rng(seed)
    return [((rng.standard_normal((co, ci, 3, 3)) * np.sqrt(2.0 / (9 * ci))).astype(np.float16),
             (rng.standard_normal(co) * 0.01).astype(np.float16)) for ci, co in UNET_SHAPES]


def test_unet_denoise_matches_reference_renderer():
    """RendererBase::DenoiseImage(pass, region) (SURVEY 8(f)-3, UNet half): same 8 spp accumulated on both sides
    (bit-identical), then the 16-pass UNet with the reference's own weight set handed over through rc_unet_set_weights.
    The fp32 path sums the same products in another order than the reference's 4-lane partial sums (and uses FMA), so the
    filtered linear image agrees to rounding noise, not bitwise: tolerance 2e-4 relative to (1 + |value|)."""
    o = maybe_oracle()
    for (w, h) in ((112, 80), (100, 70)):  # 112 = 7 x 16, 80 = 5 x 16; the second is not a multiple of 16
        pair = make_pair(scenes.cornell_box(w, h))
        spp = 8
        ref, it = _ref_render(o, pair, spp)
        noisy, it = _cuda_render(pair, spp)
        if ref is not None:
            assert bits_equal(noisy, ref.pixels(1))
            ref.denoise_unet((0, 0, w, h), it)
        pair.ctx.unet_set_weights(unet_layers(o))
        pair.ctx.denoise_unet((0, 0, w, h), flags=capi.RC_UNET_FP32)
        raw, final = pair.ctx.readback(capi.RC_BUF_RAW), pair.ctx.readback(capi.RC_BUF_FINAL)
        assert np.isfinite(raw).all()
        # the filter actually filtered: the output is not the noisy input
        assert np.abs(raw[..., :3] - pair.ctx.readback(capi.RC_BUF_FULL)[..., :3]).mean() > 1e-4
        if ref is None:
            STORED.check(f"parity/unet_fp32/{w}x{h}", noisy, raw, final)
        else:
            ref_raw, ref_final = ref.pixels(1), ref.pixels(0)
            err = np.abs(raw[..., :3] - ref_raw[..., :3]) / (1.0 + np.abs(ref_raw[..., :3]))
            assert err.max() <= 2e-4, f"{w}x{h}: UNet (fp32) filtered image differs: max rel {err.max():g}"
            assert np.abs(final[..., :3] - ref_final[..., :3]).max() <= 1e-3
            ref.close()
        pair.close()


def test_unet_tensor_core_path_matches_reference_renderer():
    """The same UNet through the tcgen05 path (fp16 operands, fp32 accumulation in TMEM, rt_unet_tc.cuh) against the
    reference's fp32 CPU filter.  Activations are rounded to fp16 between the 16 layers (as on the reference's own GPU
    path), so the bar is fp16-level agreement: max relative error 3e-2 of (1 + |value|), mean 2e-3, and > 40 dB PSNR
    against the fp32 device path on the tonemapped image.  (Without the oracle: a seeded weight set; the error bars
    against the reference's filter do not apply, the output is checked bitwise against its stored digest and must stay
    above 40 dB PSNR against the fp32 device path.)"""
    o = maybe_oracle()
    for (w, h) in ((160, 96), (100, 70)):
        pair = make_pair(scenes.cornell_box(w, h))
        spp = 8
        ref, it = _ref_render(o, pair, spp)
        _cuda_render(pair, spp)
        pair.ctx.unet_set_weights(unet_layers(o))
        pair.ctx.denoise_unet((0, 0, w, h), flags=capi.RC_UNET_FP32)
        f32_raw, f32_final = pair.ctx.readback(capi.RC_BUF_RAW), pair.ctx.readback(capi.RC_BUF_FINAL)
        if ref is not None:
            ref.denoise_unet((0, 0, w, h), it)
            ref_raw = ref.pixels(1)
            ref.close()
        pair.ctx.denoise_unet((0, 0, w, h), flags=capi.RC_UNET_TENSOR_CORES)
        raw, final = pair.ctx.readback(capi.RC_BUF_RAW), pair.ctx.readback(capi.RC_BUF_FINAL)
        assert np.isfinite(raw).all()
        mse = float(((final[..., :3] - f32_final[..., :3]) ** 2).mean())
        psnr = 10.0 * np.log10(1.0 / max(mse, 1e-12))
        print(f"unet tc {w}x{h}: PSNR vs fp32 path {psnr:.1f} dB")
        assert psnr > 40.0
        if o is None:
            STORED.check(f"parity/unet_tc/{w}x{h}", f32_raw, raw, final)
        else:
            err = np.abs(raw[..., :3] - ref_raw[..., :3]) / (1.0 + np.abs(ref_raw[..., :3]))
            print(f"unet tc {w}x{h}: max rel {err.max():.3g} mean rel {err.mean():.3g}")
            assert err.max() <= 3e-2 and err.mean() <= 2e-3, f"{w}x{h}: max rel {err.max():g}, mean rel {err.mean():g}"
        pair.close()
