"""GPU tests of the product's public path: host layer (Cuda::Renderer / Cuda::Scene, own BVH + light-tree builders)
-> C-ABI -> kernels, compared with the reference's RendererRef fed the SAME scene description.

The host layer's acceleration structures are not the reference's (different SAH splits, different light tree), so the
images cannot be bit-identical: a different light tree changes which light NEE picks for a given random number.  The
checks are therefore (a) geometric -- first-hit depth and normals are deterministic functions of camera + geometry and
must agree everywhere but at exact-t ties / silhouette pixels, (b) radiometric -- the converged images must agree
(block-averaged relative error), with the reference's own PMJ02 table uploaded so both sides integrate with the same
sample sequences.  Without the oracle library (built from the reference's sources) the same renders run with the built-in
sampler table and are checked against the digests stored in tests/golden/cuda_digests.json.
"""
import numpy as np
import pytest

from ray_b200 import capi, host, scenes
from common import STORED, maybe_oracle

pytestmark = pytest.mark.gpu


def _block_mean(img, b):
    h, w = img.shape[:2]
    h2, w2 = h // b * b, w // b * b
    return img[:h2, :w2, :3].reshape(h2 // b, b, w2 // b, b, 3).mean(axis=(1, 3))


@pytest.mark.parametrize("name,make,spp", [
    ("cornell", lambda: scenes.cornell_box(96, 96), 256),
    ("zoo", lambda: scenes.material_zoo(128, 96, filter=capi.FILTER_BOX), 192),
    ("hall_small", lambda: scenes.hall("principled", 128, 72, floor_res=32, n_columns=6, col_seg=10, col_rings=6,
                                       extra_lights=6), 192),
    ("instanced", lambda: scenes.instanced(25, 300, 96, 96), 128),
    ("textured", lambda: scenes.textured(96, 72), 192),
    ("envmap_zoo", lambda: scenes.envmap_zoo(96, 72), 192),
])
def test_host_layer_matches_reference_renderer(name, make, spp):
    o = maybe_oracle()
    desc = make()
    w, h = desc.width, desc.height
    r = host.Renderer(w, h)
    if o is not None:
        r.set_sampler_table(o.pmj_table())
    s = scenes.build(desc, r.create_scene())
    it = r.render(s, (0, 0, w, h), 0, spp)
    assert it == spp
    raw, dn, base = r.pixels(host.RAW), r.pixels(host.DEPTH_NORMALS), r.pixels(host.BASE_COLOR)
    assert np.isfinite(raw).all()
    c = r.counters()
    assert c["primary_rays"] == spp * w * h
    if o is None:
        STORED.check(f"host/{name}", raw, dn, base)
        s.close()
        r.close()
        return
    # reference: its own scene builder (BVH2) + RendererRef, multi-threaded over tiles
    osc = scenes.build(desc, o.Scene(wide=False))
    ref = o.Renderer(capi.RT_REFERENCE, w, h)
    ref.render_mt(osc, spp, 8, 32)
    ref_raw, ref_dn, ref_base = ref.pixels(1), ref.pixels(3), ref.pixels(2)
    ref.close()

    # (a) geometry: depth (w channel of the depth-normals AOV) and shading normals, averaged over spp
    d_ref, d = ref_dn[..., 3], dn[..., 3]
    rel = np.abs(d - d_ref) / np.maximum(np.abs(d_ref), 1e-3)
    frac_bad = float((rel > 1e-3).mean())
    assert frac_bad < 0.03, f"{name}: {frac_bad:.4f} of pixels disagree on first-hit depth"
    n_err = np.abs(dn[..., :3] - ref_dn[..., :3]).max(axis=-1)
    assert float((n_err > 2e-2).mean()) < 0.04, f"{name}: normals AOV differs"
    assert float((np.abs(base - ref_base).max(axis=-1) > 2e-2).mean()) < 0.04, f"{name}: base colour AOV differs"

    # (b) radiometry: block-averaged converged radiance
    bm, bm_ref = _block_mean(raw, 8), _block_mean(ref_raw, 8)
    scale = max(float(bm_ref.mean()), 1e-3)
    rel_rmse = float(np.sqrt(((bm - bm_ref) ** 2).mean())) / scale
    mean_rel = abs(float(bm.mean()) - float(bm_ref.mean())) / scale
    assert mean_rel < 0.02, f"{name}: mean radiance differs by {mean_rel:.3%}"
    assert rel_rmse < 0.12, f"{name}: block-averaged radiance rel. RMSE {rel_rmse:.3f}"
    s.close()
    r.close()
    osc.close()


def test_regions_and_resize():
    """RenderScene over disjoint regions with their own iteration counters (test_complex_mat5_regions pattern) and an
    idempotent Resize (reference tests/test_shading.cpp:103-106) give the same image as one full-frame region."""
    desc = scenes.cornell_box(64, 64)
    r = host.Renderer(64, 64)
    s = scenes.build(desc, r.create_scene())
    r.resize(32, 32)
    r.resize(64, 64)
    for _ in range(3):
        pass
    it = r.render(s, (0, 0, 64, 64), 0, 6)
    full = r.pixels(host.RAW)
    r.clear((0, 0, 0, 0))
    its = [0, 0, 0, 0]
    rects = [(0, 0, 32, 32), (32, 0, 32, 32), (0, 32, 32, 32), (32, 32, 32, 32)]
    for k in range(6):
        for i, rect in enumerate(rects):
            its[i] = r.render(s, rect, its[i], 1)
    tiled = r.pixels(host.RAW)
    assert it == 6 and its == [6, 6, 6, 6]
    assert full.tobytes() == tiled.tobytes()
    s.close()
    r.close()


def test_denoise_image_through_the_renderer_api():
    """RendererBase::DenoiseImage(region) on the stand-alone renderer: runs without an ILog error, smooths the image
    (lower high-frequency energy than the noisy input) and agrees with the reference's NLM of ITS render of the same scene
    on the image mean (the two renders are statistically, not bitwise, equal: different BVH builders)."""
    o = maybe_oracle()
    desc = scenes.cornell_box(96, 96)
    w, h, spp = 96, 96, 16
    r = host.Renderer(w, h)
    s = scenes.build(desc, r.create_scene())
    it2 = r.render(s, (0, 0, w, h), 0, spp)
    noisy = r.pixels(host.FINAL)[..., :3].copy()
    r.denoise((0, 0, w, h), it2)
    den = r.pixels(host.FINAL)[..., :3].copy()
    assert np.isfinite(den).all()

    def hf(a):
        return float(np.abs(a[1:, 1:] - a[:-1, 1:]).mean() + np.abs(a[1:, 1:] - a[1:, :-1]).mean())

    assert hf(den) < 0.8 * hf(noisy)
    assert r.stats_us()[8] > 0  # stats_t::time_denoise_us
    s.close()
    r.close()
    if o is None:
        STORED.check("host/nlm_denoise", noisy, den)
        return
    osc = scenes.build(desc, o.Scene(wide=False))
    ref = o.Renderer(capi.RT_REFERENCE, w, h)
    it = 0
    for _ in range(spp):
        it = ref.render(osc, (0, 0, w, h), it)
    ref.denoise((0, 0, w, h), it)
    ref_img = ref.pixels(0)[..., :3].copy()
    assert abs(float(den.mean()) - float(ref_img.mean())) < 0.03 * float(ref_img.mean())
    ref.close()
    osc.close()


def test_unsupported_features_are_reported_not_faked():
    """A material that names a texture the scene does not have must fail the upload, not render untextured."""
    desc = scenes.cornell_box(16, 16)
    desc.materials[0] = ("node", capi.rs_shading_node_desc.default(type=capi.NODE_DIFFUSE, base_color=(0.5, 0.5, 0.5)))
    r = host.Renderer(16, 16)
    s = scenes.build(desc, r.create_scene())
    s.add_material_node(capi.rs_shading_node_desc.default(type=capi.NODE_DIFFUSE, base_texture=(1 << 28) | 7))
    with pytest.raises(host.HostError):
        r.render(s, (0, 0, 16, 16), 0, 1)
        r.check()
    s.close()
    r.close()


def test_moved_instances_refresh_only_the_top_level():
    """SetMeshInstanceTransform + Finalize: the renderer re-sends the TLAS, instance and light records only
    (rc_update_instances), and the image equals the one a complete upload of the same scene state gives, bit for bit."""
    from ray_b200 import cuda
    desc = scenes.instanced(25, 3000, 160, 120)
    w, h = desc.width, desc.height
    r = host.Renderer(w, h)
    lib = cuda.load_library()
    ctx = r.native_context()
    s = scenes.build(desc, r.create_scene())
    r.render(s, (0, 0, w, h), 0, 2)
    one_full = total = lib.rc_scene_upload_bytes(ctx)
    assert one_full > 0
    before = r.pixels(host.RAW)

    for step in range(1, 4):  # a few animation frames
        for i in (1, 7, 13):
            x = np.asarray(desc.instances[i][1], dtype=np.float32).reshape(4, 4).copy()
            x[3, :3] += np.float32(0.15 * step)  # column-major: translation lives in the last column = row 3 here
            s.set_mesh_instance_transform(i, x)
        s.finalize()
        r.clear()
        r.render(s, (0, 0, w, h), 0, 2)
        moved = r.pixels(host.RAW)
        sent = lib.rc_scene_upload_bytes(ctx) - total
        assert 0 < sent < 0.05 * one_full, "a transform edit re-sent the geometry"
        total += sent
        r.invalidate_scene()  # complete upload of the same state
        r.clear()
        r.render(s, (0, 0, w, h), 0, 2)
        again = r.pixels(host.RAW)
        sent = lib.rc_scene_upload_bytes(ctx) - total
        assert sent >= 0.9 * one_full
        total += sent
        assert np.array_equal(moved.view(np.uint32), again.view(np.uint32))
        assert not np.array_equal(moved, before)
    s.close()
    r.close()
