"""Golden vectors (tests/golden/*.npz, made by tools/make_golden.py from the unmodified reference):
  CPU  - the oracle library reproduces them bit-for-bit (pins the oracle build), and the oracle's Cornell render agrees
         with the reference's own committed sample output samples/00_basic.tga when /root/reference is present
  GPU  - the CUDA path reproduces them bit-for-bit from the arrays stored IN the fixture (no oracle library needed for
         the trace stages; the shading stages additionally need the reference's PMJ02 table, which only the oracle has)
  GPU  - rc_render over the fixtures' arrays and the host layer's own path over small scenes render the planes stored in
         tests/golden/cuda_images.npz bit-for-bit (built-in sampler table; no oracle library needed)
"""
import ctypes as C
import glob
import os

import numpy as np
import pytest

from ray_b200 import capi, host, scenes
from ray_b200.cuda import HIT_DTYPE, RAY_DTYPE, SHADOW_DTYPE
from common import GOLDEN_ARRAYS as ARRAYS, STORED, maybe_oracle, render_golden, view_from_golden

DESCS = {"cornell_48": lambda: scenes.cornell_box(48, 48), "zoo_64x48": lambda: scenes.material_zoo(64, 48)}
GOLDEN = sorted(p for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))
                if os.path.splitext(os.path.basename(p))[0] in DESCS)
# Planes the CUDA path rendered when they were stored (tools/make_golden.py --cuda-images): the fixture scenes over the
# reference-built arrays, and scenes built by the product's own host layer, both with the built-in sampler table.  Small
# frames: float planes of Monte-Carlo noise barely compress.
CUDA_IMAGES = os.path.join(os.path.dirname(__file__), "golden", "cuda_images.npz")
GOLDEN_SPP = 4
HOST_CASES = {
    "host_cornell": (lambda: scenes.cornell_box(32, 32), 8),
    "host_zoo": (lambda: scenes.material_zoo(32, 24), 4),
    "host_textured": (lambda: scenes.textured(32, 24), 4),
    "host_envmap_zoo": (lambda: scenes.envmap_zoo(32, 24), 4),
    "host_hall_small": (lambda: scenes.hall("principled", 64, 36, floor_res=24, n_columns=4, col_seg=8, col_rings=6,
                                            extra_lights=10), 4),
    "host_instanced": (lambda: scenes.instanced(16, 400, 32, 32), 4),
}


def render_host_case(name):
    """RendererBase::RenderScene over a scene built by the host layer; returns the planes a caller reads back (the
    Cornell case also through the NLM denoiser, the zoo case also its AOVs) and the counters."""
    make, spp = HOST_CASES[name]
    desc = make()
    w, h = desc.width, desc.height
    r = host.Renderer(w, h)
    s = scenes.build(desc, r.create_scene())
    it = r.render(s, (0, 0, w, h), 0, spp)
    out = {"raw": r.pixels(host.RAW), "final": r.pixels(host.FINAL)}
    if name == "host_zoo":
        out["base_color"], out["depth_normals"] = r.pixels(host.BASE_COLOR), r.pixels(host.DEPTH_NORMALS)
    if name == "host_cornell":
        r.denoise((0, 0, w, h), it)
        out["nlm_raw"], out["nlm_final"] = r.pixels(host.RAW), r.pixels(host.FINAL)
    counters = r.counters()
    s.close()
    r.close()
    return out, counters, spp * w * h


def _name(path):
    return os.path.splitext(os.path.basename(path))[0]


def _by_xy(a):
    return a[np.argsort(a["xy"], kind="stable")]


@pytest.mark.parametrize("path", GOLDEN, ids=_name)
def test_oracle_reproduces_golden(path, oracle_mod):
    g = np.load(path)
    desc = DESCS[_name(path)]()
    w, h = [int(x) for x in g["wh"]]
    it = int(g["iteration"])
    sc = scenes.build(desc, oracle_mod.Scene(wide=True))
    v = sc.view()
    for name in ARRAYS:
        a = getattr(v, name)
        n = a.count * a.stride
        got = np.ctypeslib.as_array(C.cast(a.ptr, C.POINTER(C.c_uint8)), shape=(n,)) if n else np.zeros(0, np.uint8)
        assert got.tobytes() == g["arr_" + name].tobytes(), f"scene array {name} drifted"
    rays, hits = sc.generate_primary_rays(w, h, (0, 0, w, h), it)
    assert rays.tobytes() == g["primary_rays"].tobytes()
    _, hits1 = sc.trace_rays(it, rays, hits, False)
    assert hits1.tobytes() == g["primary_hits_out"].tobytes()
    temp = np.zeros((h, w, 4), np.float32)
    sec, sh, _, _ = sc.shade(w, h, it, True, 0, g["primary_rays"], g["primary_hits_out"], temp)
    assert sec.tobytes() == g["secondary_rays"].tobytes() and sh.tobytes() == g["shadow_rays"].tobytes()
    assert temp.tobytes() == g["temp_after_primary_shade"].tobytes()
    ref = oracle_mod.Renderer(capi.RT_REFERENCE, w, h)
    k = 0
    for _ in range(4):
        k = ref.render(sc, (0, 0, w, h), k)
    assert ref.pixels(1).tobytes() == g["image_raw_4spp"].tobytes()
    sc.close()


def _read_tga(path):
    b = open(path, "rb").read()
    idlen, _, imgtype = b[0], b[1], b[2]
    w, h, bpp, desc = int.from_bytes(b[12:14], "little"), int.from_bytes(b[14:16], "little"), b[16], b[17]
    assert imgtype == 2 and bpp in (24, 32)
    px = np.frombuffer(b, np.uint8, count=w * h * (bpp // 8), offset=18 + idlen).reshape(h, w, bpp // 8)
    if not (desc & 0x20):
        px = px[::-1]
    return px[..., 2::-1].astype(np.float32) / 255.0  # BGR -> RGB


@pytest.mark.slow
def test_oracle_cornell_agrees_with_the_references_committed_sample_image(oracle_mod):
    """reference samples/00_basic.tga is the committed output of samples/00_basic/main.cpp (256x256, 64 spp): the
    oracle's render of ray_b200.scenes.cornell_box() must look like it (PSNR; the sample was rendered by whichever backend
    the factory picked, so it is a statistical, not a bitwise, anchor)."""
    tga = "/root/reference/samples/00_basic.tga"
    if not os.path.exists(tga):
        pytest.skip("/root/reference is not present on this box")
    want = _read_tga(tga)
    desc = scenes.cornell_box(256, 256)
    sc = scenes.build(desc, oracle_mod.Scene(wide=False))
    ref = oracle_mod.Renderer(capi.RT_REFERENCE, 256, 256)
    ref.render_mt(sc, 64, os.cpu_count() or 1, 32)
    got = ref.pixels(0)[..., :3]
    mse = float(((np.clip(got, 0, 1) - want) ** 2).mean())
    psnr = 10.0 * np.log10(1.0 / max(mse, 1e-12))
    assert psnr > 28.0, f"PSNR vs samples/00_basic.tga = {psnr:.2f} dB"
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=_name)
def test_cuda_trace_reproduces_golden_without_the_oracle(path):
    """Closest-hit trace (primary, and bounce 1 with analytic lights) from the fixture's own scene arrays: no oracle
    library involved at all.  (The sampler table is only touched by transparency, which these scenes' rays with a
    zero table would still have to agree on -- the fixture's scenes have no transparent hits on these rays.)"""
    from ray_b200 import cuda
    g = np.load(path)
    keep = []
    v = view_from_golden(g, keep)
    w, h = [int(x) for x in g["wh"]]
    ctx = cuda.Context(0)
    ctx.resize(w, h)
    ctx.upload_tables(np.zeros(32 * 4096 * 2, np.uint32), g["filter_table"])
    ctx.upload_scene(v)
    cam = capi.rc_camera.from_buffer_copy(g["cam"].tobytes())
    p = ctx.make_pass(cam, (0, 0, w, h), int(g["iteration"]))
    _, hits = ctx.stage_trace_rays(p, g["primary_rays"].view(RAY_DTYPE), g["primary_hits_in"].view(HIT_DTYPE), False)
    assert hits.tobytes() == g["primary_hits_out"].tobytes()
    sec = g["secondary_rays"].view(RAY_DTYPE)
    if _name(path) != "zoo_64x48":  # the zoo has an alpha-blended sphere: its secondary rays may cross it (needs PMJ)
        hits0 = np.zeros(len(sec), dtype=HIT_DTYPE)
        hits0["obj_index"] = -1
        hits0["prim_index"] = -1
        hits0["t"] = np.float32(3.402823466e+30)
        hits0["v"] = -1.0
        _, hits2 = ctx.stage_trace_rays(p, sec, hits0, True)
        assert hits2.tobytes() == g["secondary_hits_out"].tobytes()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=_name)
def test_cuda_shading_and_image_reproduce_golden(path):
    """Primary shade, shadow rays and a 4-spp image from the fixture's arrays against the reference's outputs stored in
    it; those need the reference's PMJ02 table, so without the oracle library the same stages run with the built-in
    table and are checked against the digests stored in tests/golden/cuda_digests.json."""
    from ray_b200 import cuda
    o = maybe_oracle()
    g = np.load(path)
    keep = []
    v = view_from_golden(g, keep)
    w, h = [int(x) for x in g["wh"]]
    it = int(g["iteration"])
    ctx = cuda.Context(0)
    ctx.resize(w, h)
    ctx.upload_tables(o.pmj_table() if o else host.builtin_sampler_table(), g["filter_table"])
    ctx.upload_scene(v)
    cam = capi.rc_camera.from_buffer_copy(g["cam"].tobytes())
    p = ctx.make_pass(cam, (0, 0, w, h), it)
    ctx.fill_temp((0, 0, 0, 0))
    sec, sh = ctx.stage_shade(p, True, 0, g["primary_rays"].view(RAY_DTYPE), g["primary_hits_out"].view(HIT_DTYPE))
    if o is None:
        key = f"golden/{_name(path)}"
        STORED.check(f"{key}/primary_shade", _by_xy(sec), _by_xy(sh), ctx.readback(capi.RC_BUF_TEMP))
        ctx.stage_trace_shadow_rays(p, _by_xy(sh), cam.clamp_direct)
        STORED.check(f"{key}/primary_shadow", ctx.readback(capi.RC_BUF_TEMP))
        ctx.close()
        return
    assert _by_xy(sec).tobytes() == _by_xy(g["secondary_rays"].view(RAY_DTYPE)).tobytes()
    assert _by_xy(sh).tobytes() == _by_xy(g["shadow_rays"].view(SHADOW_DTYPE)).tobytes()
    assert ctx.readback(capi.RC_BUF_TEMP).tobytes() == g["temp_after_primary_shade"].tobytes()
    ctx.stage_trace_shadow_rays(p, g["shadow_rays"].view(SHADOW_DTYPE), cam.clamp_direct)
    assert ctx.readback(capi.RC_BUF_TEMP).tobytes() == g["temp_after_primary_shadow"].tobytes()
    ctx.clear((0, 0, 0, 0))
    for i in range(1, 5):
        ctx.render(ctx.make_pass(cam, (0, 0, w, h), i))
    assert ctx.readback(capi.RC_BUF_RAW).tobytes() == g["image_raw_4spp"].tobytes()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=_name)
def test_cuda_render_of_the_fixture_scene_is_unchanged(path):
    """The whole wavefront (rc_render, ray sort on) over the fixture's reference-built arrays renders the stored planes,
    bit for bit."""
    g = np.load(path)
    want = np.load(CUDA_IMAGES)
    w, h = [int(x) for x in g["wh"]]
    got, c = render_golden(g, GOLDEN_SPP)
    assert c["primary_rays"] == GOLDEN_SPP * w * h
    for plane, a in got.items():
        assert np.isfinite(a).all()
        ref = want[f"{_name(path)}_{plane}"]
        assert a.tobytes() == ref.tobytes(), f"{plane}: L-inf {np.abs(a - ref).max()}"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(HOST_CASES))
def test_host_layer_render_is_unchanged(name):
    """The product path (host layer: own SAH BVH8, light tree, camera, tables -> C-ABI -> kernels) renders the stored
    planes, bit for bit."""
    want = np.load(CUDA_IMAGES)
    got, c, primary = render_host_case(name)
    assert c["primary_rays"] == primary
    for plane, a in got.items():
        assert np.isfinite(a).all()
        ref = want[f"{name}_{plane}"]
        assert a.tobytes() == ref.tobytes(), f"{plane}: L-inf {np.abs(a - ref).max()}"
