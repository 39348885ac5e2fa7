"""GPU tests of lightmap baking: the texture-space (Geo) camera, the pass flags and the L1 SH output
(semantics in include/ray_cuda.h).  The reference's code for these is not part of this repository, so the checks are
analytic (rasterisation against numpy, furnace values, SH of known radiance) and self-consistency (determinism, the
flag decomposition, Geo bake vs a perspective render of the same surface)."""
import ctypes as C

import numpy as np
import pytest

from ray_b200 import capi, cuda, host, scenes
from common import HostPair

pytestmark = pytest.mark.gpu

SKIP_D, SKIP_I = capi.RC_RENDER_SKIP_DIRECT, capi.RC_RENDER_SKIP_INDIRECT
LONLY, NOBG, SH = capi.RC_RENDER_LIGHTING_ONLY, capi.RC_RENDER_NO_BACKGROUND, capi.RC_RENDER_OUTPUT_SH
Y0, Y1 = 0.282095, 0.488603


# ---- scenes ---------------------------------------------------------------------------------------------------------
def _cam(geo_instance=None, **kw):
    if geo_instance is not None:
        kw.update(type=capi.CAM_GEO, mi_index=geo_instance)
    kw.setdefault("filter", capi.FILTER_BOX)
    kw.setdefault("origin", (0.0, 4.0, 0.0))
    kw.setdefault("fwd", (0.0, -1.0, 0.0))
    kw.setdefault("up", (0.0, 0.0, -1.0))
    return capi.rs_camera_desc.default(**kw)


def _plane(half, y=0.0):
    """Quad [-half, half]^2 at height y, normal +y (winding agrees), uv = ((x + half), (z + half)) / (2 half)."""
    rows = [[-half, y, -half, 0, 1, 0, 0, 0], [half, y, -half, 0, 1, 0, 1, 0], [half, y, half, 0, 1, 0, 1, 1],
            [-half, y, half, 0, 1, 0, 0, 1]]
    return scenes.MeshDesc(np.asarray(rows, np.float32), np.asarray([0, 2, 1, 0, 3, 2], np.uint32), [])


def plane_scene(w, h, albedo=0.5, env=(0.0, 0.0, 0.0), back=(0.0, 0.0, 0.0), occluder=False, light=None,
                geo=True, cam=None, cast_shadow=True):
    """A 4 m plane (instance 0, triangles 0..1), optionally a floating grey quad that casts a shadow but is invisible to
    camera rays (instance 1) and a light.  geo=True: a Geo camera baking the plane."""
    s = scenes.SceneDesc(name="bake", width=w, height=h, env_col=env, back_col=back)
    m = s.add_node(type=capi.NODE_DIFFUSE, base_color=(albedo, albedo, albedo))
    p = _plane(2.0)
    p.groups = [(m, m, 0, 6)]
    s.meshes.append(p)
    s.instances.append((0, scenes.IDENTITY.T.reshape(16), {}))
    if occluder:
        o = _plane(0.5, 1.5)
        o.groups = [(m, m, 0, 6)]
        s.meshes.append(o)
        xf = np.eye(4, dtype=np.float32)
        xf[:3, 3] = (0.4, 0.0, -0.3)
        s.instances.append((1, xf.T.reshape(16), {"camera_visibility": False}))
    if light == "sphere":
        s.lights.append(("sphere", capi.rs_sphere_light_desc(c=capi.rs_light_common.default(
            color=(40.0, 40.0, 40.0), cast_shadow=int(cast_shadow)), position=(-0.3, 4.0, 0.2), radius=0.3)))
    elif light is not None:  # a direction the light travels
        s.lights.append(("directional", capi.rs_directional_light_desc(
            c=capi.rs_light_common.default(color=(2.0, 2.0, 2.0)), direction=tuple(float(x) for x in light), angle=1.0)))
    s.camera = cam or _cam(0 if geo else None)
    return s


def atlas_scene(w, h, n=240, seed=5):
    """Instance 1 of mesh 1 (triangles 2 ..): a seeded uv atlas with overlapping charts, slivers, degenerate
    triangles, both windings and triangles partly outside [0,1]^2, under a non-identity transform.  Nothing reaches
    u > 0.85, so the right edge of the lightmap stays uncovered."""
    rng = np.random.RandomState(seed)
    s = plane_scene(w, h)
    m = 0
    pos = rng.uniform(-1.0, 1.0, (n, 3, 3))
    nrm = rng.normal(size=(n, 3, 3))
    nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    uv = np.empty((n, 3, 2))
    for i in range(n):
        kind = i % 6
        c = rng.uniform((-0.1, -0.1), (0.55, 1.1))
        if kind == 0:  # big chart triangles (overlap each other)
            uv[i] = c + rng.uniform(-0.3, 0.3, (3, 2))
        elif kind == 1:  # sliver
            d = rng.normal(size=2)
            d /= np.linalg.norm(d)
            uv[i] = c + np.outer([0.0, 0.15, 0.3], d) + rng.normal(scale=1e-3, size=(3, 2))
        elif kind == 2:  # degenerate: repeated corner
            uv[i] = c + rng.uniform(-0.1, 0.1, (3, 2))
            uv[i, 2] = uv[i, 0]
        else:  # small triangles of either winding
            uv[i] = c + rng.uniform(-0.05, 0.05, (3, 2))
    attrs = np.concatenate([pos, nrm, uv], axis=-1).reshape(-1, 8).astype(np.float32)
    s.meshes.append(scenes.MeshDesc(attrs, np.arange(3 * n, dtype=np.uint32), [(m, m, 0, 3 * n)]))
    ang = 0.7
    xf = np.array([[np.cos(ang) * 1.5, 0, np.sin(ang) * 1.5, 0.3], [0, 0.8, 0, -0.2],
                   [-np.sin(ang) * 1.5, 0, np.cos(ang) * 1.5, 0.5], [0, 0, 0, 1]], np.float32)
    s.instances.append((1, xf.T.reshape(16), {}))
    s.camera = _cam(1)
    return s, xf


def _pair(desc):
    return HostPair(desc)


def _bake(pair, spp, flags=0, geo=(0, 0, 2), rect=None, clear=True):
    if clear:
        pair.ctx.clear((0, 0, 0, 0))
    for i in range(1, spp + 1):
        pair.ctx.render(pair.ctx.make_pass(pair.cam, rect or (0, 0, pair.w, pair.h), i, flags, geo))
    return pair.ctx.readback(capi.RC_BUF_RAW)


def _view_arrays(view):
    def arr(a, dtype, cols):
        return np.ctypeslib.as_array(C.cast(a.ptr, C.POINTER(C.c_float if dtype == np.float32 else C.c_uint32)),
                                     shape=(a.count * a.stride // 4,)).view(dtype).reshape(-1, cols).copy()
    return arr(view.vertices, np.float32, 11), arr(view.vtx_indices, np.uint32, 1).reshape(-1)


# ---- 1. rasterisation vs numpy --------------------------------------------------------------------------------------
def test_geo_rays_match_numpy_rasterisation():
    w, h = 64, 48
    desc, xf = atlas_scene(w, h)
    pair = _pair(desc)
    verts, vidx = _view_arrays(pair.view)
    first, count = 2, len(desc.meshes[1].indices) // 3
    tri = vidx.reshape(-1, 3)[first:first + count]
    uv = verts[tri][:, :, 9:11].astype(np.float64) * [w, h]  # texel units
    P = verts[tri][:, :, 0:3].astype(np.float64)
    Nv = verts[tri][:, :, 3:6].astype(np.float64)
    area2 = ((uv[:, 1, 0] - uv[:, 0, 0]) * (uv[:, 2, 1] - uv[:, 0, 1]) -
             (uv[:, 1, 1] - uv[:, 0, 1]) * (uv[:, 2, 0] - uv[:, 0, 0]))
    ok_tri = np.abs(area2) >= 2e-12
    inv_t = np.linalg.inv(xf.astype(np.float64)).T
    lo, hi = uv.min(axis=1), uv.max(axis=1)

    def edge_dist(p):  # signed distance of point p to the three edges of every triangle, inside positive
        d = []
        for a, b in ((1, 2), (2, 0), (0, 1)):
            e = uv[:, b] - uv[:, a]
            cr = e[:, 0] * (p[1] - uv[:, a, 1]) - e[:, 1] * (p[0] - uv[:, a, 0])
            d.append(np.sign(area2) * cr / np.maximum(np.linalg.norm(e, axis=1), 1e-30))
        return np.min(d, axis=0)

    # texels whose box lies strictly inside a triangle always emit; texels no triangle box touches never do
    always, never = np.zeros((h, w), bool), np.ones((h, w), bool)
    for y in range(h):
        for x in range(w):
            corners = [(x, y), (x + 1, y), (x, y + 1), (x + 1, y + 1)]
            inside = np.all([edge_dist(np.array(c, float)) > 1e-3 for c in corners], axis=0) & ok_tri
            always[y, x] = inside.any()
            never[y, x] = not ((lo[:, 0] <= x + 1 + 1e-3) & (hi[:, 0] >= x - 1e-3) & (lo[:, 1] <= y + 1 + 1e-3) &
                               (hi[:, 1] >= y - 1e-3)).any()
    assert always.sum() > 50 and never.sum() > 20

    pair.ctx.reset_stats()
    total = 0
    for it in (1, 2, 7):
        pair.ctx.clear()  # every texel active: the render below marks them converged for later iterations
        p = pair.ctx.make_pass(pair.cam, (0, 0, w, h), it, 0, (1, first, count))
        rays, hits = pair.ctx.stage_generate_geo_rays(p)
        total += len(rays)
        x, y = rays["xy"] >> 16, rays["xy"] & 0xffff
        emitted = np.zeros((h, w), bool)
        emitted[y, x] = True
        assert len(np.unique(rays["xy"])) == len(rays)
        assert emitted[always].all() and not emitted[never].any()
        assert (hits["obj_index"] == 1).all() and (hits["t"] == 0).all()
        k = hits["prim_index"] - first
        assert ((k >= 0) & (k < count)).all() and ok_tri[k].all()
        u, v = hits["u"].astype(np.float64), hits["v"].astype(np.float64)
        wgt = np.stack([1 - u - v, u, v], axis=1)
        assert (wgt >= -1e-5).all()
        pt = np.einsum("nk,nkc->nc", wgt, uv[k])
        assert ((pt[:, 0] >= x - 1e-3) & (pt[:, 0] <= x + 1 + 1e-3) & (pt[:, 1] >= y - 1e-3) &
                (pt[:, 1] <= y + 1 + 1e-3)).all()
        for i in range(len(rays)):  # the winner is the lowest-indexed containing triangle
            d = edge_dist(pt[i])[:k[i]]
            assert not (ok_tri[:k[i]] & (d > 1e-4)).any(), (i, k[i])
        Pw = (np.einsum("nk,nkc->nc", wgt, P[k]) @ xf[:3, :3].T.astype(np.float64)) + xf[:3, 3]
        Nw = np.einsum("nk,nkc->nc", wgt, Nv[k]) @ inv_t[:3, :3].T
        Nw /= np.linalg.norm(Nw, axis=1, keepdims=True)
        scale = np.abs(Pw).max()
        np.testing.assert_allclose(rays["o"], Pw, rtol=1e-5, atol=1e-5 * scale)
        np.testing.assert_allclose(rays["d"], -Nw, rtol=1e-5, atol=1e-5)
        assert (rays["cone_spread"] == 0).all() and (rays["cone_width"] > 0).all()
        # the render of the same pass emits the same rays
        pair.ctx.clear()
        before = pair.ctx.counters()["primary_rays"]
        pair.ctx.render(p)
        assert pair.ctx.counters()["primary_rays"] - before == len(rays)
    assert total > 0
    pair.close()


# ---- 2. determinism ----------------------------------------------------------------------------------------------------
def test_geo_bake_is_deterministic_and_tiles_match_the_full_frame():
    w, h, spp = 40, 32, 6
    desc, _ = atlas_scene(w, h)
    desc.lights.append(("sphere", capi.rs_sphere_light_desc(c=capi.rs_light_common.default(color=(30.0, 30.0, 30.0)),
                                                            position=(0.0, 3.0, 0.0), radius=0.3)))
    pair = _pair(desc)
    geo = (1, 2, len(desc.meshes[1].indices) // 3)
    outs = []
    for _ in range(2):
        raw = _bake(pair, spp, SH, geo)
        outs.append((raw, [pair.ctx.readback(b) for b in (capi.RC_BUF_SH_R, capi.RC_BUF_SH_G, capi.RC_BUF_SH_B)]))
    assert outs[0][0].tobytes() == outs[1][0].tobytes()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(outs[0][1], outs[1][1]))
    assert (outs[0][0][..., 3] > 0).sum() > 100
    pair.ctx.clear()
    tiles = [(0, 0, 24, 16), (24, 0, 16, 16), (0, 16, 24, 16), (24, 16, 16, 16)]
    for t in tiles:  # each tile with its own iteration counter, like separate RegionContexts
        for i in range(1, spp + 1):
            pair.ctx.render(pair.ctx.make_pass(pair.cam, t, i, SH, geo))
    assert pair.ctx.readback(capi.RC_BUF_RAW).tobytes() == outs[0][0].tobytes()
    assert pair.ctx.readback(capi.RC_BUF_SH_G).tobytes() == outs[0][1][1].tobytes()
    pair.close()


# ---- 3. furnace ----------------------------------------------------------------------------------------------------------
def test_geo_furnace():
    w = h = 16
    spp = 128
    pair = _pair(plane_scene(w, h, albedo=0.5, env=(1.0, 1.0, 1.0), back=(1.0, 1.0, 1.0)))
    interior = (slice(1, h - 1), slice(1, w - 1))
    base = _bake(pair, spp)
    lonly = _bake(pair, spp, LONLY)
    direct = _bake(pair, spp, SKIP_I)
    indirect = _bake(pair, spp, SKIP_D)
    for img, want in ((base, 0.5), (lonly, 1.0)):
        rgb = img[interior][..., :3]
        assert abs(rgb.mean() - want) < 0.02 * want, rgb.mean()
        assert np.abs(rgb - want).max() < 0.25 * want
    assert (base[..., 3] == 1.0).all() and (indirect[..., 3] == 1.0).all()
    assert direct.tobytes() == base.tobytes()
    assert (indirect[..., :3] == 0.0).all()
    pair.close()


# ---- 4. decomposition -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["persp", "geo_floor"])
def test_flag_decomposition(mode):
    desc = scenes.cornell_box(48, 48)
    geo = None
    if mode == "geo_floor":  # the floor quad: triangles 0..1 of the only mesh, uv [0,1]^2
        desc.camera = _cam(0)
        geo = (0, 0, 2)
    pair = _pair(desc)
    for it in (1, 5):
        out = {}
        for name, f in (("full", 0), ("e0", SKIP_D | SKIP_I), ("direct", SKIP_I), ("indirect", SKIP_D)):
            pair.ctx.clear()
            pair.ctx.render(pair.ctx.make_pass(pair.cam, (0, 0, pair.w, pair.h), it, f, geo))
            out[name] = pair.ctx.readback(capi.RC_BUF_RAW)[..., :3].astype(np.float64)
        lhs, rhs = out["full"] + out["e0"], out["direct"] + out["indirect"]
        assert np.isfinite(lhs).all()
        assert (np.abs(lhs - rhs) <= 1e-5 * np.abs(rhs) + 1e-6).all(), np.abs(lhs - rhs).max()
        assert out["indirect"].sum() > 0 and out["direct"].sum() > 0
    pair.close()


# ---- 5. Geo vs perspective -----------------------------------------------------------------------------------------------
def test_geo_bake_matches_a_perspective_render():
    n, spp = 96, 256
    half_extent, height = 1.5, 4.0
    fov = float(np.degrees(2 * np.arctan(half_extent / height)))
    persp = _pair(plane_scene(n, n, occluder=True, light="sphere", geo=False, cam=_cam(None, fov=fov)))
    img = _bake(persp, spp)[..., :3]
    bake_n = 64
    bake = _pair(plane_scene(bake_n, bake_n, occluder=True, light="sphere"))
    tex = _bake(bake, spp)[..., :3]
    # image right = +x, down = +z; u = (x + 2) / 4, v = (z + 2) / 4.  The view [-1.5, 1.5]^2 is texels [8, 56) of the
    # bake, and an 8x8 pixel block (0.25 m) covers exactly 4x4 texels: both block means integrate the same area
    b, tb = 8, 4
    nb = n // b
    want = img.reshape(nb, b, nb, b, 3).mean(axis=(1, 3))
    got = tex[8:56, 8:56].reshape(nb, tb, nb, tb, 3).mean(axis=(1, 3))
    shadowed = want.mean(axis=-1) < 0.5 * np.median(want.mean(axis=-1))
    assert shadowed.sum() >= 3, "the occluder casts no shadow into the view"
    err = np.abs(got - want)
    assert (err <= 0.08 * want + 0.02 * want.mean()).all(), err.max()
    persp.close()
    bake.close()


# ---- 6. NO_BACKGROUND / LIGHTING_ONLY on a perspective camera ------------------------------------------------------------
def test_no_background_and_lighting_only_on_a_perspective_camera():
    fwd = np.array([0.0, -0.35, -1.0])
    fwd /= np.linalg.norm(fwd)
    desc = plane_scene(64, 48, env=(0.3, 0.3, 0.3), back=(0.2, 0.3, 0.4), light="sphere", geo=False,
                       cam=_cam(None, origin=(0.0, 1.0, 3.0), fwd=tuple(fwd), up=(0.0, 1.0, 0.0), fov=60.0))
    pair = _pair(desc)

    def one(flags):
        pair.ctx.clear()
        pair.ctx.render(pair.ctx.make_pass(pair.cam, (0, 0, pair.w, pair.h), 1, flags))
        return pair.ctx.readback(capi.RC_BUF_RAW), pair.ctx.readback(capi.RC_BUF_BASE_COLOR)

    raw, base = one(0)
    nobg, _ = one(NOBG)
    lo, lo_base = one(LONLY)
    miss = raw[..., 3] == 0.0
    assert 100 < miss.sum() < miss.size - 100
    assert (raw[miss][:, :3] > 0).all() and (nobg[miss] == 0.0).all()
    assert nobg[~miss].tobytes() == raw[~miss].tobytes()
    assert lo_base.tobytes() == base.tobytes()
    assert lo[~miss][:, :3].mean() > 1.5 * raw[~miss][:, :3].mean()
    pair.close()


# ---- 7. SH ------------------------------------------------------------------------------------------------------------------
def _sh(pair):
    return np.stack([pair.ctx.readback(b) for b in (capi.RC_BUF_SH_R, capi.RC_BUF_SH_G, capi.RC_BUF_SH_B)], axis=2)


def test_sh_coefficient0_is_the_radiance_and_sh_leaves_raw_unchanged():
    desc = scenes.cornell_box(32, 32)
    desc.camera = _cam(0, exposure=0.5)
    pair = _pair(desc)
    with pytest.raises(cuda.CudaError):
        pair.ctx.readback(capi.RC_BUF_SH_R)
    raw_off = _bake(pair, 8, 0, (0, 0, 2))
    raw_on = _bake(pair, 8, SH, (0, 0, 2))
    assert raw_on.tobytes() == raw_off.tobytes()
    sh = _sh(pair)
    assert (raw_on[..., 3] == 1.0).all()
    np.testing.assert_allclose(sh[..., 0], Y0 * raw_on[..., :3], rtol=1e-5, atol=1e-7)
    pair.ctx.clear()
    assert (_sh(pair) == 0).all()
    pair.close()


def test_sh_furnace_and_directional_light():
    w = h = 16
    pair = _pair(plane_scene(w, h, albedo=0.5, env=(1.0, 1.0, 1.0), back=(1.0, 1.0, 1.0)))
    _bake(pair, 256, SH | LONLY)
    sh = _sh(pair)[1:-1, 1:-1].mean(axis=(0, 1))  # (3 channels, 4 coefficients), normal = +y = coefficient 1
    ratio = sh[:, 1] / sh[:, 0]
    assert np.abs(ratio - 2 * Y1 / (3 * Y0)).max() < 0.03, ratio
    assert np.abs(sh[:, [2, 3]] / sh[:, :1]).max() < 0.03
    pair.close()

    to_light = np.array([0.4, 1.0, -0.3])
    to_light /= np.linalg.norm(to_light)
    pair = _pair(plane_scene(w, h, light=tuple(-to_light)))
    _bake(pair, 64, SH | SKIP_I | LONLY)
    sh = _sh(pair)[1:-1, 1:-1].mean(axis=(0, 1, 2))
    vec = np.array([sh[3], sh[1], sh[2]])
    cosang = vec @ to_light / np.linalg.norm(vec)
    assert np.degrees(np.arccos(min(cosang, 1.0))) < 2.0
    pair.close()


def test_host_layer_bake_and_sh_data():
    w, h = 24, 24
    desc = plane_scene(w, h, light="sphere", occluder=True,
                       cam=_cam(0, output_sh=1, lighting_only=1))
    r = host.Renderer(w, h)
    assert r.sh_data() is None
    s = scenes.build(desc, r.create_scene())
    r.render(s, (0, 0, w, h), 0, 4)
    raw, sh = r.pixels(host.RAW), r.sh_data()
    lib, ctx = cuda.load_library(), r.native_context()
    rect = capi.rc_rect(0, 0, w, h)
    for ch, b in enumerate((capi.RC_BUF_SH_R, capi.RC_BUF_SH_G, capi.RC_BUF_SH_B)):
        plane = np.empty((h, w, 4), np.float32)
        assert lib.rc_readback(ctx, b, C.byref(rect), plane.ctypes.data, w) == 0
        assert plane.tobytes() == np.ascontiguousarray(sh[:, :, ch]).tobytes()
    assert (raw[..., 3] == 1.0).all() and raw[..., :3].mean() > 0
    s.close()
    r.close()


# ---- 8. two GPUs --------------------------------------------------------------------------------------------------------------
def test_two_gpu_bake_equals_one_gpu():
    if cuda.load_library().rc_device_count() < 2:
        pytest.skip("needs two GPUs")
    w, h = 32, 30
    outs = []
    for devices in (None, "0,1"):
        desc = plane_scene(w, h, light="sphere", occluder=True, cam=_cam(0, output_sh=1))
        r = host.Renderer(w, h) if devices is None else host.Renderer(w, h, devices=devices)
        s = scenes.build(desc, r.create_scene())
        r.render(s, (0, 0, w, h), 0, 6)
        outs.append((r.pixels(host.RAW), r.sh_data()))
        s.close()
        r.close()
    assert outs[0][0].tobytes() == outs[1][0].tobytes()
    assert outs[0][1].tobytes() == outs[1][1].tobytes()
    # a region inside device 0's band: the SH planes of device 1 exist (zero) and the gather succeeds
    desc = plane_scene(w, h, light="sphere", cam=_cam(0, output_sh=1))
    r = host.Renderer(w, h, devices="0,1")
    s = scenes.build(desc, r.create_scene())
    r.render(s, (0, 0, w, 4), 0, 2)
    sh = r.sh_data()
    assert sh is not None and (sh[:4] != 0).any() and (sh[h // 2:] == 0).all()
    s.close()
    r.close()


# ---- 9. reported, not faked ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["ortho", "uv_index", "removed_instance"])
def test_unsupported_bakes_are_reported(case):
    w, h = 16, 16
    cam = {"ortho": _cam(None, type=capi.CAM_ORTHO), "uv_index": _cam(0, uv_index=1),
           "removed_instance": _cam(1)}[case]
    desc = plane_scene(w, h, occluder=True, env=(1.0, 1.0, 1.0), cam=cam)
    r = host.Renderer(w, h)
    s = r.create_scene()
    if case == "removed_instance":
        scenes.build(desc, s)
        r.render(s, (0, 0, w, h), 0, 1)  # instance 1 exists: fine
        r.clear()
        s.remove_mesh_instance(1)
        s.finalize()
    else:
        with pytest.raises(host.HostError):
            scenes.build(desc, s)
    before = r.counters()["primary_rays"]
    with pytest.raises(host.HostError):
        r.render(s, (0, 0, w, h), 0, 1)
    assert r.counters()["primary_rays"] == before
    s.close()
    r.close()


def test_out_of_range_geo_targets_are_refused():
    pair = _pair(plane_scene(16, 16, env=(1.0, 1.0, 1.0)))
    _bake(pair, 1)
    before = pair.ctx.readback(capi.RC_BUF_RAW)
    n_tris = pair.view.tri_materials.count
    for geo in ((1, 0, 2), (0, n_tris - 1, 2), (0, 0xffffffff, 2)):
        with pytest.raises(cuda.CudaError):
            pair.ctx.render(pair.ctx.make_pass(pair.cam, (0, 0, 16, 16), 2, 0, geo))
    with pytest.raises(cuda.CudaError):
        pair.ctx.stage_generate_geo_rays(pair.ctx.make_pass(pair.cam, (0, 0, 16, 16), 2, 0, (0, 0, n_tris + 1)))
    assert pair.ctx.readback(capi.RC_BUF_RAW).tobytes() == before.tobytes()
    pair.close()


def test_split_passes_refused_with_a_light_that_casts_no_shadow():
    """Such a light's contribution is added at the surface it lights without a shadow ray, so the kernels cannot tell
    it from emission: SKIP_DIRECT / SKIP_INDIRECT / OUTPUT_SH are refused instead of splitting it wrongly."""
    pair = _pair(plane_scene(16, 16, light="sphere", cast_shadow=False))
    raw = _bake(pair, 2, LONLY)  # flags that do not split the light still render
    assert raw[..., :3].mean() > 0
    for f in (SKIP_D, SKIP_I, SH, SKIP_D | LONLY):
        with pytest.raises(cuda.CudaError, match="cast_shadow"):
            pair.ctx.render(pair.ctx.make_pass(pair.cam, (0, 0, 16, 16), 3, f, (0, 0, 2)))
    assert pair.ctx.readback(capi.RC_BUF_RAW).tobytes() == raw.tobytes()
    pair.close()

    w = h = 16
    desc = plane_scene(w, h, light="sphere", cast_shadow=False, cam=_cam(0, skip_direct_lighting=1))
    r = host.Renderer(w, h)
    s = scenes.build(desc, r.create_scene())
    with pytest.raises(host.HostError, match="cast_shadow"):
        r.render(s, (0, 0, w, h), 0, 1)
    assert r.counters()["primary_rays"] == 0
    s.close()
    r.close()


def test_candidate_lists_over_the_memory_cap_are_refused():
    """70 triangles whose uv covers all of [0,1]^2 at 2048^2: 70 * 2^22 > 2^28 candidate entries."""
    n = 2048
    desc = plane_scene(n, n)
    k = 70
    rng = np.random.RandomState(3)
    uv = np.array([[-0.01, -0.01], [2.1, -0.01], [-0.01, 2.1]])
    rows = [list(rng.uniform(-1, 1, 3)) + [0.0, 1.0, 0.0] + list(uv[j]) for _ in range(k) for j in range(3)]
    desc.meshes.append(scenes.MeshDesc(np.asarray(rows, np.float32), np.arange(3 * k, dtype=np.uint32),
                                       [(0, 0, 0, 3 * k)]))
    desc.instances.append((1, scenes.IDENTITY.T.reshape(16), {}))
    pair = _pair(desc)
    geo = (1, 2, k)
    with pytest.raises(cuda.CudaError, match="2\\^28"):
        pair.ctx.render(pair.ctx.make_pass(pair.cam, (0, 0, n, n), 1, 0, geo))
    with pytest.raises(cuda.CudaError, match="2\\^28"):
        pair.ctx.stage_generate_geo_rays(pair.ctx.make_pass(pair.cam, (0, 0, n, n), 1, 0, geo))
    assert not pair.ctx.readback(capi.RC_BUF_RAW).any()
    raw = _bake(pair, 1, 0, (1, 2, k - 10))  # 60 triangles fit
    assert (raw[..., 3] == 1.0).all()
    pair.close()
