"""CPU: the product's host layer (own SAH BVH8 builder, triangle blocks, instances, light tree, tables) validated
WITHOUT a GPU by running the reference's own Ref:: traversal / shading code (oracle/_ref) over the arrays it builds,
next to the reference's own Cpu::Scene built from the same description."""
import ctypes as C
import os

import numpy as np
import pytest

from ray_b200 import capi, host, scenes
from ray_b200.cuda import HIT_DTYPE


def _arr(a, dtype):
    n = a.count * a.stride // np.dtype(dtype).itemsize
    if n == 0:
        return np.zeros(0, dtype)
    return np.ctypeslib.as_array(C.cast(a.ptr, C.POINTER(C.c_uint8)), shape=(a.count * a.stride,)).view(dtype).copy()


SCENES = {
    "cornell": lambda: scenes.cornell_box(64, 64),
    "zoo": lambda: scenes.material_zoo(96, 72),
    "instanced": lambda: scenes.instanced(16, 400, 64, 64),
    "hall_small": lambda: scenes.hall("principled", 96, 54, floor_res=24, n_columns=4, col_seg=8, col_rings=6,
                                      extra_lights=10),
}


@pytest.fixture(scope="module", params=list(SCENES))
def host_built(request):
    desc = SCENES[request.param]()
    hs = scenes.build(desc, host.Scene(None))
    assert host.load_library().rh_error_count(None) == 0, host.load_library().rh_last_error(None)
    yield request.param, desc, hs
    hs.close()


@pytest.fixture(scope="module")
def built(host_built, oracle_mod):
    name, desc, hs = host_built
    osc = scenes.build(desc, oracle_mod.Scene(wide=True))
    yield name, desc, hs, osc
    osc.close()


def test_bvh8_structure(host_built):
    name, desc, hs = host_built
    v = hs.view()
    nodes = _arr(v.wnodes, np.uint8).reshape(-1, 224)
    bmin = nodes[:, :96].copy().view(np.float32).reshape(-1, 3, 8)
    bmax = nodes[:, 96:192].copy().view(np.float32).reshape(-1, 3, 8)
    child = nodes[:, 192:].copy().view(np.uint32).reshape(-1, 8)
    tri_idx = _arr(v.tri_indices, np.uint32)
    assert len(tri_idx) % 8 == 0 and len(tri_idx) == v.mtris.count * 8
    is_leaf = (child[:, 0] & 0x80000000) != 0
    # every non-degenerate triangle sits in exactly one BLAS leaf block
    seen = np.zeros(v.tri_materials.count, np.int32)
    inst = _arr(v.mesh_instances, np.uint8).reshape(-1, 144)
    blas_roots = set(int(x) for x in inst[:, 4:8].copy().view(np.uint32).ravel())
    visited = set()
    for root in blas_roots:
        stack = [root]
        while stack:
            n = stack.pop()
            if n in visited:
                continue
            visited.add(n)
            if is_leaf[n]:
                first, cnt = int(child[n, 0] & 0x7fffffff), int(child[n, 1])
                assert first % 8 == 0 and 1 <= cnt <= 8
                ids = tri_idx[first:first + 8]
                assert (ids[cnt:] == ids[cnt - 1]).all(), "padding must repeat the last triangle"
                np.add.at(seen, ids[:cnt], 1)
            else:
                for k in range(8):
                    c = int(child[n, k])
                    if c == 0x7fffffff:
                        assert (bmin[n, :, k] == 0).all() and (bmax[n, :, k] == 0).all()
                        continue
                    # child box inside... the child's own children boxes
                    if not is_leaf[c]:
                        valid = child[c] != 0x7fffffff
                        assert (bmin[c][:, valid].min(axis=1) >= bmin[n, :, k] - 1e-6).all()
                        assert (bmax[c][:, valid].max(axis=1) <= bmax[n, :, k] + 1e-6).all()
                    stack.append(c)
    assert seen.max() == 1
    assert int((seen == 1).sum()) >= desc.triangle_count() - 2  # at most a couple of degenerate triangles
    # the TLAS root exists and its leaves reference every instance once
    assert v.tlas_root != 0xffffffff
    leaves, stack = [], [int(v.tlas_root)]
    while stack:
        n = stack.pop()
        if is_leaf[n]:
            leaves.append(int(child[n, 0] & 0x7fffffff))
        else:
            stack += [int(c) for c in child[n] if c != 0x7fffffff]
    assert sorted(leaves) == list(range(v.mesh_instances.count))


def _planes(mtris, tri_indices):
    """triangle id -> its plane-form data, from the 8-wide triangle blocks and their triangle ids"""
    m = mtris.reshape(-1, 3, 4, 8)  # block, {n,u,v}, comp, lane
    ti = tri_indices.reshape(-1, 8)
    out = {}
    for b in range(len(ti)):
        for lane in range(8):
            out[int(ti[b, lane])] = m[b, :, :, lane].tobytes()
    return out


def test_triangle_planes_equal_the_references(built):
    """Same triangle => bit-identical plane-form data as Ray::PreprocessTri produced for the reference's own scene."""
    name, desc, hs, osc = built
    hv, ov = hs.view(), osc.view()
    hp, op = _planes(_arr(hv.mtris, np.float32), _arr(hv.tri_indices, np.uint32)), \
        _planes(_arr(ov.mtris, np.float32), _arr(ov.tri_indices, np.uint32))
    # global triangle ids are assigned identically (append order of meshes / index triples)
    common = set(hp) & set(op)
    assert len(common) >= desc.triangle_count() - 2
    bad = [t for t in common if hp[t] != op[t]]
    assert not bad, f"{len(bad)} triangles have different plane data"
    assert np.array_equal(_arr(hv.tri_materials, np.uint16), _arr(ov.tri_materials, np.uint16))
    assert _arr(hv.materials, np.uint8).tobytes() == _arr(ov.materials, np.uint8).tobytes()


def test_primary_hits_match_reference_scene(built, oracle_mod):
    """Ref::TraceRays over the host layer's arrays vs over the reference's own scene: same nearest hit for every
    primary ray (triangle id, instance, t/u/v) except where two candidates tie exactly."""
    name, desc, hs, osc = built
    w, h = desc.width, desc.height
    rays, hits = osc.generate_primary_rays(w, h, (0, 0, w, h), 1)
    _, o_hits = osc.trace_rays(1, rays, hits, False)
    vs = oracle_mod.ViewScene(hs.view(), hs.camera())
    _, h_hits = vs.trace_rays(1, rays, hits, False)
    hit = o_hits["v"] >= 0
    assert np.array_equal(hit, h_hits["v"] >= 0)
    same = (o_hits["prim_index"] == h_hits["prim_index"]) & (o_hits["obj_index"] == h_hits["obj_index"])
    frac = float((same | ~hit).mean())
    assert frac > 0.995, f"{name}: only {frac:.4f} of primary rays agree on the triangle hit"
    m = hit & same
    if name == "instanced":
        # non-trivial instance transforms: the host layer inverts them in double precision (Gauss-Jordan), the reference
        # with a float cofactor expansion (Core.cpp:1390-1431), so object-space rays differ in the last bits
        assert np.allclose(o_hits["t"][m], h_hits["t"][m], rtol=3e-5, atol=1e-6)
        assert np.allclose(o_hits["u"][m], h_hits["u"][m], rtol=0, atol=2e-4)
    else:
        assert np.array_equal(o_hits["t"][m], h_hits["t"][m]) and np.array_equal(o_hits["u"][m], h_hits["u"][m])


def test_camera_matches_reference(built):
    name, desc, hs, osc = built
    a, b = hs.camera(), osc.camera()
    for f, _ in capi.rc_camera._fields_:
        x, y = getattr(a, f), getattr(b, f)
        if hasattr(x, "__len__"):
            assert np.allclose(list(x), list(y), rtol=0, atol=1e-7), f
        else:
            assert x == pytest.approx(y, rel=1e-6, abs=1e-7), f


def test_lights_and_light_tree(built, oracle_mod):
    """Same analytic/triangle lights as the reference registers; the host layer's own light tree is a different tree, so
    check it through the integrator: radiance of the same samples rendered by Ref:: code over either scene converges to
    the same image."""
    name, desc, hs, osc = built
    hv, ov = hs.view(), osc.view()
    hl = _arr(hv.lights, np.uint8).reshape(-1, 64)
    ol = _arr(ov.lights, np.uint8).reshape(-1, 64)
    assert hv.lights.count == ov.lights.count and hv.li_indices.count == ov.li_indices.count
    assert hv.visible_lights_count == ov.visible_lights_count and hv.blocker_lights_count == ov.blocker_lights_count
    # type / flags word and colour of every light (payload floats may differ in the last bit for transformed vectors)
    order_h = np.lexsort(hl[:, :16].T[::-1])
    order_o = np.lexsort(ol[:, :16].T[::-1])
    assert np.array_equal(hl[order_h][:, :16], ol[order_o][:, :16])
    assert hv.light_cwnodes.count >= 1
    w, h = desc.width, desc.height
    spp = 6
    vs = oracle_mod.ViewScene(hv, hs.camera())
    img_h, n_h = oracle_mod.render_with_stages(vs, osc, w, h, spp)
    img_o, n_o = oracle_mod.render_with_stages(osc, osc, w, h, spp)
    assert np.isfinite(img_h).all()
    assert abs(n_h - n_o) / n_o < 0.02
    mh, mo = float(img_h[..., :3].mean()), float(img_o[..., :3].mean())
    assert abs(mh - mo) / max(mo, 1e-6) < 0.06, (mh, mo)


def _expanded_rgba(t):
    """Level-0 texels of an rc_texture as (h, w, 4) with the channel expansion of TexStorage*::Fetch applied."""
    w, h, n = int(t.res[0][0]), int(t.res[0][1]), int(t.channels)
    a = np.ctypeslib.as_array(C.cast(t.pixels[0], C.POINTER(C.c_uint8)), shape=(h, w, n))
    return np.concatenate([a] + [a[..., n - 1:n]] * (4 - n), axis=-1)


def test_textures_and_textured_materials_match_reference(oracle_mod):
    """SURVEY 8(f)-1 on the host side: AddTexture's storage choice / handle bits / normal-map repacking and the
    material lowering with textures (alpha -> Mix with Transparent, emission -> additive Mix, triangle-light tex_index)
    give the reference's material_t / light_t bytes and the reference's texels."""
    desc = scenes.textured(32, 24)
    hs = scenes.build(desc, host.Scene(None))
    osc = scenes.build(desc, oracle_mod.Scene(wide=True))
    assert host.load_library().rh_error_count(None) == 0, host.load_library().rh_last_error(None)
    hv, ov = hs.view(), osc.view()
    assert _arr(hv.materials, np.uint8).tobytes() == _arr(ov.materials, np.uint8).tobytes()
    assert hv.texture_count == ov.texture_count == len(desc.textures)
    href = {hv.textures[i].handle: hv.textures[i] for i in range(hv.texture_count)}
    for i in range(ov.texture_count):
        to = ov.textures[i]
        th = href[to.handle]
        assert [tuple(th.res[k]) for k in range(12)] == [tuple(to.res[k]) for k in range(12)]
        assert np.array_equal(_expanded_rgba(th), _expanded_rgba(to)), hex(to.handle)
    hl = _arr(hv.lights, np.uint32).reshape(-1, 16)
    ol = _arr(ov.lights, np.uint32).reshape(-1, 16)
    tri_h = sorted(int(x[6]) for x in hl if (x[0] & 7) == 5)  # light_t::tri.tex_index of LIGHT_TYPE_TRI lights
    tri_o = sorted(int(x[6]) for x in ol if (x[0] & 7) == 5)
    assert tri_h == tri_o and any(t != 0xffffffff for t in tri_h)
    hs.close()
    osc.close()


def test_environment_quadtree_matches_reference(oracle_mod):
    """SURVEY 8(f)-2 on the host side: the stand-alone scene's restatement of PrepareEnvMapQTree gives the reference's
    quad-tree bit for bit (same libm, same summation order), and the same environment fields."""
    desc = scenes.envmap_zoo(32, 24)
    hs = scenes.build(desc, host.Scene(None))
    osc = scenes.build(desc, oracle_mod.Scene(wide=True))
    assert host.load_library().rh_error_count(None) == 0, host.load_library().rh_last_error(None)
    hv, ov = hs.view(), osc.view()
    assert hv.qtree_levels == ov.qtree_levels >= 3
    assert (hv.env_map, hv.back_map, hv.env_light_index) == (ov.env_map, ov.back_map, ov.env_light_index)
    assert (hv.env_map_rotation, hv.back_map_rotation) == (ov.env_map_rotation, ov.back_map_rotation)
    for i in range(ov.qtree_levels):
        n = 4 ** (ov.qtree_levels - 1 - i) * 4
        a = np.ctypeslib.as_array(C.cast(ov.qtree_mips[i], C.POINTER(C.c_uint32)), shape=(n,))
        b = np.ctypeslib.as_array(C.cast(hv.qtree_mips[i], C.POINTER(C.c_uint32)), shape=(n,))
        assert np.array_equal(a, b), f"quad-tree level {i}"
    hs.close()
    osc.close()


def test_filter_tables_match_reference(oracle_mod):
    for filt, width in ((capi.FILTER_GAUSSIAN, 1.5), (capi.FILTER_BLACKMAN_HARRIS, 1.5), (capi.FILTER_BLACKMAN_HARRIS, 2.0)):
        desc = scenes.cornell_box(16, 16)
        desc.camera.filter = filt
        desc.camera.filter_width = width
        osc = scenes.build(desc, oracle_mod.Scene(wide=True))
        ref = osc.filter_table()
        mine = host.builtin_filter_table(filt, width)
        assert np.abs(ref - mine).max() <= 2e-6
        osc.close()


def test_builtin_sampler_table_is_a_02_sequence_per_dimension():
    t = host.builtin_sampler_table().reshape(32, 4096, 2)
    for d in (0, 1, 7, 31):
        pts = t[d].astype(np.float64) / 2.0 ** 32
        for m in (4, 6, 8, 12):  # first 2^m points: one point in every elementary interval of area 2^-m
            n = 1 << m
            p = pts[:n]
            for a in range(m + 1):
                ix = np.floor(p[:, 0] * (1 << a)).astype(np.int64)
                iy = np.floor(p[:, 1] * (1 << (m - a))).astype(np.int64)
                cells = ix * (1 << (m - a)) + iy
                assert len(np.unique(cells)) == n, (d, m, a)
    assert len({t[d].tobytes() for d in range(32)}) == 32


def test_view_render_reproduces_renderer_ref(oracle_mod):
    """oracle.view_render (the multi-threaded Ref:: stage sequence the at-size GPU parity tests compare against) over the
    reference's OWN arrays is RendererRef, bit for bit."""
    desc = scenes.cornell_box(48, 40)
    osc = scenes.build(desc, oracle_mod.Scene(wide=True))
    ref = oracle_mod.Renderer(capi.RT_REFERENCE, 48, 40)
    it = 0
    for _ in range(3):
        it = ref.render(osc, (0, 0, 48, 40), it)
    raw = ref.pixels(1)
    full, n_rays, n_shadow = oracle_mod.view_render(osc.view(), osc.camera(), osc, 48, 40, 3, threads=3)
    assert np.array_equal(full, raw)
    assert n_rays > 3 * 48 * 40 and n_shadow > 0
    ref.close()
    osc.close()


GOLDEN = {"cornell_48": lambda: scenes.cornell_box(48, 48), "zoo_64x48": lambda: scenes.material_zoo(64, 48)}


@pytest.mark.parametrize("name", list(GOLDEN))
def test_host_layer_matches_the_references_stored_scene(name):
    """The arrays the reference's own Cpu::Scene built for a small scene, stored in tests/golden/<name>.npz: the host
    layer, fed the same description, gives the same triangle plane data, per-triangle materials, material records,
    lights (type / flags word and colour), camera and pixel-filter table."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))
    desc = GOLDEN[name]()
    hs = scenes.build(desc, host.Scene(None))
    assert host.load_library().rh_error_count(None) == 0, host.load_library().rh_last_error(None)
    hv = hs.view()
    hp = _planes(_arr(hv.mtris, np.float32), _arr(hv.tri_indices, np.uint32))
    op = _planes(g["arr_mtris"].view(np.float32), g["arr_tri_indices"].view(np.uint32))
    common = set(hp) & set(op)
    assert len(common) >= desc.triangle_count() - 2
    bad = [t for t in common if hp[t] != op[t]]
    assert not bad, f"{len(bad)} triangles have different plane data"
    assert _arr(hv.tri_materials, np.uint8).tobytes() == g["arr_tri_materials"].tobytes()
    assert _arr(hv.materials, np.uint8).tobytes() == g["arr_materials"].tobytes()

    hl = _arr(hv.lights, np.uint8).reshape(-1, 64)
    ol = g["arr_lights"].reshape(-1, 64)
    assert len(hl) == len(ol) and hv.li_indices.count * 4 == len(g["arr_li_indices"])
    assert (hv.visible_lights_count, hv.blocker_lights_count) == \
        (int(g["s_visible_lights_count"]), int(g["s_blocker_lights_count"]))
    order_h, order_o = np.lexsort(hl[:, :16].T[::-1]), np.lexsort(ol[:, :16].T[::-1])
    assert np.array_equal(hl[order_h][:, :16], ol[order_o][:, :16])

    a, b = hs.camera(), capi.rc_camera.from_buffer_copy(g["cam"].tobytes())
    for f, _ in capi.rc_camera._fields_:
        x, y = getattr(a, f), getattr(b, f)
        if hasattr(x, "__len__"):
            assert np.allclose(list(x), list(y), rtol=0, atol=1e-7), f
        else:
            assert x == pytest.approx(y, rel=1e-6, abs=1e-7), f
    if b.filter != capi.FILTER_BOX:
        assert np.abs(host.builtin_filter_table(b.filter, desc.camera.filter_width) - g["filter_table"]).max() <= 2e-6
    hs.close()
