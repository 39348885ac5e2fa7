"""GPU parity AT SIZE: the configurations BASELINE.json is quoted on, not the toy frames of test_parity_gpu.py.

  * hall-250k (253,964 triangles, ~50 k BVH8 nodes) diffuse and principled at 1920x1080 (configs #2 / #3: 16-bit pixel
    coordinates at 1920, deep stacks, the 18-bit sort key at work), oracle-built BVH8, raw image bitwise
  * Cornell box 256x256 x 64 spp (config #1) against RendererRef, raw image bitwise
  * a TLAS over 1024 instances of one BLAS with rotations + non-uniform scales (config #5 in miniature), bitwise
  * the PRODUCT path (host layer: own SAH BVH8 / light tree / camera -> C-ABI -> kernels) at 1080p on hall-250k against the
    reference's Ref:: stage functions run over the host layer's own arrays (oracle.view_render), bitwise.

The reference side is the unmodified reference code on all host threads (oracle.view_render == RendererRef bit for bit,
tests/test_host_cpu.py::test_view_render_reproduces_renderer_ref).  Without the oracle library the CUDA side runs on the
host layer's arrays with the built-in tables and is checked against the digests stored in tests/golden/cuda_digests.json.
"""
import copy

import numpy as np
import pytest

from ray_b200 import capi, host, scenes
from common import STORED, make_pair, maybe_oracle

pytestmark = [pytest.mark.gpu, pytest.mark.slow]


def _same(a, b):
    """bitwise equality up to the sign of zero (x + (-0) accumulations), NaNs equal"""
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def _report(a, b):
    d = np.abs(a - b)
    return f"L-inf {d.max():g}, {int((d > 0).any(-1).sum())} of {a.shape[0] * a.shape[1]} pixels differ"


def _counts(c):
    return np.asarray([c["primary_rays"], c["secondary_rays"], c["shadow_rays"]], np.uint64)


def _cuda_render(pair, spp):
    pair.ctx.clear((0, 0, 0, 0))
    for i in range(1, spp + 1):
        pair.ctx.render(pair.make_pass(i, flags=capi.RC_RENDER_ASYNC))
    pair.ctx.sync()
    return pair.ctx.readback(capi.RC_BUF_RAW)


@pytest.mark.parametrize("variant", ["diffuse", "principled"])
def test_hall_250k_1080p_is_bit_identical_to_the_reference(variant):
    o = maybe_oracle()
    spp = 2
    pair = make_pair(scenes.hall(variant, 1920, 1080))
    assert pair.view.wnodes.count > 40000 and pair.desc.triangle_count() > 250000
    raw = _cuda_render(pair, spp)
    c = pair.ctx.counters()
    assert c["primary_rays"] == spp * 1920 * 1080
    if o is None:
        STORED.check(f"size/hall_{variant}", raw, _counts(c))
        pair.close()
        return
    ref, n_rays, n_shadow = o.view_render(pair.view, pair.cam, pair.osc, pair.w, pair.h, spp)
    assert c["primary_rays"] + c["secondary_rays"] == n_rays and c["shadow_rays"] == n_shadow
    assert _same(raw, ref), _report(raw, ref)
    pair.close()


def test_cornell_256_64spp_is_bit_identical_to_renderer_ref():
    """config #1: samples/00_basic at its own size and sample count, against the reference's RendererRef"""
    o = maybe_oracle()
    w = h = 256
    spp = 64
    pair = make_pair(scenes.cornell_box(w, h))
    if o is None:
        STORED.check("size/cornell_256_64spp", _cuda_render(pair, spp))
        pair.close()
        return
    ref = o.Renderer(capi.RT_REFERENCE, w, h)
    ref.render_mt(pair.osc, spp, o.host_threads(), 32)
    ref_raw = ref.pixels(1)
    ref.close()
    raw = _cuda_render(pair, spp)
    assert _same(raw, ref_raw), _report(raw, ref_raw)
    pair.close()


def test_tlas_1024_instances_is_bit_identical_to_the_reference():
    o = maybe_oracle()
    spp = 2
    pair = make_pair(scenes.instanced(1024, 4000, 768, 512))
    assert pair.view.mesh_instances.count >= 1024
    raw = _cuda_render(pair, spp)
    c = pair.ctx.counters()
    if o is None:
        STORED.check("size/tlas_1024", raw, _counts(c))
        pair.close()
        return
    ref, n_rays, n_shadow = o.view_render(pair.view, pair.cam, pair.osc, pair.w, pair.h, spp)
    assert c["primary_rays"] + c["secondary_rays"] == n_rays and c["shadow_rays"] == n_shadow
    assert _same(raw, ref), _report(raw, ref)
    pair.close()


def _camera_only(desc):
    d = copy.copy(desc)
    d.meshes, d.instances, d.lights, d.textures = [], [], [], []
    d.materials = []
    d.env_map = d.back_map = capi.RS_INVALID
    return d


@pytest.mark.parametrize("variant", ["diffuse", "principled"])
def test_product_path_on_its_own_arrays_is_bit_identical_hall_250k_1080p(variant):
    """Public path (RendererBase::RenderScene on the stand-alone host layer) vs the reference's stage functions over the
    host layer's arrays: same image, bit for bit, at the bench workload."""
    o = maybe_oracle()
    w, h, spp = 1920, 1080, 2
    desc = scenes.hall(variant, w, h)
    r = host.Renderer(w, h)
    if o is not None:
        r.set_sampler_table(o.pmj_table())
    s = scenes.build(desc, r.create_scene())
    it = r.render(s, (0, 0, w, h), 0, spp)
    assert it == spp
    raw = r.pixels(host.RAW)
    c = r.counters()
    if o is None:
        STORED.check(f"size/product_hall_{variant}", raw, _counts(c))
        s.close()
        r.close()
        return
    cam_scene = scenes.build(_camera_only(desc), o.Scene(wide=True))
    ref, n_rays, n_shadow = o.view_render(s.view(), s.camera(), cam_scene, w, h, spp)
    assert c["primary_rays"] + c["secondary_rays"] == n_rays and c["shadow_rays"] == n_shadow
    assert _same(raw, ref), _report(raw, ref)
    cam_scene.close()
    s.close()
    r.close()
