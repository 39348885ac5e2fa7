"""GPU: what a context allocates on the device goes away with it, and what it configures on its device holds for that
device -- a second context on another GPU runs the same kernels as the first."""
import ctypes as C

import numpy as np
import pytest
import torch

from ray_b200 import capi, cuda, host, scenes
from test_multi_gpu import _n_devices, _unet_layers

pytestmark = pytest.mark.gpu

W = H = 1024  # one leaked frame plane (float4 per pixel) is 16 MiB


def _first_tlas_node(view):
    """Lowest node index of the top level: the host layer stores the TLAS after every BLAS."""
    words = np.ctypeslib.as_array((C.c_uint32 * (view.wnodes.count * 56)).from_address(view.wnodes.ptr))
    child = words.reshape(view.wnodes.count, 56)[:, 48:]
    seen, stack = set(), [view.tlas_root]
    while stack:
        n = stack.pop()
        seen.add(n)
        if not child[n, 0] & 0x80000000:
            stack += [int(c) for c in child[n] if c != 0x7fffffff]
    return min(seen)


def _view_lut():
    g = np.linspace(0.0, 1.0, 48) ** 1.2
    r, gg, b = np.meshgrid(g, g, g, indexing="ij")
    q = lambda x: np.round(np.clip(x, 0, 1) * 1023).astype(np.uint32)
    return (q(r) | (q(gg) << 10) | (q(b * b) << 20)).ravel(order="F")


def _cycle(desc, hs, layers):
    """Every entry point that allocates on the device, on one context, then its destruction."""
    ctx = cuda.Context(0)
    ctx.resize(W, H)
    ctx.upload_tables(host.builtin_sampler_table(), host.builtin_filter_table(capi.FILTER_GAUSSIAN, 1.5))
    view = hs.view()
    ctx.upload_scene(view)
    ctx.set_view_lut(1, _view_lut())
    cam = hs.camera()
    cam.view_transform = 1
    full = (0, 0, W, H)
    ctx.render(ctx.make_pass(cam, full, 1))  # sorted (the default)

    geo_cam = hs.camera()
    geo_cam.type = capi.CAM_GEO
    tris = len(desc.meshes[desc.instances[0][0]].indices) // 3  # instance 0 is mesh 0: triangles [0, tris)
    bake = ctx.make_pass(geo_cam, full, 1, capi.RC_RENDER_OUTPUT_SH, (0, 0, tris))
    ctx.render(bake)
    assert np.isfinite(ctx.readback(capi.RC_BUF_SH_R, (0, 0, 8, 8))).all()

    ctx.denoise_nlm(full, 1)
    ctx.unet_set_weights(layers)
    ctx.denoise_unet(full, capi.RC_UNET_TENSOR_CORES)
    ctx.denoise_unet(full, capi.RC_UNET_FP32)
    boxes = np.random.default_rng(3).random((50000, 6), dtype=np.float32)
    boxes[:, 3:] += boxes[:, :3]
    ctx.build_lbvh(boxes)
    ctx.update_instances(view, _first_tlas_node(view))

    p = ctx.make_pass(cam, full, 2)
    rays, hits = ctx.stage_generate_primary_rays(p)
    rays, hits = ctx.stage_trace_rays(p, rays, hits, True)
    secondary, shadow = ctx.stage_shade(p, True, 0, rays, hits)
    ctx.stage_trace_shadow_rays(p, shadow, 0.0)
    ctx.stage_sort_rays(secondary)
    assert len(ctx.stage_generate_geo_rays(bake)[0]) > 0

    ctx.resize(W // 2, H // 3)
    ctx.resize(W, H)
    ctx.render(bake)  # the SH planes came back with the resize
    ctx.close()


def test_destroy_releases_every_device_allocation():
    desc = scenes.envmap_zoo(W, H)  # textured (the RGBE environment map) with an importance-sampling quad-tree
    hs = scenes.build(desc, host.Scene(None))
    layers = _unet_layers()
    torch.cuda.mem_get_info(0)
    _cycle(desc, hs, layers)  # loads the modules; cub and the driver set up what they keep
    before, _ = torch.cuda.mem_get_info(0)
    _cycle(desc, hs, layers)
    after, _ = torch.cuda.mem_get_info(0)
    hs.close()
    assert before - after <= 2 << 20, f"{(before - after) / 2**20:.1f} MiB of device memory not returned"


@pytest.mark.skipif(_n_devices() < 2, reason="needs at least 2 CUDA devices")
def test_tensor_core_unet_runs_the_same_on_a_second_device():
    """k_unet_conv_tc needs more dynamic shared memory than the default; the attribute that allows it is set per
    device, so the context on device 1 must set it for itself."""
    desc = scenes.cornell_box(96, 64)
    w, h = desc.width, desc.height
    layers = _unet_layers(seed=9)
    out = []
    for device in (0, 1):
        hs = scenes.build(desc, host.Scene(None))
        ctx = cuda.Context(device)
        cam = hs.camera()
        ctx.resize(w, h)
        ctx.upload_tables(host.builtin_sampler_table(), None if cam.filter == capi.FILTER_BOX else
                          host.builtin_filter_table(cam.filter, desc.camera.filter_width))
        ctx.upload_scene(hs.view())
        for it in range(1, 5):
            ctx.render(ctx.make_pass(cam, (0, 0, w, h), it))
        ctx.unet_set_weights(layers)
        ctx.denoise_unet((0, 0, w, h), capi.RC_UNET_TENSOR_CORES)
        out.append((ctx.readback(capi.RC_BUF_RAW), ctx.readback(capi.RC_BUF_FINAL)))
        ctx.close()
        hs.close()
    assert out[0][0].tobytes() == out[1][0].tobytes()
    assert out[0][1].tobytes() == out[1][1].tobytes()
