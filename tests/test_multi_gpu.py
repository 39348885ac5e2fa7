"""GPU (needs >= 2 devices, skipped otherwise): the frame sharded over several GPUs of one process (rc_comm_* behind
RendererBase) is the SAME image as one GPU's, bit for bit -- full-frame regions, interleaved sub-regions with their own
iteration counters, the NLM denoise that has to see across the band borders, and the UNet denoise that runs on device 0 after a peer gather."""
import numpy as np
import pytest

from ray_b200 import capi, cuda, host, scenes

pytestmark = pytest.mark.gpu

# (input channels, output channels) of the 16 convolutions (rt_unet.cuh unet_layer; skip tensors included)
UNET_SHAPES = [(9, 32), (32, 32), (32, 48), (48, 64), (64, 80), (80, 96), (96, 96), (160, 112), (112, 112), (160, 96),
               (96, 96), (128, 64), (64, 64), (73, 64), (64, 32), (32, 3)]


def _unet_layers(seed=5):
    """A seeded weight set of the network's shapes: both sides run the same filter, whatever its weights."""
    rng = np.random.default_rng(seed)
    return [((rng.standard_normal((co, ci, 3, 3)) * np.sqrt(2.0 / (9 * ci))).astype(np.float16),
             (rng.standard_normal(co) * 0.01).astype(np.float16)) for ci, co in UNET_SHAPES]


def _n_devices():
    try:
        return cuda.load_library().rc_device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_n_devices() < 2, reason="needs at least 2 CUDA devices")
@pytest.mark.parametrize("make", [lambda: scenes.cornell_box(96, 70),
                                  lambda: scenes.hall("principled", 160, 90, floor_res=32, n_columns=6, col_seg=10,
                                                      col_rings=6, extra_lights=6)])
def test_multi_device_frame_equals_single_device_frame(make):
    desc = make()
    w, h, spp = desc.width, desc.height, 5
    n = min(_n_devices(), 8)
    one = host.Renderer(w, h, device=0)
    s1 = scenes.build(desc, one.create_scene())
    one.render(s1, (0, 0, w, h), 0, spp)
    ref_raw, ref_final, ref_base = one.pixels(host.RAW), one.pixels(host.FINAL), one.pixels(host.BASE_COLOR)

    many = host.Renderer(w, h, devices=",".join(str(i) for i in range(n)))
    assert many.lib.rh_device_count(many.h) == n
    sn = scenes.build(desc, many.create_scene())
    many.render(sn, (0, 0, w, h), 0, spp)
    assert many.pixels(host.RAW).tobytes() == ref_raw.tobytes()
    assert many.pixels(host.FINAL).tobytes() == ref_final.tobytes()
    assert many.pixels(host.BASE_COLOR).tobytes() == ref_base.tobytes()
    c1, cn = one.counters(), many.counters()
    assert c1["primary_rays"] == cn["primary_rays"] and c1["secondary_rays"] == cn["secondary_rays"]

    # sub-regions that straddle the band borders, each with its own iteration counter
    many.clear((0, 0, 0, 0))
    one.clear((0, 0, 0, 0))
    rects = [(0, 0, w // 2, h), (w // 2, 0, w - w // 2, h // 3), (w // 2, h // 3, w - w // 2, h - h // 3)]
    its1, itsn = [0] * 3, [0] * 3
    for _ in range(3):
        for i, r in enumerate(rects):
            its1[i] = one.render(s1, r, its1[i], 1)
            itsn[i] = many.render(sn, r, itsn[i], 1)
    assert many.pixels(host.RAW).tobytes() == one.pixels(host.RAW).tobytes()

    # NLM denoise reads across band borders
    one.denoise((0, 0, w, h), its1[0])
    many.denoise((0, 0, w, h), itsn[0])
    assert many.pixels(host.RAW).tobytes() == one.pixels(host.RAW).tobytes()
    # UNet denoise: the whole network runs on device 0 after its input planes were gathered there
    layers = _unet_layers()
    for r_, it_ in ((one, its1[0]), (many, itsn[0])):
        r_.set_unet_weights(layers, capi.RC_UNET_FP32)
        r_.denoise_unet((0, 0, w, h), it_)
    assert many.pixels(host.RAW).tobytes() == one.pixels(host.RAW).tobytes()
    assert many.pixels(host.FINAL).tobytes() == one.pixels(host.FINAL).tobytes()
    for x in (s1, sn):
        x.close()
    one.close()
    many.close()
