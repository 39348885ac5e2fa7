"""CPU: the float64 UNet reference (tests/unet_ref.py) that the GPU tests of both device paths rely on -- its
convolution convention, its transfer functions and its layer table."""
import os
import re

import numpy as np

import unet_ref as U
from test_parity_gpu import UNET_SHAPES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_conv_matches_a_naive_loop():
    """3 x 3 cross-correlation, OIHW weights, zero padding: pins the tap order and the weight layout."""
    rng = np.random.default_rng(1)
    h, w, cin, cout = 5, 7, 3, 2
    x = rng.standard_normal((h, w, cin))
    k = rng.standard_normal((cout, cin, 3, 3))
    b = rng.standard_normal(cout)
    want = np.zeros((h, w, cout))
    for y in range(h):
        for xx in range(w):
            for o in range(cout):
                s = b[o]
                for c in range(cin):
                    for ky in range(3):
                        for kx in range(3):
                            yy, xs = y + ky - 1, xx + kx - 1
                            if 0 <= yy < h and 0 <= xs < w:
                                s += k[o, c, ky, kx] * x[yy, xs, c]
                want[y, xx, o] = s
    np.testing.assert_allclose(U.conv3x3(x, k, b), want, rtol=1e-12, atol=1e-12)
    # without row padding the first and last rows are the halo
    np.testing.assert_allclose(U.conv3x3(x, k, b, pad_rows=False), U.conv3x3(x, k, b)[1:-1], rtol=1e-12, atol=1e-12)


def test_transfer_functions_round_trip():
    v = np.logspace(-9, 4, 20001)
    back = U.output_hdr(U.input_hdr(v))
    rel = np.abs(back - v) / v
    assert rel.max() <= 1e-6, f"output_hdr(input_hdr(v)) off by {rel.max():.3g} relative at v = {v[rel.argmax()]:.6g}"


def _gap(f0, f1, x):
    a, b = float(f0(x)), float(f1(x))
    return abs(a - b) / max(abs(a), abs(b))


def test_transfer_functions_are_continuous_at_their_knots():
    """Both pieces of each transfer function meet at the knots to 1e-6 relative: checks the transcribed constants."""
    lin_in = lambda v: U.A * v * U.IN_NORM
    pow_in = lambda v: (U.B * v ** U.C + U.D) * U.IN_NORM
    log_in = lambda v: (U.E * np.log(v + U.F) + U.G) * U.IN_NORM
    lin_out = lambda x: x / U.A
    pow_out = lambda x: ((x - U.D) / U.B) ** U.INV_C
    exp_out = lambda x: np.exp((x - U.G) / U.E) - U.F
    gaps = {"input_hdr at y0": _gap(lin_in, pow_in, U.Y0), "input_hdr at y1": _gap(pow_in, log_in, U.Y1),
            "output_hdr at x0": _gap(lin_out, pow_out, U.X0), "output_hdr at x1": _gap(pow_out, exp_out, U.X1)}
    assert max(gaps.values()) <= 1e-6, gaps
    # and the functions themselves take the intended branch on each side of a knot
    assert float(U.input_hdr(U.Y0)) == lin_in(U.Y0) and float(U.output_hdr(U.X1 / U.OUT_NORM * 1.001)) > 0


def test_layer_table_matches_the_network_shape_and_skip_wiring():
    assert [(c1 + c2, co) for c1, c2, co, *_ in U.LAYERS] == UNET_SHAPES
    assert U.SKIP == {7: 3, 9: 2, 11: 1, 13: "input"}
    # the skip tensor of each decoder layer has the channels and the grid that layer expects
    for i, src in U.SKIP.items():
        cin1, cin2, _, level, up, _ = U.LAYERS[i]
        assert up
        if src == "input":
            assert cin2 == 9 and level == 0
        else:
            s = U.LAYERS[src]
            assert cin2 == s[2] and level == s[3] + (1 if s[5] else 0)
        prev = U.LAYERS[i - 1]
        assert cin1 == prev[2] and level + 1 == prev[3] + (1 if prev[5] else 0)


def test_layer_table_matches_the_kernels_table():
    """The table the kernels use (rt_unet.cuh unet_layer) states the same network."""
    src = open(os.path.join(ROOT, "ray_b200", "csrc", "rt_unet.cuh")).read()
    body = src[src.index("unet_layer(int i)"):]
    body = body[:body.index("};")]
    rows = re.findall(r"\{(\d+),\s*(\d+),\s*(\d+),\s*(\d+),\s*(true|false),\s*(true|false)\}", body)
    got = [(int(a), int(b), int(c), int(d), e == "true", f == "true") for a, b, c, d, e, f in rows]
    assert got == U.LAYERS


def test_forward_is_shape_consistent_and_pools():
    rng = np.random.default_rng(3)
    layers = [((rng.standard_normal((co, ci, 3, 3)) * np.sqrt(2.0 / (9 * ci))).astype(np.float16),
               (rng.standard_normal(co) * 0.1).astype(np.float16)) for ci, co in UNET_SHAPES]
    net = U.UNet(layers)
    h, w = 20, 35
    full = rng.uniform(0, 2, (h, w, 4)).astype(np.float32)
    alb = rng.uniform(0, 1, (h, w, 4)).astype(np.float32)
    dn = rng.uniform(-1, 1, (h, w, 4)).astype(np.float32)
    f = U.features(full, alb, dn)
    assert f.shape == (32, 48, 9) and not f[h:].any() and not f[:, w:].any()
    t, last = net.forward(f)
    for i, (_, _, cout, level, _, pool) in enumerate(U.LAYERS[:15]):
        sh = level + (1 if pool else 0)
        assert t[i].shape == (32 >> sh, 48 >> sh, cout), i
    assert last.shape == (32, 48, 3)
    # pooling of layer 1 is the 2 x 2 max of its convolution
    s, _ = net.per_layer(1, t[0])
    np.testing.assert_array_equal(t[1], U.pool2(np.maximum(s, 0.0)))
