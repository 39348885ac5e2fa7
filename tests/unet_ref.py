"""A float64 statement of the UNet denoiser, written from the network's description in rt_unet.cuh (pass table,
transfer functions, feature layout, padding, pooling, up-sampling, concatenation order) and not from its kernels.

The tests of both device paths (tests/test_unet_reference_gpu.py) compare with it layer by layer and end to end.
Activations are (rows, cols, channels) float64 arrays on the frame rounded up to a multiple of 16.
"""
import numpy as np
import torch

# (cin1, cin2, cout, level, up, pool) of the 16 convolutions in pass order.  cin1: channels of the main input (the
# previous tensor, up-sampled 2x when `up`); cin2: of the skip tensor concatenated after it; level: log2 of the
# down-scale of the convolution grid; pool: 2 x 2 max pooling of the output.
LAYERS = [
    (9, 0, 32, 0, False, False),  # enc_conv0: the 9 input features
    (32, 0, 32, 0, False, True),  # enc_conv1
    (32, 0, 48, 1, False, True),  # enc_conv2
    (48, 0, 64, 2, False, True),  # enc_conv3
    (64, 0, 80, 3, False, True),  # enc_conv4
    (80, 0, 96, 4, False, False),  # enc_conv5a
    (96, 0, 96, 4, False, False),  # enc_conv5b
    (96, 64, 112, 3, True, False),  # dec_conv4a: up(5b) ++ enc_conv3's pooled output
    (112, 0, 112, 3, False, False),  # dec_conv4b
    (112, 48, 96, 2, True, False),  # dec_conv3a: up(4b) ++ enc_conv2
    (96, 0, 96, 2, False, False),  # dec_conv3b
    (96, 32, 64, 1, True, False),  # dec_conv2a: up(3b) ++ enc_conv1
    (64, 0, 64, 1, False, False),  # dec_conv2b
    (64, 9, 64, 0, True, False),  # dec_conv1a: up(2b) ++ the network input
    (64, 0, 32, 0, False, False),  # dec_conv1b
    (32, 0, 3, 0, False, False),  # dec_conv0 -> output_hdr
]
SKIP = {7: 3, 9: 2, 11: 1, 13: "input"}  # decoder layer -> the tensor concatenated after its up-sampled input

_f32 = np.float32
# HDR transfer function constants (Convolution.h), as the float literals of rt_unet.cuh
A, B, C, D, E, F, G = (float(_f32(x)) for x in (1.41283765e+03, 1.64593172e+00, 4.31384981e-01, -2.94139609e-03,
                                                 1.92653254e-01, 6.26026094e-03, 9.98620152e-01))
Y0, Y1, X0, X1 = (float(_f32(x)) for x in (1.57945760e-06, 3.22087631e-02, 2.23151711e-03, 3.70974749e-01))
IN_NORM, OUT_NORM = float(_f32(0.318967164)), float(_f32(3.13511896))
INV_C = float(_f32(1.0) / _f32(C))  # `1.0f / c`: the exponent is itself a float
SRGB_KNOT = float(_f32(0.0031308))
SRGB_EXP = float(_f32(1.0) / _f32(2.4))


def input_hdr(v):
    """The transfer function applied to the colour input (three branches split at Y0 and Y1)."""
    v = np.asarray(v, np.float64)
    with np.errstate(all="ignore"):
        return np.where(v <= Y0, A * v * IN_NORM,
                        np.where(v <= Y1, (B * np.power(np.maximum(v, 0.0), C) + D) * IN_NORM,
                                 (E * np.log(np.maximum(v + F, 1e-300)) + G) * IN_NORM))


def output_hdr(v):
    """Inverse of input_hdr, applied to the last layer's output (branches split at X0 and X1 of v * OUT_NORM)."""
    x = np.asarray(v, np.float64) * OUT_NORM
    with np.errstate(all="ignore"):
        return np.where(x <= X0, x / A,
                        np.where(x <= X1, np.power(np.maximum((x - D) / B, 0.0), INV_C), np.exp((x - G) / E) - F))


def output_branch(v):
    """0, 1 or 2: which branch of output_hdr a last-layer value takes."""
    x = np.asarray(v, np.float64) * OUT_NORM
    return np.where(x <= X0, 0, np.where(x <= X1, 1, 2))


def standard_transform(c, inv_gamma=1.0):
    """FINAL from RAW under the Standard view transform: the sRGB OETF, then 1 / gamma, then a clamp to [0, 1]."""
    c = np.asarray(c, np.float64)
    with np.errstate(all="ignore"):
        t = np.where(c < SRGB_KNOT, float(_f32(12.92)) * c,
                     float(_f32(1.055)) * np.power(np.maximum(c, 0.0), SRGB_EXP) - float(_f32(0.055)))
        if inv_gamma != 1.0:
            t = np.power(t, float(inv_gamma))
    return np.clip(t, 0.0, 1.0)


def round16(n):
    return (n + 15) // 16 * 16


def features(full, albedo, depth_normals):
    """The 9 network inputs on the rounded frame: input_hdr(colour), albedo, 0.5 n + 0.5; zero outside the frame."""
    h, w = full.shape[:2]
    f = np.zeros((round16(h), round16(w), 9))
    f[:h, :w, 0:3] = input_hdr(full[..., :3])
    f[:h, :w, 3:6] = albedo[..., :3]
    f[:h, :w, 6:9] = 0.5 * np.asarray(depth_normals[..., :3], np.float64) + 0.5
    return f


def conv3x3(x, w, b=None, pad_rows=True):
    """3 x 3 cross-correlation of x (rows, cols, cin) with OIHW weights w (cout, cin, 3, 3), zero padding of one pixel
    at the left and right (and top and bottom with pad_rows; without, the first and last rows of x are the halo and
    the result has two rows fewer), plus bias b.  Returns (rows, cols, cout)."""
    t = torch.from_numpy(np.ascontiguousarray(np.asarray(x, np.float64).transpose(2, 0, 1)))[None]
    k = torch.from_numpy(np.asarray(w, np.float64))
    bb = None if b is None else torch.from_numpy(np.asarray(b, np.float64))
    y = torch.nn.functional.conv2d(t, k, bias=bb, padding=(1, 1) if pad_rows else (0, 1))
    return y[0].permute(1, 2, 0).numpy()


def pool2(x):
    """2 x 2 max pooling (rows and cols even)."""
    r, c = x.shape[0] // 2, x.shape[1] // 2
    return x[:2 * r, :2 * c].reshape(r, 2, c, 2, -1).max(axis=(1, 3))


def up2(x):
    """Nearest 2x up-sampling."""
    return np.repeat(np.repeat(x, 2, axis=0), 2, axis=1)


def to_fp16(x):
    return np.asarray(x, np.float64).astype(np.float16).astype(np.float64)


class UNet:
    """The network with one weight set: 16 x (fp16 OIHW weights, fp16 biases), as rc_unet_set_weights takes them."""

    def __init__(self, layers):
        assert len(layers) == 16
        self.w = [np.asarray(w, np.float16).astype(np.float64) for w, _ in layers]
        self.b = [np.asarray(b, np.float16).astype(np.float64) for _, b in layers]
        for i, (cin1, cin2, cout, *_rest) in enumerate(LAYERS):
            assert self.w[i].shape == (cout, cin1 + cin2, 3, 3) and self.b[i].shape == (cout,), i

    def per_layer(self, i, x1, x2=None, pad_rows=True, bounds=True):
        """Layer i on given inputs, both on its convolution grid: x1 the main input (already up-sampled for a decoder
        layer), x2 the skip tensor.  Returns (S, Aabs): the pre-activation sum of w x + b and the sum of |w x| + |b|
        (None with bounds=False), before ReLU and pooling."""
        x = x1 if x2 is None else np.concatenate([x1, x2], axis=2)
        s = conv3x3(x, self.w[i], self.b[i], pad_rows)
        if not bounds:
            return s, None
        return s, conv3x3(np.abs(x), np.abs(self.w[i]), np.abs(self.b[i]), pad_rows)

    def abs_conv(self, i, x1, x2, pad_rows=True):
        """sum of |w| |x| without the bias, over the inputs given (zeros elsewhere)."""
        x = np.concatenate([x1, x2], axis=2)
        return conv3x3(np.abs(x), np.abs(self.w[i]), None, pad_rows)

    def forward(self, feats, emulate_fp16=False):
        """All 16 layers on the network input `feats` (rounded frame).  Returns (tensors, last): tensors[i] is the output
        of pass i < 15 after ReLU and pooling, `last` the ReLU output of pass 15 (apply output_hdr for RAW).  With
        emulate_fp16 the features and every hidden layer's output are rounded to fp16, as the tensor-core path stores
        them."""
        x0 = to_fp16(feats) if emulate_fp16 else np.asarray(feats, np.float64)
        out = []
        for i, (_cin1, _cin2, _cout, _level, up, pool) in enumerate(LAYERS):
            x1 = x0 if i == 0 else out[i - 1]
            if up:
                x1 = up2(x1)
            x2 = None
            if i in SKIP:
                x2 = x0 if SKIP[i] == "input" else out[SKIP[i]]
            s, _ = self.per_layer(i, x1, x2, bounds=False)
            y = np.maximum(s, 0.0)
            if pool:
                y = pool2(y)
            if emulate_fp16 and i < 15:
                y = to_fp16(y)
            out.append(y)
        return out[:15], out[15]
