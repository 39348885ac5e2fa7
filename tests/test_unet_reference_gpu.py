"""GPU: both UNet denoiser paths checked layer by layer against the float64 statement of the network (unet_ref.py).

Every intermediate tensor is read back through rc_debug_unet_tensor, and each layer is recomputed in float64 from the
DEVICE's own input tensors, so errors do not compound and the bounds are rigorous rounding-error bounds:
  K = 9 cin, A = sum |w x| + |b|, S = sum w x + b, R = max(0, S), E = (K + 2) 2^-24 A
  fp32 path (FFMA):         |dev - R| <= E  (+ sum |w| 4 2^-24 |f| over the features computed in-kernel, passes 0, 13)
  tensor-core path (fp16):  |dev - R| <= ulp16(R + 2E) + 2E  (the 2 allows an fp32 accumulator that truncates)
Pooled layers are compared with the 2 x 2 max of the bounds (max and ReLU are monotone and 1-Lipschitz), pass 15 with
output_hdr of the bounds (output_hdr is monotone).  The inputs are synthetic planes written straight into the frame
(no render, so the display transform is Standard with gamma 1) plus one 8-sample Cornell-box render.

Frame sizes and what they reach:
  1x1        rounded to 16 x 16; the level-4 grid is 1 x 1; one partial 128-pixel tile per row
  100x70     not a multiple of 16: zero features in the rounded margin
  272x48     level 0 = 2 tiles + 16 px, level 1 = 1 tile + 8 px, odd level-4 width (17)
  16x1200    narrow: the haloed TMA box spans ~7 image rows of the flattened tensor; ~4 tiles per CTA at level 0
  1920x1080  ~55 / 15 / 3.7 tiles per CTA at levels 0 / 1 / 2: the persistent loop, the accumulator parity and the ring
             wrap-arounds run.  Its layers are checked on a seeded set of >= 48 full rows each (first and last two
             included); every other size is checked completely.
"""
import numpy as np
import pytest

import unet_ref as U
from common import make_pair
from ray_b200 import capi, cuda, scenes
from test_parity_gpu import UNET_SHAPES, _cuda_render

pytestmark = pytest.mark.gpu

U24 = 2.0 ** -24
PATHS = {"fp32": capi.RC_UNET_FP32, "tc": capi.RC_UNET_TENSOR_CORES}
SIZES = [(1, 1), (100, 70), (272, 48), (16, 1200), (1920, 1080)]
SAMPLED_ROWS = 48  # per layer at 1920 x 1080


def ulp16(x):
    a = np.maximum(np.abs(x), 2.0 ** -14)
    return 2.0 ** (np.floor(np.log2(a)) - 10)


def ulp32(x):
    a = np.maximum(np.abs(x), 2.0 ** -126)
    return 2.0 ** (np.floor(np.log2(a)) - 23)


def synthetic_weights(seed=11):
    """He-scaled fp16 weights, N(0, 0.1) hidden biases; the last layer's channels are biased so that its outputs take
    every branch of output_hdr (X0 / OUT_NORM = 7.1e-4 and X1 / OUT_NORM = 0.118 are the knots)."""
    rng = np.random.default_rng(seed)
    out = []
    for i, (ci, co) in enumerate(UNET_SHAPES):
        w = rng.standard_normal((co, ci, 3, 3)) * np.sqrt(2.0 / (9 * ci))
        b = rng.standard_normal(co) * 0.1
        if i == 15:  # one channel near 0, one around the middle branch, one reaching the exponential branch
            w *= np.array([0.002, 0.05, 0.1])[:, None, None, None]
            b = np.array([0.0003, 0.05, 0.3])
        out.append((w.astype(np.float16), b.astype(np.float16)))
    return out


def synthetic_planes(w, h, seed):
    """FULL, BASE_COLOR, DEPTH_NORMALS planes: colour 90 % log-uniform in [1e-9, 1e4], 5 % exact 0, 5 % the knots
    Y0, Y1 and their float neighbours; albedo uniform in [0, 1]; unit normals; FULL.w uniform in [0, 1]."""
    rng = np.random.default_rng(seed)
    n = w * h * 3
    col = np.exp(rng.uniform(np.log(1e-9), np.log(1e4), n)).astype(np.float32)
    kind = rng.uniform(size=n)
    col[kind < 0.05] = 0.0
    knots = []
    for k in (U.Y0, U.Y1):
        k = np.float32(k)
        knots += [k, np.nextafter(k, np.float32(0)), np.nextafter(k, np.float32(1))]
    pick = (kind >= 0.05) & (kind < 0.10)
    col[pick] = np.array(knots, np.float32)[rng.integers(0, len(knots), int(pick.sum()))]
    full = np.zeros((h, w, 4), np.float32)
    full[..., :3] = col.reshape(h, w, 3)
    full[..., 3] = rng.uniform(0, 1, (h, w))
    alb = np.zeros((h, w, 4), np.float32)
    alb[..., :3] = rng.uniform(0, 1, (h, w, 3))
    nrm = rng.standard_normal((h, w, 3))
    nrm /= np.linalg.norm(nrm, axis=2, keepdims=True)
    dn = np.zeros((h, w, 4), np.float32)
    dn[..., :3] = nrm
    dn[..., 3] = rng.uniform(1, 10, (h, w))
    return full, alb, dn


class Case:
    """One frame in a CUDA context: the planes, the weights, and both paths run once with pass = -1."""

    def __init__(self, w, h, name, ctx=None, planes=None, layers=None, inv_gamma=1.0):
        self.w, self.h, self.name = w, h, name
        self.wr, self.hr = U.round16(w), U.round16(h)
        self.own_ctx = ctx is None
        if ctx is None:
            ctx = cuda.Context(0)
            ctx.resize(w, h)
        self.ctx = ctx
        if planes is None:
            planes = synthetic_planes(w, h, seed=w * 7919 + h)
            for which, p in zip((capi.RC_BUF_FULL, capi.RC_BUF_BASE_COLOR, capi.RC_BUF_DEPTH_NORMALS), planes):
                ctx.debug_write_plane(which, p)
        self.full, self.alb, self.dn = planes
        self.layers = layers or synthetic_weights()
        self.inv_gamma = inv_gamma
        ctx.unet_set_weights(self.layers)
        self.net = U.UNet(self.layers)
        self.feats = U.features(self.full, self.alb, self.dn)
        self.out = {}
        for path, flags in PATHS.items():
            self.run(path)
            self.out[path] = (ctx.readback(capi.RC_BUF_RAW), ctx.readback(capi.RC_BUF_FINAL))

    def run(self, path, rect=None, pass_index=-1):
        self.ctx.denoise_unet(rect or (0, 0, self.w, self.h), flags=PATHS[path], pass_index=pass_index)

    @property
    def sampled(self):
        return self.w * self.h > 1_000_000

    def close(self):
        if self.own_ctx:
            self.ctx.close()


@pytest.fixture(scope="module", params=[f"{w}x{h}" for w, h in SIZES] + ["cornell_100x70"])
def case(request):
    if request.param == "cornell_100x70":
        pair = make_pair(scenes.cornell_box(100, 70))
        _cuda_render(pair, 8)
        ctx = pair.ctx
        planes = tuple(ctx.readback(b) for b in (capi.RC_BUF_FULL, capi.RC_BUF_BASE_COLOR, capi.RC_BUF_DEPTH_NORMALS))
        assert pair.cam.view_transform == 0, "the float64 FINAL below is the Standard view transform"
        c = Case(100, 70, request.param, ctx=ctx, planes=planes,
                 inv_gamma=float(np.float32(1.0) / np.float32(pair.cam.gamma)))
        yield c
        pair.close()
        return
    w, h = (int(v) for v in request.param.split("x"))
    c = Case(w, h, request.param)
    yield c
    c.close()


# ---- reading the device's tensors on their logical grids ---------------------------------------------------------------
def _runs(rows):
    """Contiguous runs [a, b) of a sorted row list."""
    out = []
    for r in rows:
        if out and out[-1][1] == r:
            out[-1][1] = r + 1
        else:
            out.append([r, r + 1])
    return out


class Tensors:
    """The device tensors of one path as logical (rows, cols, channels) float64 grids: no border, real channels only.
    A tensor-core tensor stored already up-sampled is returned on its stored (2x) grid."""

    def __init__(self, case, path):
        self.c, self.path, self.flags = case, path, PATHS[path]

    def channels(self, t):
        return 9 if t == 15 else U.LAYERS[t][2]

    def nrows(self, t):
        n, _, _ = self.c.ctx.debug_unet_dims(t, self.flags)
        return n - 2 if self.path == "tc" else n

    def rows(self, t, a, b):
        """Logical rows [a, b) of tensor t, zero rows outside the grid (the convolution's zero padding)."""
        n = self.nrows(t)
        lo, hi = max(a, 0), min(b, n)
        ctx = self.c.ctx
        if self.path == "tc":
            raw = ctx.debug_unet_tensor(t, self.flags, (lo + 1, max(hi - lo, 0)))
            core = raw[:, 1:-1, :self.channels(t)]
        else:
            core = ctx.debug_unet_tensor(t, self.flags, (lo, max(hi - lo, 0)))
        cols, ch = core.shape[1], core.shape[2]
        out = np.zeros((b - a, cols, ch))
        if hi > lo:
            out[lo - a:hi - a] = core
        return out

    def main_input(self, i, a, b):
        """Layer i's first input on its convolution grid, rows [a, b)."""
        c = self.c
        if i == 0:
            if self.path == "tc":
                return self.rows(15, a, b)
            return _feat_rows(c.feats, a, b)
        if U.LAYERS[i][4] and self.path == "fp32":  # up-sample the coarse tensor
            ca, cb = a >> 1, ((b - 1) >> 1) + 1
            coarse = self.rows(i - 1, ca, cb)
            return U.up2(coarse)[a - 2 * ca:b - 2 * ca]
        return self.rows(i - 1, a, b)

    def skip_input(self, i, a, b):
        if i not in U.SKIP:
            return None
        src = U.SKIP[i]
        if src == "input":
            return self.rows(15, a, b) if self.path == "tc" else _feat_rows(self.c.feats, a, b)
        return self.rows(src, a, b)


def _feat_rows(f, a, b):
    out = np.zeros((b - a,) + f.shape[1:])
    lo, hi = max(a, 0), min(b, f.shape[0])
    out[lo - a:hi - a] = f[lo:hi]
    return out


def _row_sample(n, seed):
    """All rows, or at 1920 x 1080 a seeded set of SAMPLED_ROWS rows that includes the first and last two."""
    if n <= SAMPLED_ROWS + 4:
        return list(range(n))
    rng = np.random.default_rng(seed)
    pick = set(rng.choice(np.arange(2, n - 2), SAMPLED_ROWS - 4, replace=False).tolist()) | {0, 1, n - 2, n - 1}
    return sorted(pick)


def _fail_msg(path, i, what, dev, lo, hi, bad):
    idx = tuple(int(v) for v in np.argwhere(bad)[0])
    return (f"{path} path, pass {i} {what}: {int(bad.sum())} of {bad.size} values outside the bound; first at "
            f"(row, col, channel) = {idx}: device {dev[idx]!r}, reference interval [{lo[idx]!r}, {hi[idx]!r}]")


def _layer_bounds(case, tens, path, i, ca, cb):
    """float64 [lo, hi] of layer i's ReLU output at convolution rows [ca, cb), before pooling."""
    net = case.net
    cin1, cin2, _, _, _, _ = U.LAYERS[i]
    x1 = tens.main_input(i, ca - 1, cb + 1)
    x2 = tens.skip_input(i, ca - 1, cb + 1)
    s, a = net.per_layer(i, x1, x2, pad_rows=False)
    e = (9 * (cin1 + cin2) + 2) * U24 * a
    if path == "fp32":
        if i == 0:  # features computed in fp32 inside the kernel: the main input of pass 0, the skip input of 13
            e = e + 4 * U24 * net.abs_conv(i, x1, np.zeros(x1.shape[:2] + (0,)), pad_rows=False)
        elif i == 13:
            e = e + 4 * U24 * net.abs_conv(i, np.zeros_like(x1), x2, pad_rows=False)
        return np.maximum(s - e, 0.0), np.maximum(s + e, 0.0), s, e
    lo, hi = np.maximum(s - 2 * e, 0.0), np.maximum(s + 2 * e, 0.0)
    if i == 15:
        return lo, hi, s, 2 * e
    u = ulp16(hi)
    return np.maximum(lo - u, 0.0), hi + u, s, 2 * e


def check_layer(case, path, i):
    tens = Tensors(case, path)
    ctx, flags = case.ctx, PATHS[path]
    _, _, cout, level, _, pool = U.LAYERS[i]
    h_conv = case.hr >> level
    seed = 1000 * i + (7 if path == "tc" else 3)
    if i == 15:
        ys = _row_sample(case.h, seed) if case.sampled else list(range(case.h))
    else:
        ys = _row_sample(h_conv >> (1 if pool else 0), seed) if case.sampled else list(range(h_conv >> (1 if pool else 0)))
    for ya, yb in _runs(ys):
        ca, cb = (2 * ya, 2 * yb) if pool else (ya, yb)
        lo, hi, s, e = _layer_bounds(case, tens, path, i, ca, cb)
        if i == 15:
            raw = ctx.readback(capi.RC_BUF_RAW, (0, ya, case.w, yb - ya)).astype(np.float64)
            final = ctx.readback(capi.RC_BUF_FINAL, (0, ya, case.w, yb - ya)).astype(np.float64)
            rlo = U.output_hdr(lo[:, :case.w])
            rhi = U.output_hdr(hi[:, :case.w])
            rlo, rhi = rlo - 8 * ulp32(rlo), rhi + 8 * ulp32(rhi)
            dev = raw[..., :3]
            bad = (dev < rlo) | (dev > rhi) | ~np.isfinite(dev)
            assert not bad.any(), _fail_msg(path, i, f"RAW rows [{ya}, {yb})", dev, rlo, rhi, bad)
            want = U.standard_transform(dev, case.inv_gamma)
            err = np.abs(final[..., :3] - want)
            assert err.max() <= 1e-6, (f"{path} path, pass 15 FINAL rows [{ya}, {yb}): {err.max():g} from the Standard "
                                       f"transform of RAW at {np.unravel_index(err.argmax(), err.shape)}")
            fw = case.full[ya:yb, :, 3]
            assert raw[..., 3].astype(np.float32).tobytes() == fw.tobytes(), f"{path}: RAW.w is not FULL.w"
            assert final[..., 3].astype(np.float32).tobytes() == np.clip(fw, 0, 1).tobytes(), f"{path}: FINAL.w"
            continue
        if pool:
            lo, hi = U.pool2(lo), U.pool2(hi)
        if path == "tc" and i + 1 < 16 and U.LAYERS[i + 1][4]:  # stored up-sampled: 4 equal replicas per pixel
            st = tens.rows(i, 2 * ya, 2 * yb)
            reps = [st[dy::2, dx::2] for dy in (0, 1) for dx in (0, 1)]
            for r in reps[1:]:
                assert np.array_equal(r, reps[0]), f"tc path, pass {i}: the up-sampled replicas differ (rows [{ya}, {yb}))"
            dev = reps[0]
        else:
            dev = tens.rows(i, ya, yb)
        bad = (dev < lo) | (dev > hi) | ~np.isfinite(dev)
        assert not bad.any(), _fail_msg(path, i, f"rows [{ya}, {yb})", dev, lo, hi, bad)


def check_tc_storage(case, t):
    """A tensor-core tensor's zero border and padded channels are exactly zero (they are the convolution's padding)."""
    ctx, flags = case.ctx, PATHS["tc"]
    n, cols, cs = ctx.debug_unet_dims(t, flags)
    ch = 9 if t == 15 else U.LAYERS[t][2]
    rows = _row_sample(n, 99 + t) if case.sampled else list(range(n))
    for a, b in _runs(rows):
        st = ctx.debug_unet_tensor(t, flags, (a, b - a))
        assert not st[:, :, ch:].any(), f"tc tensor {t}: a padded channel (>= {ch}) is not zero in rows [{a}, {b})"
        assert not st[:, 0].any() and not st[:, cols - 1].any(), f"tc tensor {t}: border column not zero, rows [{a}, {b})"
        if a == 0:
            assert not st[0].any(), f"tc tensor {t}: top border row not zero"
        if b == n:
            assert not st[-1].any(), f"tc tensor {t}: bottom border row not zero"


@pytest.mark.parametrize("path", list(PATHS))
def test_every_layer_is_within_its_rounding_bound(case, path):
    case.run(path)  # RAW / FINAL are shared by the two paths
    if path == "tc":
        for t in range(16):
            check_tc_storage(case, t)
        # the network input: fp16 of the float64 features
        tens = Tensors(case, "tc")
        ys = _row_sample(case.hr, 5) if case.sampled else list(range(case.hr))
        for a, b in _runs(ys):
            dev, f = tens.rows(15, a, b), case.feats[a:b]
            bad = np.abs(dev - f) > ulp16(f)
            assert not bad.any(), _fail_msg("tc", 15, f"network input rows [{a}, {b})", dev, f - ulp16(f), f + ulp16(f), bad)
    for i in range(16):
        check_layer(case, path, i)


def test_inputs_exercise_every_branch(case):
    """The synthetic inputs reach what the bounds above rely on: every branch of both transfer functions and ReLUs that
    clip on both sides in every hidden layer."""
    if case.name.startswith("cornell") or case.w * case.h < 1000:
        pytest.skip("a rendered image or a frame too small to cover every branch")
    col = case.full[..., :3].astype(np.float64)
    frac_in = [float(np.mean(m)) for m in (col <= U.Y0, (col > U.Y0) & (col <= U.Y1), col > U.Y1)]
    assert min(frac_in) >= 0.01, f"input_hdr branch fractions {frac_in}"
    raw = case.out["fp32"][0][..., :3].astype(np.float64)
    k0, k1 = float(U.output_hdr(U.X0 / U.OUT_NORM)), float(U.output_hdr(U.X1 / U.OUT_NORM))
    frac_out = [float(np.mean(m)) for m in ((raw > 0) & (raw <= k0), (raw > k0) & (raw <= k1), raw > k1)]
    assert min(frac_out) >= 0.01, f"output_hdr branch fractions {frac_out}"
    for path, flags in PATHS.items():
        for t in range(15):
            n = case.ctx.debug_unet_dims(t, flags)[0]
            rows = (0, n) if not case.sampled or n <= 16 else (n // 2 - 8, 16)
            st = case.ctx.debug_unet_tensor(t, flags, rows)
            ch = U.LAYERS[t][2]
            core = st[:, 1:-1, :ch] if path == "tc" else st
            zeros = float(np.mean(core == 0))
            assert 0.05 <= zeros <= 0.95, f"{path} tensor {t}: {zeros:.3f} of the values are exact zeros"


def test_end_to_end_matches_float64_network(case):
    """The whole network against the float64 reference: the fp32 path to 2e-4 relative to (1 + |ref|); the tensor-core
    path against the reference rounded to fp16 between layers, max 3e-2 and mean 2e-3 relative."""
    if case.sampled:
        pytest.skip("1920x1080 is checked layer by layer on sampled rows")
    _, last = case.net.forward(case.feats)
    ref = U.output_hdr(last[:case.h, :case.w])
    raw = case.out["fp32"][0][..., :3].astype(np.float64)
    err = np.abs(raw - ref) / (1.0 + np.abs(ref))
    print(f"unet fp32 {case.name}: max rel {err.max():.3g} mean rel {err.mean():.3g}")
    assert err.max() <= 2e-4, f"fp32 path {case.name}: max rel {err.max():g} at {np.unravel_index(err.argmax(), err.shape)}"
    _, last16 = case.net.forward(case.feats, emulate_fp16=True)
    ref16 = U.output_hdr(last16[:case.h, :case.w])
    raw = case.out["tc"][0][..., :3].astype(np.float64)
    err = np.abs(raw - ref16) / (1.0 + np.abs(ref16))
    print(f"unet tc {case.name}: max rel {err.max():.3g} mean rel {err.mean():.3g}")
    assert err.max() <= 3e-2 and err.mean() <= 2e-3, f"tc path {case.name}: max rel {err.max():g}, mean rel {err.mean():g}"


def _partition(w, h, xs, ys):
    xe, ye = [0] + [x for x in xs if 0 < x < w] + [w], [0] + [y for y in ys if 0 < y < h] + [h]
    return [(x0, y0, x1 - x0, y1 - y0) for y0, y1 in zip(ye, ye[1:]) for x0, x1 in zip(xe, xe[1:])]


PARTITIONS = {"aligned": ((48, 160), (16, 32)), "odd": ((37, 81, 150), (19,))}


@pytest.mark.parametrize("path", list(PATHS))
def test_calling_forms_equal_the_full_run(case, path):
    """Passes 0..15 one at a time, and pass-major calls over a partition of the frame (region origins on the 16-pixel
    grid, and odd ones), give the full-frame pass = -1 result bit for bit."""
    if case.name not in ("272x48", "100x70"):
        pytest.skip("calling forms are checked at 272x48 and 100x70")
    ctx = case.ctx
    want_raw, want_final = case.out[path]
    n_t = 16 if path == "tc" else 15
    case.run(path)
    want_t = [ctx.debug_unet_tensor(t, PATHS[path]) for t in range(n_t)]
    for p in range(16):
        case.run(path, pass_index=p)
    assert np.array_equal(ctx.readback(capi.RC_BUF_RAW), want_raw), f"{path}: passes one at a time, RAW"
    assert np.array_equal(ctx.readback(capi.RC_BUF_FINAL), want_final), f"{path}: passes one at a time, FINAL"
    for t in range(n_t):
        assert np.array_equal(ctx.debug_unet_tensor(t, PATHS[path]), want_t[t]), f"{path}: passes one at a time, tensor {t}"
    for name, (xs, ys) in PARTITIONS.items():
        rects = _partition(case.w, case.h, xs, ys)
        # leave tensors and outputs of a different input behind, so a region that computes too little shows
        ctx.debug_write_plane(capi.RC_BUF_FULL, case.full[::-1, ::-1].copy())
        case.run(path)
        ctx.debug_write_plane(capi.RC_BUF_FULL, case.full)
        for p in range(16):
            for r in rects:
                case.run(path, rect=r, pass_index=p)
        raw, final = ctx.readback(capi.RC_BUF_RAW), ctx.readback(capi.RC_BUF_FINAL)
        bad = np.argwhere((raw != want_raw).any(axis=2))
        assert not len(bad), (f"{path} path, {name} partition {rects}: RAW differs from the full-frame call at "
                              f"{len(bad)} pixels, first (y, x) = {tuple(bad[0])}")
        assert np.array_equal(final, want_final), f"{path} path, {name} partition: FINAL differs"
