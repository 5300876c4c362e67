"""-m gpu: --precision tf32 for cunet/art (fp32 activations, tcgen05 kind::tf32 convolutions, fp32 epilogues).

Per layer: the five layer kinds through the tf32 kernel (w2x_run_conv_layer_f32) against torch.nn.functional in float64, with inputs and
weights that TF32 represents exactly, so the only error left is the fp32 accumulation order.  Whole model: tf32 engines against the
fp32 oracle at the fp16 suite's thresholds (infer: at the measured bound given there), every entry point that takes a loaded engine, and the case tf32 exists for -- activations
beyond the fp16 range."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import onnx_io, tiling
from oracle.models import make_model

pytestmark = pytest.mark.gpu


def _tf32(a):
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0xFFF + ((u >> 13) & 1)) & 0xFFFFE000).astype(np.uint32).view(np.float32)


def _rand(rng, shape, scale):
    return _tf32(rng.uniform(-1, 1, size=shape) * scale)


def _t64(a, perm=True):
    t = torch.from_numpy(np.asarray(a, np.float64))
    return t.permute(0, 3, 1, 2) if perm else t


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous().numpy()


def _case(kind, n, h, w, cin, cout, xscale=1.0, seed=7):
    """-> (x NHWC f32, packed weights f32, bias[npad], skip or None, reference NHWC f64, magnitude NHWC f64 = the same sum over |terms|)"""
    rng = np.random.default_rng(seed)
    x = _rand(rng, (n, h, w, cin), xscale)
    xt, xa = _t64(x), _t64(np.abs(x))
    lrelu = lambda t: F.leaky_relu(t, 0.1)
    ceil16 = lambda c: (c + 15) // 16 * 16
    if kind in (0, 1):
        k = 3 if kind == 0 else 2
        wt = _rand(rng, (cout, cin, k, k), 1 / np.sqrt(k * k * cin))
        b = _tf32(rng.uniform(-0.1, 0.1, size=cout))
        s = 1 if kind == 0 else 2
        ref = lrelu(F.conv2d(xt, _t64(wt, False), _t64(b, False), stride=s))
        mag = F.conv2d(xa, _t64(np.abs(wt), False), _t64(np.abs(b), False), stride=s)
        wp = np.zeros((ceil16(cout), k * k * cin), np.float32)
        wp[:cout] = wt.transpose(0, 2, 3, 1).reshape(cout, k * k * cin)
        bp = np.zeros(ceil16(cout), np.float32); bp[:cout] = b
        return x, wp, bp, None, _nhwc(ref), _nhwc(mag)
    if kind == 2:
        wt = _rand(rng, (cin, cout, 2, 2), 1 / np.sqrt(cin))
        b = _tf32(rng.uniform(-0.1, 0.1, size=cout))
        skip = _rand(rng, (n, 2 * h + 8, 2 * w + 8, cout), 0.5)
        st = _t64(skip)[:, :, 4:-4, 4:-4]
        ref = lrelu(F.conv_transpose2d(xt, _t64(wt, False), _t64(b, False), stride=2)) + st
        mag = F.conv_transpose2d(xa, _t64(np.abs(wt), False), _t64(np.abs(b), False), stride=2) + st.abs()
        wp = np.ascontiguousarray(wt.transpose(2, 3, 1, 0).reshape(4 * cout, cin))
        return x, wp, np.tile(b, 4), skip, _nhwc(ref), _nhwc(mag)
    if kind == 3:
        wt = _rand(rng, (cin, 3, 4, 4), 1 / np.sqrt(4 * cin))
        b = _tf32(rng.uniform(-0.1, 0.1, size=3))
        ref = F.conv_transpose2d(xt, _t64(wt, False), _t64(b, False), stride=2, padding=3)
        mag = F.conv_transpose2d(xa, _t64(np.abs(wt), False), _t64(np.abs(b), False), stride=2, padding=3)
        wp = np.zeros((16, 4 * cin), np.float32)
        bp = np.zeros(16, np.float32)
        for py in range(2):
            for px in range(2):
                for co in range(3):
                    row = (py * 2 + px) * 4 + co
                    bp[row] = b[co]
                    for wy in range(2):
                        for wx in range(2):
                            wp[row, (wy * 2 + wx) * cin:(wy * 2 + wx + 1) * cin] = wt[:, co, 2 + py - 2 * wy, 2 + px - 2 * wx]
        return x, wp, bp, None, _nhwc(ref), _nhwc(mag)
    if kind == 4:
        wt = _rand(rng, (3, cin, 3, 3), 1 / np.sqrt(9 * cin))
        b = _tf32(rng.uniform(0.2, 0.6, size=3))
        skip = np.zeros((n, h - 2 + 40, w - 2 + 40, 4), np.float32)
        skip[..., :3] = _rand(rng, (n, h - 2 + 40, w - 2 + 40, 3), 0.5)
        st = _t64(skip[..., :3])[:, :, 20:-20, 20:-20]
        ref = torch.clamp(F.conv2d(xt, _t64(wt, False), _t64(b, False)) + st, 0, 1)
        mag = F.conv2d(xa, _t64(np.abs(wt), False), _t64(np.abs(b), False)) + st.abs()
        wp = np.zeros((16, 9 * cin), np.float32)
        wp[:3] = wt.transpose(0, 2, 3, 1).reshape(3, 9 * cin)
        bp = np.zeros(16, np.float32); bp[:3] = b
        return x, wp, bp, skip, _nhwc(ref), _nhwc(mag)
    raise ValueError(kind)


# the shapes of tests/test_gpu_conv.py::CASES (the head-kernel rows there have no tf32 counterpart: their shapes run through the same
# tf32 kernel here), plus one layer whose activations are near 1e5, beyond the fp16 range
CASES = [
    (0, 1, 20, 24, 64, 64, 1.0), (0, 8, 100, 100, 64, 64, 1.0), (0, 1, 60, 52, 128, 64, 1.0), (0, 3, 45, 77, 64, 128, 1.0),
    (0, 2, 61, 45, 32, 64, 1.0), (0, 1, 126, 126, 64, 128, 1.0), (0, 1, 117, 117, 128, 256, 1.0), (0, 1, 115, 115, 256, 128, 1.0),
    (0, 1, 226, 226, 128, 64, 1.0), (1, 2, 60, 60, 64, 64, 1.0), (1, 1, 234, 234, 128, 128, 1.0), (2, 2, 26, 26, 64, 64, 1.0),
    (2, 1, 17, 17, 128, 128, 1.0), (2, 1, 113, 113, 128, 128, 1.0), (3, 2, 50, 50, 64, 3, 1.0), (4, 2, 58, 58, 64, 3, 1.0),
    (3, 3, 33, 17, 64, 3, 1.0), (4, 3, 26, 146, 64, 3, 1.0),
    (0, 2, 40, 40, 64, 64, 1.0e5),
]


@pytest.mark.parametrize("kind,n,h,w,cin,cout,xscale", CASES)
def test_tf32_layer_matches_torch_fp64(kind, n, h, w, cin, cout, xscale, built_lib):
    import w2x
    x, wp, bp, skip, ref, mag = _case(kind, n, h, w, cin, cout, xscale)
    got = w2x.run_conv_layer_f32(kind, x, wp, bp, cout, skip=skip).astype(np.float64)
    c = ref.shape[-1]
    assert got.shape[:3] == ref.shape[:3]
    err = np.abs(got[..., :c] - ref)
    # TF32 products of TF32 inputs are exact in fp32; what remains is fp32 accumulation: 2^-16 of the magnitude sum. fp16 storage of the
    # output alone (up to 2^-11 relative) would not meet this.
    tol = 2.0 ** -16 * mag + 1e-6
    assert (err <= tol).all(), (float(err.max()), float((err / tol).max()))
    if xscale > 65504:
        assert np.abs(ref).max() > 65504   # the case really leaves the fp16 range
    if got.shape[-1] > c:
        assert (got[..., c:] == 0).all()


# ---- whole model ---------------------------------------------------------------------------------------------------------------
def _psnr(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


def _engine(path, scale, tile, batch, blend=1 / 16, tta=False, precision=None, device=0):
    import w2x
    precision = w2x.PRECISION_TF32 if precision is None else precision
    e = w2x.Img2Img()
    msgs = []
    e.setMessageCallback(lambda s, m: msgs.append((s, m)))
    assert e.build(path, w2x.BuildConfig.fixed(batch, tile, device=device, precision=precision)), msgs
    assert e.load(path, w2x.RenderConfig(deviceId=device, precision=precision, batchSize=batch, height=tile, width=tile, scaling=scale,
                                         overlap=(blend, blend), tta=tta)), msgs
    return e, msgs


def _model_fn(model_t):
    def f(x):
        with torch.no_grad():
            return model_t(torch.from_numpy(np.ascontiguousarray(x))).numpy()
    return f


def _meets_render_bar(dst, ref):
    diff = np.abs(dst.astype(np.int32) - ref.astype(np.int32))
    return (diff <= 1).mean() >= 0.999 and _psnr(dst, ref) >= 50, ((diff <= 1).mean(), int(diff.max()), _psnr(dst, ref))


@pytest.mark.parametrize("scale,tile", [(2, 64), (1, 128), (2, 128)])
def test_tf32_infer_matches_fp32_oracle(scale, tile, built_lib, models_dir):
    model_t, path = models_dir[1][scale]
    e, msgs = _engine(path, scale, tile, 2)
    x = np.random.default_rng(0).random((2, 3, tile, tile), dtype=np.float32)
    x = (np.rint(x * 255) / 255).astype(np.float32)
    y = e.infer(x)
    assert y is not None, msgs
    ref = _model_fn(model_t)(x)
    err = np.abs(y - ref)
    # The fp16 suite's bar is 2.5e-3.  Measured here on a B200: 2.8e-3 to 2.9e-3.  The activations are stored as full fp32 and the tensor
    # core drops their low 13 bits (truncation, not rounding), a bias the fp16 path's round-to-nearest storage does not have; rounding
    # the stored activations to TF32 would remove it at the cost of fp32 outputs per layer (test_tf32_layer_matches_torch_fp64).
    # 3.5e-3 stays below 1 LSB of the u8 output (3.9e-3).
    assert err.max() < 3.5e-3, err.max()
    assert _psnr(y * 255, ref * 255) > 55
    e.close()


@pytest.mark.parametrize("w,h,scale,tile,batch,blend,tta", [
    (256, 256, 2, 64, 1, 1 / 16, False),     # cfg1 shape
    (150, 97, 2, 64, 4, 1 / 8, False),       # padding slots in the last batch, ragged edges
    (90, 70, 2, 64, 3, 0.0, False),          # no blending
    (420, 400, 1, 400, 2, 1 / 16, False),    # cunet 1x, tile 400
    (150, 100, 1, 128, 4, 1 / 16, True),     # TTA
])
def test_tf32_render_matches_oracle(w, h, scale, tile, batch, blend, tta, built_lib, models_dir):
    model_t, path = models_dir[1][scale]
    e, msgs = _engine(path, scale, tile, batch, blend, tta)
    src = tiling.synthetic_frame(w, h, 5)
    dst = e.render(src)
    assert dst is not None, msgs
    ref = tiling.render(src, _model_fn(model_t), tile, e.output_tile_size, scale, blend, batch, tta=tta)
    assert dst.shape == ref.shape == (h * scale, w * scale, 3)
    ok, info = _meets_render_bar(dst, ref)
    assert ok, info
    assert np.array_equal(e.render(src), dst)                  # a re-render is byte-identical
    e.close()


def test_tf32_layers_run_the_tf32_kernels(built_lib, models_dir):
    for scale in (1, 2):
        _, path = models_dir[1][scale]
        e, _ = _engine(path, scale, 64, 2)
        kernels = []
        i = 0
        while (k := e.layer_kernel(i)) is not None:
            kernels.append(k)
            i += 1
        assert len(kernels) == 22
        for i, k in enumerate(kernels):
            want = "first-layer fp32" if i in (0, 8) else "igemm-tf32"   # the two RGB first layers run on the CUDA cores
            assert k.startswith(want), (i, k)
        e.close()


def test_tf32_submit_wait_equals_render(built_lib, models_dir):
    import w2x
    _, path = models_dir[1][2]
    e, msgs = _engine(path, 2, 64, 4)
    frames = [tiling.synthetic_frame(120, 80, s) for s in range(4)]
    sync = [e.render(f).copy() for f in frames]
    pin_in = [w2x.PinnedArray((80, 120, 3)) for _ in frames]
    pin_out = [w2x.PinnedArray((160, 240, 3)) for _ in frames]
    tickets = []
    for f, pi, po in zip(frames, pin_in, pin_out):
        pi.array[...] = f
        tickets.append(e.submit(pi.ptr, 120, 80, po.ptr))
        assert tickets[-1] >= 0, msgs
    for t, po, s in zip(tickets, pin_out, sync):
        assert e.wait(t)
        assert np.array_equal(po.array, s)
    e.close()
    for p in pin_in + pin_out:
        p.free()


@pytest.mark.parametrize("nbands,tta,scale", [(2, False, 2), (3, False, 2), (2, True, 1)])
def test_tf32_banded_on_one_gpu_is_byte_identical(nbands, tta, scale, built_lib, models_dir):
    import w2x
    _, path = models_dir[1][scale]
    tile = 128 if scale == 1 else 64
    engines = [_engine(path, scale, tile, 3, tta=tta)[0] for _ in range(nbands)]
    for (w, h) in [(150, 230), (70, 331)]:
        src = tiling.synthetic_frame(w, h, 7)
        ref = engines[0].render(src)
        got = w2x.render_banded(engines, src)
        assert got is not None, engines[0].last_error
        assert np.array_equal(got, ref), (w, h)
    for e in engines:
        e.close()


def test_banded_refuses_mixed_precisions(built_lib, models_dir):
    import w2x
    _, path = models_dir[1][2]
    a, _ = _engine(path, 2, 64, 3, precision=w2x.PRECISION_FP16)
    b, _ = _engine(path, 2, 64, 3)
    assert w2x.render_banded([a, b], tiling.synthetic_frame(150, 230, 7)) is None
    assert "identically configured" in a.last_error
    a.close()
    b.close()


def test_swin_unet_tf32_is_refused_by_name(built_lib, tmp_path):
    import w2x
    import __graft_entry__
    _, path = __graft_entry__.make_synthetic_model(str(tmp_path), 2, 0, model="swin_unet/art")
    e = w2x.Img2Img()
    msgs = []
    e.setMessageCallback(lambda s, m: msgs.append(m))
    assert not e.build(path, w2x.BuildConfig.fixed(1, 64, precision=w2x.PRECISION_TF32))
    assert "tf32 is not available for swin_unet models" in msgs[-1]
    assert e.build(path, w2x.BuildConfig.fixed(1, 64))
    assert not e.load(path, w2x.RenderConfig(precision=w2x.PRECISION_TF32, batchSize=1, height=64, width=64, scaling=2))
    assert "tf32 is not available for swin_unet models" in msgs[-1]
    e.close()


def test_tf32_holds_activations_beyond_fp16_range(built_lib, tmp_path):
    """unet1.conv1.conv.0 (weight and bias) x 2^17 and unet1.conv1.conv.2 (weight) x 2^-17: the same function (LeakyReLU is positively
    homogeneous, powers of two are exact), but the tensor between the two layers now reaches ~1e5."""
    import w2x
    original = make_model("cunet", 2, 1234)
    scaled = make_model("cunet", 2, 1234)
    sd = scaled.state_dict()
    with torch.no_grad():
        sd["unet1.conv1.conv.0.weight"].mul_(2.0 ** 17)
        sd["unet1.conv1.conv.0.bias"].mul_(2.0 ** 17)
        sd["unet1.conv1.conv.2.weight"].mul_(2.0 ** -17)
    path = w2x.model_path(str(tmp_path), "cunet/art", 0, 2)
    os.makedirs(os.path.dirname(path), exist_ok=True)
    onnx_io.export_cunet(scaled, path)
    src = tiling.synthetic_frame(150, 97, 5)
    ref = tiling.render(src, _model_fn(original), 64, 56, 2, 1 / 16, 4)
    e, msgs = _engine(path, 2, 64, 4)
    dst = e.render(src)
    assert dst is not None, msgs
    ok, info = _meets_render_bar(dst, ref)
    assert ok, info
    e.close()
    # the fp16 engine on the same file overflows between the two layers: the test reaches the range tf32 exists for
    e16, msgs = _engine(path, 2, 64, 4, precision=w2x.PRECISION_FP16)
    d16 = e16.render(src)
    assert d16 is not None, msgs
    assert not _meets_render_bar(d16, ref)[0]
    e16.close()


def test_cli_tf32_build_then_render(built_lib, tmp_path):
    import subprocess
    import w2x
    from __graft_entry__ import make_synthetic_model
    from test_cli_videoio import CLI, _fake_tools, _fake_video

    d = str(tmp_path)
    tools = _fake_tools(d)
    _, onnx_path = make_synthetic_model(os.path.join(d, "models"), 2, 0)
    base = [CLI, "--model", "cunet/art", "--scale", "2", "--noise", "0", "--batchSize", "2", "--tileSize", "64", "--precision", "tf32"]
    r = subprocess.run(base + ["build"], capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    frames = np.random.default_rng(1).integers(0, 256, (3, 76, 100, 3), dtype=np.uint8)
    os.makedirs(os.path.join(d, "in"))
    os.makedirs(os.path.join(d, "out"))
    _fake_video(os.path.join(d, "in", "clip.mkv"), frames, rate="24/1")
    r = subprocess.run(base + ["render", "-i", os.path.join(d, "in", "clip.mkv"), "-o", os.path.join(d, "out"), "--ffmpegDir", tools],
                       capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    eng = w2x.Img2Img()
    assert eng.load(onnx_path, w2x.RenderConfig(precision=w2x.PRECISION_TF32, batchSize=2, height=64, width=64, scaling=2))
    want = np.stack([eng.render(f) for f in frames])
    eng.close()
    got = np.fromfile(os.path.join(d, "out", "clip(cunet_art)(noise0)(scale2).mp4"), np.uint8).reshape(want.shape)
    assert np.array_equal(got, want)
