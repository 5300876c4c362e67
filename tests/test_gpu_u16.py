"""-m gpu: 16 bits per channel (w2x_render_u16, w2x_submit_u16, w2x_pool_submit_u16, Img2Img.render_u16, the CLI's --bitDepth 16).

The kernels are bit-exact against NumPy.  On fp16 engines a u16 frame 257 F feeds the model exactly the tiles of the u8 frame F
(tests/test_u16.py), so render_u16(257 F) is within 129 of 257 render(F) everywhere; against the fp32 PyTorch oracle every engine meets the
suite's u8 bar in u16 units, and the 16-bit output is closer to the fp32 model than the 8-bit one."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import u16_oracle
from alpha_oracle import render_canvas
from oracle import tiling

pytestmark = pytest.mark.gpu


def _frame16(w, h, seed):
    return np.random.default_rng(seed).integers(0, 65536, size=(h, w, 3), dtype=np.uint16)


# ---- kernels -----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,tile,out_tile,scale,blend", [
    (256, 256, 64, 56, 2, 1 / 16),
    (97, 61, 64, 56, 2, 1 / 8),         # ragged: frame smaller than a tile in y
    (20, 20, 64, 56, 2, 1 / 16),        # single tile, all four borders replicated
    (333, 201, 128, 72, 1, 1 / 32),
])
def test_unpack_u16_is_bit_exact(w, h, tile, out_tile, scale, blend, built_lib):
    import w2x
    src = _frame16(w, h, 1)
    g = tiling.calculate_tiles(w, h, w * scale, h * scale, tile, tile, out_tile, out_tile, scale, blend, blend)
    augs = [i % 8 for i in range(g.count)]
    got = w2x.unpack_tiles_u16(src, g.in_rects, augs, tile)
    rgb = src[..., ::-1]
    for i, (r, k) in enumerate(zip(g.in_rects, augs)):
        ref = u16_oracle.normalize_u16(tiling.augment(tiling.pad_roi(rgb, r), k)).astype(np.float16)
        assert np.array_equal(got[i, :, :, :3].view(np.uint16), np.ascontiguousarray(ref).view(np.uint16)), (i, k)
        assert (got[i, :, :, 3] == 0).all()


def test_unpack_u16_all_augmentations_on_border_tiles_and_strided_rows(built_lib):
    import w2x
    wide = _frame16(300, 90, 2)
    src = wide[:, 7:7 + 211]                     # strided rows; on the device, rows of 1266 bytes: every other one starts mid-word
    assert src.strides[0] == 1800
    rects = [(-20, -13, 64, 64), (180, 40, 64, 64), (100, 30, 64, 64), (-5, 60, 64, 64)]
    for k in range(8):
        got = w2x.unpack_tiles_u16(src, rects, [k] * len(rects), 64)
        for i, r in enumerate(rects):
            ref = u16_oracle.normalize_u16(tiling.augment(tiling.pad_roi(src[..., ::-1], r), k)).astype(np.float16)
            assert np.array_equal(got[i, :, :, :3].view(np.uint16), np.ascontiguousarray(ref).view(np.uint16)), (i, k)


def _stitch_canvas(tiles_f16, g, cw, ch, out_tile):
    canvas = np.zeros((ch, cw, 3), np.float32)
    ov = g.out_overlap
    weights = tiling.create_tile_weights(ov[0], ov[1], out_tile, out_tile) if (ov[0] or ov[1]) else None
    for i, rect in enumerate(g.out_rects):
        o = tiles_f16[i, :, :, :3].astype(np.float32)
        if weights is not None:
            o = tiling.apply_weights(o, rect, cw, ch, weights)
        x, y, w, h = rect
        canvas[y:y + h, x:x + w] += o[:h, :w]
    return canvas


@pytest.mark.parametrize("w,h,tile,out_tile,scale,blend", [
    (256, 256, 64, 56, 2, 1 / 16),
    (97, 61, 64, 56, 2, 1 / 8),
    (333, 201, 128, 72, 1, 1 / 32),
    (150, 97, 64, 224, 4, 1 / 16),
])
def test_stitch_u16_is_bit_exact(w, h, tile, out_tile, scale, blend, built_lib):
    import w2x
    g = tiling.calculate_tiles(w, h, w * scale, h * scale, tile, tile, out_tile, out_tile, scale, blend, blend)
    tiles = np.random.default_rng(2).uniform(-0.1, 1.1, size=(g.count, out_tile, out_tile, 4)).astype(np.float16)
    got = w2x.stitch_tiles_u16(tiles, g.nx, g.ny, g.out_overlap[0], g.out_overlap[1], w * scale, h * scale)
    ref = u16_oracle.pack_u16(_stitch_canvas(tiles, g, w * scale, h * scale, out_tile))[..., ::-1]
    assert np.array_equal(got, ref)
    assert (got == 0).any() and (got == 65535).any()             # saturation on both sides


def test_stitch_u16_rounding_is_nearest_even(built_lib):
    import w2x
    # fp16 values whose product with 65535 is an exact .5 in fp32: 0.5 * 65535 = 32767.5 and 0.25 * 65535 = 16383.75 (no tie),
    # 2^-17 * 65535 = 0.49999..., plus values outside [0, 1]
    vals = np.array([0.5, 0.25, 2.0 ** -17, 2.0 ** -16 * 3, -3.0, 7.0, 1.0, 0.0], np.float16)
    tiles = np.zeros((1, 8, 8, 4), np.float16)
    tiles[0, 0, :, 0] = vals
    tiles[0, 1, :, 1] = vals[::-1]
    got = w2x.stitch_tiles_u16(tiles, 1, 1, 0, 0, 8, 8)
    ref = u16_oracle.pack_u16(tiles[0, :, :, :3].astype(np.float32))[..., ::-1]
    assert np.array_equal(got, ref)
    assert got[0, 0, 2] == 32768                                   # rint(32767.5) is even
    assert got[0, 4, 2] == 0 and got[0, 5, 2] == 65535


# ---- engines -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def u16_models(tmp_path_factory):
    """(family, scale) -> (PyTorch model, ONNX path) in a directory of this module's own (the tf32 build leaves its artefact there)."""
    import __graft_entry__
    d = str(tmp_path_factory.mktemp("u16_models"))
    return {(fam, scale): __graft_entry__.make_synthetic_model(d, scale, 0, model=fam + "/art")
            for fam, scale in (("cunet", 1), ("cunet", 2), ("swin_unet", 4))}


def _engine(path, scale, tile, batch, tta=False, tf32=False, blend=1 / 16):
    import w2x
    prec = w2x.PRECISION_TF32 if tf32 else w2x.PRECISION_FP16
    e = w2x.Img2Img()
    msgs = []
    e.setMessageCallback(lambda s, m: msgs.append((s, m)))
    assert e.build(path, w2x.BuildConfig.fixed(batch, tile, precision=prec)), msgs
    assert e.load(path, w2x.RenderConfig(precision=prec, batchSize=batch, height=tile, width=tile, scaling=scale, overlap=(blend, blend),
                                         tta=tta)), msgs
    return e


def _model_fn(model_t):
    def f(x):
        with torch.no_grad():
            return model_t(torch.from_numpy(np.ascontiguousarray(x))).numpy()
    return f


# name: (family, scale, tile, batch, tta, tf32)
FP16_ENGINES = {
    "cunet2x_t64_b3": ("cunet", 2, 64, 3, False, False),
    "cunet1x_t128": ("cunet", 1, 128, 2, False, False),
    "cunet2x_t64_b3_tta": ("cunet", 2, 64, 3, True, False),
    "swin4x_t64": ("swin_unet", 4, 64, 2, False, False),
}
ENGINES = dict(FP16_ENGINES, cunet2x_t64_b3_tf32=("cunet", 2, 64, 3, False, True))


def _make(name, models):
    fam, scale, tile, batch, tta, tf32 = ENGINES[name]
    model_t, path = models[(fam, scale)]
    return _engine(path, scale, tile, batch, tta, tf32), model_t, (scale, tile, batch, tta)


def _size(name):
    return (100, 70) if "tta" in name else (150, 97)


@pytest.mark.parametrize("name", list(FP16_ENGINES))
def test_widened_u8_frame_is_within_129_of_257_times_render(name, built_lib, u16_models):
    e, model_t, (scale, tile, batch, tta) = _make(name, u16_models)
    w, h = _size(name)
    f = tiling.synthetic_frame(w, h, 1)
    out8 = e.render(f)
    out16 = e.render_u16(f.astype(np.uint16) * np.uint16(257))
    assert out16 is not None, e.last_error
    assert out16.shape == (h * scale, w * scale, 3) and out16.dtype == np.uint16
    d = np.abs(out16.astype(np.int64) - 257 * out8.astype(np.int64))
    assert d.max() <= 129, int(d.max())
    # the reason for the feature: the 16-bit output is closer to the fp32 model than the 8-bit one
    ref = render_canvas(f, _model_fn(model_t), tile, e.output_tile_size, scale, 1 / 16, batch, tta=tta)[..., ::-1]
    rms16 = np.sqrt(np.mean((out16.astype(np.float64) / 65535 - ref) ** 2))
    rms8 = np.sqrt(np.mean((out8.astype(np.float64) / 255 - ref) ** 2))
    assert rms16 < rms8, (rms16, rms8)
    e.close()


@pytest.mark.parametrize("name", list(ENGINES))
def test_against_fp32_oracle(name, built_lib, u16_models):
    e, model_t, (scale, tile, batch, tta) = _make(name, u16_models)
    w, h = _size(name)
    src = _frame16(w, h, 3)
    got = e.render_u16(src)
    assert got is not None, e.last_error
    ref = u16_oracle.render_u16(src, _model_fn(model_t), tile, e.output_tile_size, scale, 1 / 16, batch, tta=tta)
    diff = np.abs(got.astype(np.int64) - ref.astype(np.int64))
    mse = np.mean(diff.astype(np.float64) ** 2)
    psnr = 99.0 if mse == 0 else 10 * np.log10(65535.0 ** 2 / mse)
    assert (diff <= 257).mean() >= 0.999 and psnr >= 50, ((diff <= 257).mean(), int(diff.max()), psnr)
    assert np.array_equal(e.render_u16(src), got)               # a re-render is identical
    e.close()


def _pinned16(shape):
    import w2x
    h, w = shape
    p = w2x.PinnedArray((h, w, 6))
    return p, p.array.view(np.uint16).reshape(h, w, 3)


def _submit16(eng, f, scaling):
    h, w = f.shape[:2]
    pin_in, a_in = _pinned16((h, w))
    pin_out, a_out = _pinned16((h * scaling, w * scaling))
    try:
        a_in[...] = f
        t = eng.submit_u16(pin_in.ptr, w, h, pin_out.ptr)
        return a_out.copy() if t >= 0 and eng.wait(t) else None
    finally:
        pin_in.free()
        pin_out.free()


def test_paths_agree(built_lib, u16_models):
    import w2x
    e, _, _ = _make("cunet2x_t64_b3", u16_models)
    _, path = u16_models[("cunet", 2)]
    frames = [_frame16(150, 97, 4), _frame16(131, 70, 5), _frame16(150, 97, 6)]
    want = [e.render_u16(f) for f in frames]
    for f, wnt in zip(frames, want):
        assert np.array_equal(_submit16(e, f, 2), wnt)
    pool = w2x.Img2ImgPool([0, 0])
    assert pool.load(path, w2x.RenderConfig(batchSize=3, height=64, width=64, scaling=2, overlap=(1 / 16, 1 / 16)))
    pins = [(_pinned16(f.shape[:2]), _pinned16((f.shape[0] * 2, f.shape[1] * 2))) for f in frames]
    tickets = []
    for f, ((pi, ai), (po, _)) in zip(frames, pins):
        ai[...] = f
        tickets.append(pool.submit_u16(pi.ptr, f.shape[1], f.shape[0], po.ptr))
    for t, ((pi, _), (po, ao)), wnt in zip(tickets, pins, want):
        assert t >= 0 and pool.wait(t)
        assert np.array_equal(ao, wnt)
        pi.free()
        po.free()
    pool.close()
    e.close()


def test_interleaved_calls_equal_fresh_engines(built_lib, u16_models):
    """render, render_u16, render_bgra, render_resized and submit_u16 in one sequence on frames that grow, shrink and grow again: every
    call returns what the same call returns on a fresh engine."""
    from alpha_oracle import masked_frame
    e, _, _ = _make("cunet2x_t64_b3", u16_models)
    _, path = u16_models[("cunet", 2)]
    calls = [("bgr", tiling.synthetic_frame(150, 97, 7)), ("u16", _frame16(150, 97, 8)), ("bgra", masked_frame(131, 70, 9)),
             ("u16", _frame16(131, 70, 10)), ("resized", tiling.synthetic_frame(131, 70, 11)), ("submit_u16", _frame16(210, 160, 12)),
             ("u16", _frame16(90, 60, 13)), ("bgr", tiling.synthetic_frame(90, 60, 14)), ("submit_u16", _frame16(230, 170, 15)),
             ("u16", _frame16(240, 180, 16)), ("resized", tiling.synthetic_frame(100, 70, 17)), ("u16", _frame16(100, 70, 18))]

    def call(k, eng, f):
        if k == "bgr":
            return eng.render(f)
        if k == "u16":
            return eng.render_u16(f)
        if k == "bgra":
            return eng.render_bgra(f)
        if k == "resized":
            return eng.render_resized(f, (f.shape[1] * 3 // 2, f.shape[0] * 3 // 2))
        return _submit16(eng, f, 2)

    got = [call(k, e, f) for k, f in calls]
    for (k, f), g in zip(calls, got):
        fresh = _engine(path, 2, 64, 3)
        want = call(k, fresh, f)
        fresh.close()
        assert g is not None and np.array_equal(g, want), (k, f.shape)
    e.close()


def test_strided_buffers(built_lib, u16_models):
    e, _, _ = _make("cunet2x_t64_b3", u16_models)
    for w, h in ((150, 97), (151, 61)):                            # an odd width too
        src = _frame16(w, h, 19)
        want = e.render_u16(src)
        wide_src = np.zeros((h, w + 21, 3), np.uint16)
        wide_src[:, 5:5 + w] = src
        # dst rows of 6 (2w + 37) bytes: not a multiple of 16, so the stitch takes its scalar store path
        wide_dst = np.full((2 * h, 2 * w + 37, 3), 7, np.uint16)
        assert wide_dst.strides[0] % 16 != 0
        view = wide_dst[:, 9:9 + 2 * w]
        out = e.render_u16(wide_src[:, 5:5 + w], view)
        assert out is not None, e.last_error
        assert np.array_equal(view, want)
        assert (wide_dst[:, :9] == 7).all() and (wide_dst[:, 9 + 2 * w:] == 7).all()
    e.close()


def test_launch_count_equals_render(built_lib, u16_models):
    e, _, _ = _make("cunet2x_t64_b3", u16_models)
    f = tiling.synthetic_frame(150, 97, 20)
    e.render(f)                                                    # warm: frame buffers built
    n0 = e.launch_count
    e.render(f)
    n1 = e.launch_count
    e.render_u16(f.astype(np.uint16) * np.uint16(257))
    n2 = e.launch_count
    assert n2 - n1 == n1 - n0, (n1 - n0, n2 - n1)
    e.close()


def test_errors_return_zero_with_a_message(built_lib, u16_models):
    import w2x
    l = w2x.lib()
    fresh = w2x.Img2Img()
    assert fresh.render_u16(np.zeros((8, 8, 3), np.uint16)) is None
    assert "no engine loaded" in fresh.last_error
    fresh.close()
    assert l.w2x_render_u16(None, None, 8, 8, 48, None, 96) == 0
    assert l.w2x_submit_u16(None, None, 8, 8, 48, None, 96) == -1
    e, _, _ = _make("cunet2x_t64_b3", u16_models)
    src = np.zeros((8, 8, 3), np.uint16)
    dst = np.zeros((16, 16, 3), np.uint16)
    raw = np.zeros(2 * dst.nbytes + 16, np.uint8)
    p = lambda a, off=0: C.c_void_p(a.ctypes.data + off)
    for fn, bad in ((l.w2x_render_u16, 0), (l.w2x_submit_u16, -1)):
        assert fn(e._h, None, 8, 8, 48, p(dst), 96) == bad and "null image pointer" in e.last_error
        assert fn(e._h, p(src), 8, 8, 48, None, 96) == bad and "null image pointer" in e.last_error
        assert fn(e._h, p(src), 8, 8, 46, p(dst), 96) == bad and "6 bytes per pixel" in e.last_error
        assert fn(e._h, p(src), 8, 8, 48, p(dst), 94) == bad and "6 bytes per pixel" in e.last_error
        assert fn(e._h, p(src), 8, 8, 49, p(raw), 96) == bad and "odd" in e.last_error
        assert fn(e._h, p(src), 8, 8, 48, p(raw), 97) == bad and "odd" in e.last_error
        assert fn(e._h, p(raw, 1), 8, 8, 48, p(dst), 96) == bad and "odd" in e.last_error
        assert fn(e._h, p(src), 8, 8, 48, p(raw, 1), 96) == bad and "odd" in e.last_error
        assert fn(e._h, p(src), 0, 8, 48, p(dst), 96) == bad
    assert e.render_u16(_frame16(40, 30, 21)) is not None       # the engine still works
    e.close()


def test_cli_bit_depth_16_still_and_video(built_lib, tmp_path):
    import w2x
    from __graft_entry__ import make_synthetic_model
    from test_alpha import BASE, CLI, _tools

    d = str(tmp_path)
    tools = _tools(d)
    _, onnx_path = make_synthetic_model(os.path.join(d, "models"), 2, 0)
    r = subprocess.run([CLI, *BASE, "build"], capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    for sub in ("in", "out16", "out8", "out_plain", "out_pool"):
        os.makedirs(os.path.join(d, sub))
    still = _frame16(100, 76, 22)
    still.astype("<u2").tofile(os.path.join(d, "in", "still.png"))
    with open(os.path.join(d, "in", "still.png.meta"), "w") as f:
        f.write("width=100\nheight=76\nr_frame_rate=25/1\nnb_frames=N/A\n")
    frames = np.random.default_rng(1).integers(0, 65536, (3, 76, 100, 3), dtype=np.uint16)
    frames.astype("<u2").tofile(os.path.join(d, "in", "clip.mkv"))
    with open(os.path.join(d, "in", "clip.mkv.meta"), "w") as f:
        f.write("width=100\nheight=76\nr_frame_rate=24/1\nnb_frames=3\n")

    r = subprocess.run([CLI, *BASE, "render", "-i", os.path.join(d, "in"), "-o", os.path.join(d, "out16"), "--ffmpegDir", tools,
                        "--bitDepth", "16"], capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    eng = w2x.Img2Img()
    assert eng.load(onnx_path, w2x.RenderConfig(batchSize=2, height=64, width=64, scaling=2))
    png = os.path.join(d, "out16", "still(cunet_art)(noise0)(scale2).png")
    want = eng.render_u16(still)
    assert np.array_equal(np.fromfile(png, "<u2").reshape(want.shape), want)
    assert "-pix_fmt bgr48le" in open(png + ".cmd").read() and "-pix_fmt rgb48be" in open(png + ".cmd").read()
    vid = os.path.join(d, "out16", "clip(cunet_art)(noise0)(scale2).mp4")
    got = np.fromfile(vid, "<u2").reshape(3, 152, 200, 3)
    for i in range(3):
        assert np.array_equal(got[i], eng.render_u16(frames[i])), i
    assert "-pix_fmt bgr48le" in open(vid + ".cmd").read() and "-pix_fmt yuv420p" in open(vid + ".cmd").read()
    eng.close()
    # --bitDepth 8 is the run without the flag, byte for byte (8-bit inputs for this one)
    f8 = np.random.default_rng(2).integers(0, 256, (3, 76, 100, 3), dtype=np.uint8)
    os.makedirs(os.path.join(d, "in8"))
    f8.tofile(os.path.join(d, "in8", "clip.mkv"))
    with open(os.path.join(d, "in8", "clip.mkv.meta"), "w") as f:
        f.write("width=100\nheight=76\nr_frame_rate=24/1\nnb_frames=3\n")
    f8[0].tofile(os.path.join(d, "in8", "still.png"))
    with open(os.path.join(d, "in8", "still.png.meta"), "w") as f:
        f.write("width=100\nheight=76\nr_frame_rate=25/1\nnb_frames=N/A\n")
    for out, extra in (("out8", ["--bitDepth", "8"]), ("out_plain", [])):
        r = subprocess.run([CLI, *BASE, "render", "-i", os.path.join(d, "in8"), "-o", os.path.join(d, out), "--ffmpegDir", tools, *extra],
                           capture_output=True, text=True, cwd=d)
        assert r.returncode == 0, r.stdout + r.stderr
    for name in ("clip(cunet_art)(noise0)(scale2).mp4", "still(cunet_art)(noise0)(scale2).png"):
        assert open(os.path.join(d, "out8", name), "rb").read() == open(os.path.join(d, "out_plain", name), "rb").read()
        assert open(os.path.join(d, "out8", name + ".cmd")).read().replace("out8", "OUT") == \
            open(os.path.join(d, "out_plain", name + ".cmd")).read().replace("out_plain", "OUT")
    # --device list: the still through the pool
    r = subprocess.run([CLI, *BASE, "--device", "0,0", "render", "-i", os.path.join(d, "in", "still.png"), "-o", os.path.join(d, "out_pool"),
                        "--ffmpegDir", tools, "--bitDepth", "16"], capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    assert np.array_equal(np.fromfile(os.path.join(d, "out_pool", "still(cunet_art)(noise0)(scale2).png"), "<u2").reshape(want.shape), want)
