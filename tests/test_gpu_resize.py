"""-m gpu: output at any size up to the model's scale (w2x_render_resized, w2x_submit_resized, w2x_pool_submit_resized, the resample kernels
alone through w2x_resample, and the CLI's --outputScale).

The contract is defined on top of render: out = clamp(rint(R_y(R_x(render(src))))) with R torch's float64 antialiased bicubic interpolate
(tests/test_resize.py: torch_resample, held to the float64 formula there).
The device works in fp32, so the bar is max |diff| <= 1 with at least 99.9 % of the values exact.  The paths of one engine (render_resized,
submit_resized, the pool, a re-render) run the same kernels on the same canvas and must agree byte for byte."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from alpha_oracle import masked_frame
from oracle import tiling
from test_gpu_alpha import ENGINES, _engine
from test_resize import torch_resample as oracle

pytestmark = pytest.mark.gpu


def _assert_bars(got, want, what=""):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    d = np.abs(got.astype(np.int32) - want.astype(np.int32))
    assert d.max() <= 1 and (d == 0).mean() >= 0.999, (what, int(d.max()), float((d == 0).mean()))


# ---- the kernels -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,dw,dh", [(1, 1, 1, 1), (1, 300, 1, 113), (300, 1, 113, 1), (97, 65, 13, 9), (7, 7, 1, 1), (7, 5, 1, 5),
                                       (3840, 2160, 2880, 1620), (640, 360, 640, 240), (640, 360, 427, 360), (256, 256, 64, 64)])
def test_resample_kernel_matches_torch(w, h, dw, dh, built_lib):
    import w2x
    src = np.random.default_rng(w * 7 + h).integers(0, 256, (h, w, 3), dtype=np.uint8)
    _assert_bars(w2x.resample(src, (dw, dh)), oracle(src, (dw, dh)), (w, h, dw, dh))


def test_resample_kernel_identity_is_exact(built_lib):
    import w2x
    src = np.random.default_rng(3).integers(0, 256, (65, 97, 3), dtype=np.uint8)
    assert np.array_equal(w2x.resample(src, (97, 65)), src)


def test_resample_kernel_one_axis_is_the_1d_resample(built_lib):
    """An axis left at its size has the single weight 1: resizing x then y equals resizing both at once, exactly."""
    import w2x
    src = np.random.default_rng(4).integers(0, 256, (120, 200, 3), dtype=np.uint8)
    only_x = w2x.resample(src, (150, 120))
    _assert_bars(only_x, oracle(src, (150, 120)))
    assert np.array_equal(w2x.resample(src, (150, 120)), only_x)
    assert np.array_equal(w2x.resample(src, (200, 120)), src)


def test_resample_kernel_strided_buffers(built_lib):
    import w2x
    wide = np.random.default_rng(5).integers(0, 256, (90, 300, 3), dtype=np.uint8)
    src = wide[:, 17:17 + 257]
    assert src.strides[0] > 3 * 257
    want = w2x.resample(np.ascontiguousarray(src), (101, 37))
    _assert_bars(want, oracle(src, (101, 37)))
    out = np.full((37, 140, 3), 7, np.uint8)
    view = out[:, 11:112]
    w2x.resample(src, (101, 37), view)
    assert np.array_equal(view, want)
    assert (out[:, :11] == 7).all() and (out[:, 112:] == 7).all()


# ---- engines -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def resize_models(tmp_path_factory):
    """(family, scale) -> (PyTorch model, ONNX path), in a directory of this module's own (the engines built here, tf32 among them, leave
    their artefacts next to these files)."""
    import __graft_entry__
    d = str(tmp_path_factory.mktemp("resize_models"))
    return {(fam, scale): __graft_entry__.make_synthetic_model(d, scale, 0, model=fam + "/art")
            for fam, scale in (("cunet", 1), ("cunet", 2), ("swin_unet", 4))}


def _make(name, models):
    fam, scale, tile, batch, tta, tf32 = ENGINES[name]
    _, path = models[(fam, scale)]
    return _engine(path, scale, tile, batch, tta, tf32), path


def _pinned_submit(submit, wait, f, size):
    import w2x
    h, w = f.shape[:2]
    pin_in, pin_out = w2x.PinnedArray((h, w, 3)), w2x.PinnedArray((size[1], size[0], 3))
    try:
        pin_in.array[...] = f
        t = submit(pin_in.ptr, w, h, pin_out.ptr, size)
        return pin_out.array.copy() if t >= 0 and wait(t) else None
    finally:
        pin_in.free()
        pin_out.free()


def _sizes(cw, ch):
    """Reductions whose output bands end inside canvas bands, a one-row-short frame, one axis left alone, and a strong reduction."""
    return [(cw * 3 // 4, ch * 3 // 4), (cw // 2 + 1, ch // 3), (cw - 1, ch), (cw, ch * 2 // 3), (max(cw // 7, 1), max(ch // 5, 1))]


@pytest.mark.parametrize("name", list(ENGINES))
def test_render_resized_against_oracle(name, built_lib, resize_models):
    e, _ = _make(name, resize_models)
    f = tiling.synthetic_frame(150, 97, 21)
    canvas = e.render(f)
    assert canvas is not None, e.last_error
    for size in _sizes(canvas.shape[1], canvas.shape[0]):
        got = e.render_resized(f, size)
        assert got is not None, e.last_error
        _assert_bars(got, oracle(canvas, size), (name, size))
    e.close()


@pytest.mark.parametrize("name", list(ENGINES))
def test_resized_paths_agree(name, built_lib, resize_models):
    import w2x
    fam, scale, tile, batch, tta, tf32 = ENGINES[name]
    e, path = _make(name, resize_models)
    f = tiling.synthetic_frame(150, 97, 22)
    size = (150 * scale * 2 // 3, 97 * scale * 3 // 5)
    got = e.render_resized(f, size)
    assert got is not None, e.last_error
    assert np.array_equal(_pinned_submit(e.submit_resized, e.wait, f, size), got)
    pool = w2x.Img2ImgPool([0, 0])
    msgs = []
    pool.setMessageCallback(lambda s, m: msgs.append((s, m)))
    prec = w2x.PRECISION_TF32 if tf32 else w2x.PRECISION_FP16
    assert pool.load(path, w2x.RenderConfig(precision=prec, batchSize=batch, height=tile, width=tile, scaling=scale, overlap=(1 / 16, 1 / 16),
                                            tta=tta)), msgs
    for _ in range(2):   # both engines of the pool
        assert np.array_equal(_pinned_submit(pool.submit_resized, pool.wait, f, size), got), msgs
    pool.close()
    assert np.array_equal(e.render_resized(f, size), got)      # a re-render is byte-identical
    e.close()


@pytest.mark.parametrize("name", list(ENGINES))
def test_identity_size_is_render(name, built_lib, resize_models):
    e, _ = _make(name, resize_models)
    f = tiling.synthetic_frame(150, 97, 23)
    n0 = e.launch_count
    want = e.render(f)
    n1 = e.launch_count
    got = e.render_resized(f, (want.shape[1], want.shape[0]))
    n2 = e.launch_count
    assert got is not None, e.last_error
    assert np.array_equal(got, want)
    assert n2 - n1 == n1 - n0
    assert np.array_equal(_pinned_submit(e.submit_resized, e.wait, f, (want.shape[1], want.shape[0])), want)
    e.close()


def test_strided_host_buffers(built_lib, resize_models):
    e, _ = _make("cunet2x_t64_b3", resize_models)
    f = tiling.synthetic_frame(150, 97, 24)
    want = e.render_resized(f, (201, 130))
    wide_src = np.zeros((97, 171, 3), np.uint8)
    wide_src[:, 5:155] = f
    wide_dst = np.full((130, 230, 3), 7, np.uint8)
    view = wide_dst[:, 9:210]
    assert e.render_resized(wide_src[:, 5:155], (201, 130), view) is not None, e.last_error
    assert np.array_equal(view, want)
    assert (wide_dst[:, :9] == 7).all() and (wide_dst[:, 210:] == 7).all()
    e.close()


def test_interleaved_calls_equal_fresh_engines(built_lib, resize_models):
    """render, render_bgra, submit, render_resized and submit_resized in one sequence on frames and sizes that grow, shrink and grow again,
    with a refused frame between two resized ones: every call returns what the same call returns on a fresh engine."""
    from test_gpu_engine_state import _submit
    e, path = _make("cunet2x_t64_b3", resize_models)
    calls = [("resized", tiling.synthetic_frame(150, 97, 30), (200, 150)), ("bgr", tiling.synthetic_frame(150, 97, 31), None),
             ("resized", tiling.synthetic_frame(150, 97, 32), (120, 80)), ("submit_resized", tiling.synthetic_frame(210, 160, 33), (400, 300)),
             ("bgra", masked_frame(131, 70, 34), None), ("resized", tiling.synthetic_frame(131, 70, 35), (262, 100)),
             ("too_small", tiling.synthetic_frame(4, 80, 36), (6, 100)), ("resized", tiling.synthetic_frame(131, 70, 37), (262, 100)),
             ("submit", tiling.synthetic_frame(90, 60, 38), None), ("submit_resized", tiling.synthetic_frame(90, 60, 39), (45, 30)),
             ("resized", tiling.synthetic_frame(240, 180, 40), (479, 359)), ("bgr", tiling.synthetic_frame(100, 70, 41), None),
             ("submit_resized", tiling.synthetic_frame(240, 180, 42), (300, 200))]

    def call(k, eng, f, size):
        if k == "bgr":
            return eng.render(f)
        if k == "bgra":
            return eng.render_bgra(f)
        if k == "submit":
            return _submit(eng, f)
        if k == "submit_resized":
            return _pinned_submit(eng.submit_resized, eng.wait, f, size)
        return eng.render_resized(f, size)

    got = [call(k, e, f, size) for k, f, size in calls]
    for (k, f, size), g in zip(calls, got):
        if k == "too_small":
            assert g is None
            continue
        fresh = _engine(path, 2, 64, 3)
        want = call(k, fresh, f, size)
        fresh.close()
        assert g is not None and np.array_equal(g, want), (k, f.shape, size)
    e.close()


def test_errors_return_zero_with_a_message(built_lib, resize_models):
    import w2x
    l = w2x.lib()
    fresh = w2x.Img2Img()
    assert fresh.render_resized(np.zeros((8, 8, 3), np.uint8), (4, 4)) is None
    assert "no engine loaded" in fresh.last_error
    fresh.close()
    assert l.w2x_render_resized(None, None, 8, 8, 24, None, 8, 8, 24) == 0
    assert l.w2x_submit_resized(None, None, 8, 8, 24, None, 8, 8, 24) == -1
    assert l.w2x_pool_submit_resized(None, None, 8, 8, 24, None, 8, 8, 24) == -1
    e, path = _make("cunet2x_t64_b3", resize_models)
    src = np.zeros((64, 64, 3), np.uint8)
    dst = np.zeros((128, 128, 3), np.uint8)
    p = lambda a: C.c_void_p(a.ctypes.data)
    for fn, bad in ((l.w2x_render_resized, 0), (l.w2x_submit_resized, -1)):
        assert fn(e._h, None, 64, 64, 192, p(dst), 100, 100, 300) == bad and "null image pointer" in e.last_error
        assert fn(e._h, p(src), 64, 64, 192, None, 100, 100, 300) == bad and "null image pointer" in e.last_error
        for dw, dh in ((0, 100), (100, 0), (129, 100), (100, 129), (-1, -1)):
            assert fn(e._h, p(src), 64, 64, 192, p(dst), dw, dh, 384) == bad and "outside" in e.last_error, (dw, dh)
        assert fn(e._h, p(src), 64, 64, 192, p(dst), 100, 100, 299) == bad and "stride" in e.last_error
        assert fn(e._h, p(src), 64, 64, 191, p(dst), 100, 100, 300) == bad and "stride" in e.last_error
        assert fn(e._h, p(src), 0, 64, 192, p(dst), 100, 100, 300) == bad
    assert l.w2x_resample(0, None, 8, 8, 24, p(dst), 4, 4, 12) == 0
    assert l.w2x_resample(0, p(src), 8, 8, 24, p(dst), 9, 4, 27) == 0          # no enlargement
    assert l.w2x_resample(0, p(src), 8, 8, 24, p(dst), 4, 4, 11) == 0
    assert l.w2x_resample_table(5, 6, None, None, None, 0) == 0
    f = tiling.synthetic_frame(64, 64, 50)
    assert e.render_resized(f, (100, 90)) is not None, e.last_error     # the engine still works
    # the pool: sizes below 1 are refused at submit, the others by the engine that takes the frame (its wait fails)
    pool = w2x.Img2ImgPool([0])
    msgs = []
    pool.setMessageCallback(lambda s, m: msgs.append((s, m)))
    assert pool.load(path, w2x.RenderConfig(batchSize=3, height=64, width=64, scaling=2, overlap=(1 / 16, 1 / 16))), msgs
    assert l.w2x_pool_submit_resized(pool._h, p(src), 64, 64, 192, p(dst), 0, 100, 384) == -1 and "below 1x1" in msgs[-1][1]
    assert _pinned_submit(pool.submit_resized, pool.wait, f, (129, 100)) is None and "outside" in msgs[-1][1]
    assert np.array_equal(_pinned_submit(pool.submit_resized, pool.wait, f, (100, 90)), e.render_resized(f, (100, 90)))
    pool.close()
    e.close()


# ---- the CLI -----------------------------------------------------------------------------------------------------------------------
def test_cli_output_scale_still_and_video(built_lib, tmp_path):
    import w2x
    from __graft_entry__ import make_synthetic_model
    from test_alpha import BASE, CLI, _tools

    d = str(tmp_path)
    tools = _tools(d)
    _, onnx_path = make_synthetic_model(os.path.join(d, "models"), 2, 0)
    r = subprocess.run([CLI, *BASE, "build"], capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    os.makedirs(os.path.join(d, "in"))
    still = tiling.synthetic_frame(100, 76, 13)
    still.tofile(os.path.join(d, "in", "still.png"))
    with open(os.path.join(d, "in", "still.png.meta"), "w") as f:
        f.write("width=100\nheight=76\nr_frame_rate=25/1\nnb_frames=N/A\n")
    frames = np.random.default_rng(1).integers(0, 256, (3, 76, 100, 3), dtype=np.uint8)
    frames.tofile(os.path.join(d, "in", "clip.mkv"))
    with open(os.path.join(d, "in", "clip.mkv.meta"), "w") as f:
        f.write("width=100\nheight=76\nr_frame_rate=24/1\nnb_frames=3\n")
    eng = w2x.Img2Img()
    assert eng.load(onnx_path, w2x.RenderConfig(batchSize=2, height=64, width=64, scaling=2))
    size = (150, 114)      # lround(100 * 1.5) x lround(76 * 1.5)
    want_still = eng.render_resized(still, size)
    want_clip = np.stack([eng.render_resized(x, size) for x in frames])
    plain_clip = np.stack([eng.render(x) for x in frames])
    eng.close()

    def render(out, *extra):
        os.makedirs(os.path.join(d, out))
        r = subprocess.run([CLI, *BASE, "render", "-i", os.path.join(d, "in"), "-o", os.path.join(d, out), "--ffmpegDir", tools, *extra],
                           capture_output=True, text=True, cwd=d)
        assert r.returncode == 0, r.stdout + r.stderr
        return os.path.join(d, out)

    for out, extra in (("out", ["--outputScale", "1.5"]), ("out_pool", ["--device", "0,0", "--outputScale", "1.5"])):
        o = render(out, *extra)
        png = os.path.join(o, "still(cunet_art)(noise0)(scale2)(150x114).png")
        mp4 = os.path.join(o, "clip(cunet_art)(noise0)(scale2)(150x114).mp4")
        assert np.array_equal(np.fromfile(png, np.uint8).reshape(want_still.shape), want_still), out
        assert np.array_equal(np.fromfile(mp4, np.uint8).reshape(want_clip.shape), want_clip), out
        for path in (png, mp4):
            assert " -s 150x114 " in open(path + ".cmd").read(), (out, path)
    # F == --scale: the frames of a render without the flag
    o = render("out_full", "--outputScale", "2")
    got = np.fromfile(os.path.join(o, "clip(cunet_art)(noise0)(scale2)(200x152).mp4"), np.uint8).reshape(plain_clip.shape)
    assert np.array_equal(got, plain_clip)
    o = render("out_plain")
    assert open(os.path.join(o, "clip(cunet_art)(noise0)(scale2).mp4"), "rb").read() == plain_clip.tobytes()
