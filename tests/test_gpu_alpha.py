"""-m gpu: images with an alpha channel (w2x_render_bgra, Img2Img.render_bgra, the CLI's --alpha).

The colour bleed is integer arithmetic and must equal tests/alpha_oracle.py bit for bit.  A tile's model output does not depend on its
batch or slot, so the colour of a BGRA render equals w2x_render of the bled frame byte for byte and its alpha follows from a render of
the grey frame; against the fp32 PyTorch oracle the alpha meets the suite's render bar."""
import os
import subprocess

import numpy as np
import pytest
import torch

import alpha_oracle
from alpha_oracle import BLEED_ROUNDS, alpha_bleed, masked_frame
from oracle import tiling

pytestmark = pytest.mark.gpu


# ---- the bleed kernel ------------------------------------------------------------------------------------------------------------
def _pattern(kind, w, h, seed=0):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    if kind == "blobs":
        a[..., 3] = masked_frame(w, h, seed)[..., 3] if w > 1 and h > 1 else 0
    elif kind == "one":
        a[..., 3] = 0
        a[h // 3, w // 2, 3] = 200
    elif kind == "zero":
        a[..., 3] = 0
    else:
        a[..., 3] = 255
    return a


@pytest.mark.parametrize("rounds", [8, 18, 28])
@pytest.mark.parametrize("kind", ["blobs", "one", "zero", "full"])
@pytest.mark.parametrize("w,h", [(1, 1), (257, 65)])
def test_bleed_kernel_matches_oracle(w, h, kind, rounds, built_lib):
    import w2x
    a = _pattern(kind, w, h)
    assert np.array_equal(w2x.alpha_bleed(a, rounds), alpha_bleed(a, rounds))


@pytest.mark.parametrize("rounds", [8, 28])
def test_bleed_kernel_matches_oracle_1080p(rounds, built_lib):
    import w2x
    a = _pattern("blobs", 1920, 1080, 3)
    assert np.array_equal(w2x.alpha_bleed(a, rounds), alpha_bleed(a, rounds))


def test_bleed_kernel_strided_source(built_lib):
    import w2x
    wide = _pattern("blobs", 300, 70, 4)
    a = wide[:, 17:17 + 257]
    assert a.strides[0] > 4 * 257
    assert np.array_equal(w2x.alpha_bleed(a, 18), alpha_bleed(a, 18))


# ---- engines -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def alpha_models(tmp_path_factory):
    """(family, scale) -> (PyTorch model, ONNX path), in a directory of this module's own: the engines built here (tf32 among them) leave
    their artefacts next to these files, not next to the session's shared models."""
    import __graft_entry__
    d = str(tmp_path_factory.mktemp("alpha_models"))
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


def _psnr(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


# name: (family, scale, tile, batch, tta, tf32)
ENGINES = {
    "cunet2x_t64_b3": ("cunet", 2, 64, 3, False, False),
    "cunet1x_t128": ("cunet", 1, 128, 2, False, False),
    "swin4x_t64": ("swin_unet", 4, 64, 2, False, False),
    "cunet2x_t64_b3_tf32": ("cunet", 2, 64, 3, False, True),
    "cunet1x_t128_tta": ("cunet", 1, 128, 2, True, False),
}


def _make(name, alpha_models):
    fam, scale, tile, batch, tta, tf32 = ENGINES[name]
    model_t, path = alpha_models[(fam, scale)]
    return _engine(path, scale, tile, batch, tta, tf32), model_t, (fam, scale, tile, batch, tta)


def test_opaque_frame_is_render_plus_255(built_lib, alpha_models):
    e, _, _ = _make("cunet2x_t64_b3", alpha_models)
    src = np.empty((97, 150, 4), np.uint8)
    src[..., :3] = tiling.synthetic_frame(150, 97, 1)
    src[..., 3] = 255
    n0 = e.launch_count
    ref = e.render(src[..., :3])
    n1 = e.launch_count
    got = e.render_bgra(src)
    n2 = e.launch_count
    assert got is not None, e.last_error
    assert np.array_equal(got[..., :3], ref)
    assert (got[..., 3] == 255).all()
    # no alpha pass: at most the scan on top of render's launches (render may stitch band by band)
    assert n2 - n1 <= (n1 - n0) + 1, (n1 - n0, n2 - n1)
    e.close()


@pytest.mark.parametrize("name", list(ENGINES))
def test_transparent_frame(name, built_lib, alpha_models):
    e, model_t, (fam, scale, tile, batch, tta) = _make(name, alpha_models)
    rounds = BLEED_ROUNDS[(fam, scale)]
    src = masked_frame(150, 97, 2)
    assert (src[..., 3] == 0).mean() > 0.2 and ((src[..., 3] > 0) & (src[..., 3] < 255)).any()
    got = e.render_bgra(src)
    assert got is not None, e.last_error
    assert got.shape == (97 * scale, 150 * scale, 4)
    # colour: the render of the bled frame, byte for byte
    bled = alpha_bleed(src, rounds)
    assert np.array_equal(got[..., :3], e.render(np.ascontiguousarray(bled[..., :3])))
    # alpha: the grey frame's render, channel mean (from the packed bytes here, so within 1)
    grey = e.render(np.repeat(src[..., 3:], 3, axis=2))
    mean = np.rint(grey.astype(np.float64).mean(axis=2))
    assert np.abs(got[..., 3].astype(np.int32) - mean).max() <= 1
    # against the fp32 oracle: the suite's render bar
    ref = alpha_oracle.render_bgra(src, _model_fn(model_t), tile, e.output_tile_size, scale, 1 / 16, batch, tta=tta, rounds=rounds)
    diff = np.abs(got[..., 3].astype(np.int32) - ref[..., 3].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999 and _psnr(got[..., 3], ref[..., 3]) >= 50, ((diff <= 1).mean(), int(diff.max()), _psnr(got[..., 3], ref[..., 3]))
    assert np.array_equal(e.render_bgra(src), got)              # a re-render is byte-identical
    e.close()


def test_colour_under_alpha_zero_does_not_matter(built_lib, alpha_models):
    e, _, _ = _make("cunet2x_t64_b3", alpha_models)
    src = masked_frame(150, 97, 5)
    other = src.copy()
    hidden = src[..., 3] == 0
    other[..., :3][hidden] = np.random.default_rng(9).integers(0, 256, (int(hidden.sum()), 3), dtype=np.uint8)
    a, b = e.render_bgra(src), e.render_bgra(other)
    assert a is not None and b is not None
    assert np.array_equal(a, b)
    e.close()


def test_interleaved_calls_equal_fresh_engines(built_lib, alpha_models):
    """render, submit, render_bgra and render_banded (over this engine and a second one) in one sequence on frames that grow, shrink and
    grow again: every call returns what the same call returns on fresh engines."""
    import w2x
    from test_gpu_engine_state import _submit
    e, _, _ = _make("cunet2x_t64_b3", alpha_models)
    _, path = alpha_models[("cunet", 2)]
    e2 = _engine(path, 2, 64, 3)
    opaque = masked_frame(150, 97, 6)
    opaque[..., 3] = 255
    calls = [("bgr", tiling.synthetic_frame(150, 97, 7)), ("bgra", masked_frame(131, 70, 8)), ("bgra", opaque),
             ("bgr", tiling.synthetic_frame(131, 70, 9)), ("bgra", masked_frame(150, 97, 10)), ("bgra", opaque[:70, :131].copy()),
             ("bgr", tiling.synthetic_frame(150, 97, 11)), ("submit", tiling.synthetic_frame(210, 160, 12)),
             ("banded", tiling.synthetic_frame(96, 150, 13)), ("bgra", masked_frame(230, 170, 14)), ("submit", tiling.synthetic_frame(90, 60, 15)),
             ("banded", tiling.synthetic_frame(240, 180, 16)), ("bgr", tiling.synthetic_frame(100, 70, 17))]

    def call(k, engines, f):
        if k == "bgr":
            return engines[0].render(f)
        if k == "bgra":
            return engines[0].render_bgra(f)
        if k == "submit":
            return _submit(engines[0], f)
        return w2x.render_banded(engines, f)

    got = [call(k, [e, e2], f) for k, f in calls]
    for (k, f), g in zip(calls, got):
        fresh = [_engine(path, 2, 64, 3) for _ in range(2 if k == "banded" else 1)]
        want = call(k, fresh, f)
        for x in fresh:
            x.close()
        assert g is not None and np.array_equal(g, want), (k, f.shape)
    e.close()
    e2.close()


def test_strided_host_buffers(built_lib, alpha_models):
    e, _, _ = _make("cunet2x_t64_b3", alpha_models)
    src = masked_frame(150, 97, 12)
    want = e.render_bgra(src)
    wide_src = np.zeros((97, 171, 4), np.uint8)
    wide_src[:, 5:155] = src
    wide_dst = np.full((194, 333, 4), 7, np.uint8)
    view = wide_dst[:, 9:309]
    out = e.render_bgra(wide_src[:, 5:155], view)
    assert out is not None, e.last_error
    assert np.array_equal(view, want)
    assert (wide_dst[:, :9] == 7).all() and (wide_dst[:, 309:] == 7).all()
    e.close()


def test_errors_return_zero_with_a_message(built_lib, alpha_models):
    import ctypes as C
    import w2x
    l = w2x.lib()
    fresh = w2x.Img2Img()
    assert fresh.render_bgra(np.zeros((8, 8, 4), np.uint8)) is None
    assert "no engine loaded" in fresh.last_error
    fresh.close()
    assert l.w2x_render_bgra(None, None, 8, 8, 32, None, 64) == 0
    e, _, _ = _make("cunet2x_t64_b3", alpha_models)
    src = np.zeros((8, 8, 4), np.uint8)
    dst = np.zeros((16, 16, 4), np.uint8)
    p = lambda a: C.c_void_p(a.ctypes.data)
    assert l.w2x_render_bgra(e._h, None, 8, 8, 32, p(dst), 64) == 0 and "null image pointer" in e.last_error
    assert l.w2x_render_bgra(e._h, p(src), 8, 8, 32, None, 64) == 0 and "null image pointer" in e.last_error
    assert l.w2x_render_bgra(e._h, p(src), 8, 8, 24, p(dst), 64) == 0 and "stride" in e.last_error
    assert l.w2x_render_bgra(e._h, p(src), 8, 8, 32, p(dst), 48) == 0 and "stride" in e.last_error
    assert l.w2x_render_bgra(e._h, p(src), 0, 8, 32, p(dst), 64) == 0
    assert l.w2x_alpha_bleed(0, None, 8, 8, 32, 8, p(dst)) == 0
    assert l.w2x_alpha_bleed(0, p(src), 8, 8, 16, 8, p(dst)) == 0
    assert e.render_bgra(src) is not None                      # the engine still works
    e.close()


def test_cli_alpha_still_and_video(built_lib, tmp_path):
    import w2x
    from __graft_entry__ import make_synthetic_model
    from test_alpha import BASE, CLI, _tools

    d = str(tmp_path)
    tools = _tools(d)
    _, onnx_path = make_synthetic_model(os.path.join(d, "models"), 2, 0)
    r = subprocess.run([CLI, *BASE, "build"], capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    os.makedirs(os.path.join(d, "in"))
    os.makedirs(os.path.join(d, "out"))
    os.makedirs(os.path.join(d, "out_plain"))
    still = masked_frame(100, 76, 13)
    still.tofile(os.path.join(d, "in", "still.png"))
    with open(os.path.join(d, "in", "still.png.meta"), "w") as f:
        f.write("width=100\nheight=76\nr_frame_rate=25/1\nnb_frames=N/A\n")
    frames = np.random.default_rng(1).integers(0, 256, (3, 76, 100, 3), dtype=np.uint8)
    frames.tofile(os.path.join(d, "in", "clip.mkv"))
    with open(os.path.join(d, "in", "clip.mkv.meta"), "w") as f:
        f.write("width=100\nheight=76\nr_frame_rate=24/1\nnb_frames=3\n")
    r = subprocess.run([CLI, *BASE, "render", "-i", os.path.join(d, "in"), "-o", os.path.join(d, "out"), "--ffmpegDir", tools, "--alpha"],
                       capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "--alpha applies to still images; " + os.path.join(d, "in", "clip.mkv") + " is rendered without alpha" in r.stdout
    eng = w2x.Img2Img()
    assert eng.load(onnx_path, w2x.RenderConfig(batchSize=2, height=64, width=64, scaling=2))
    want = eng.render_bgra(still)
    eng.close()
    png = os.path.join(d, "out", "still(cunet_art)(noise0)(scale2).png")
    assert np.array_equal(np.fromfile(png, np.uint8).reshape(want.shape), want)
    assert "-pix_fmt bgra" in open(png + ".cmd").read()
    r = subprocess.run([CLI, *BASE, "render", "-i", os.path.join(d, "in", "clip.mkv"), "-o", os.path.join(d, "out_plain"), "--ffmpegDir", tools],
                       capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    name = "clip(cunet_art)(noise0)(scale2).mp4"
    assert open(os.path.join(d, "out", name), "rb").read() == open(os.path.join(d, "out_plain", name), "rb").read()
    # --device list: the still goes through the pool's first engine
    os.makedirs(os.path.join(d, "out_pool"))
    r = subprocess.run([CLI, *BASE, "--device", "0,0", "render", "-i", os.path.join(d, "in", "still.png"), "-o", os.path.join(d, "out_pool"),
                        "--ffmpegDir", tools, "--alpha"], capture_output=True, text=True, cwd=d)
    assert r.returncode == 0, r.stdout + r.stderr
    assert np.array_equal(np.fromfile(os.path.join(d, "out_pool", "still(cunet_art)(noise0)(scale2).png"), np.uint8).reshape(want.shape), want)
