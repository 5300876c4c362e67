"""-m gpu: an engine's cached frame state.  A frame the engine refuses must leave nothing behind that a later frame of the previous size
would reuse: after it, every entry point renders exactly what a fresh engine renders."""
import numpy as np
import pytest

from alpha_oracle import masked_frame
from oracle import tiling

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cunet2x(tmp_path_factory):
    """A cunet/art 2x ONNX file in a directory of this module's own (the engines built here leave their artefacts next to it)."""
    import __graft_entry__
    _, path = __graft_entry__.make_synthetic_model(str(tmp_path_factory.mktemp("engine_state_models")), 2, 0)
    return path


def _engine(path, tta=False):
    import w2x
    e = w2x.Img2Img()
    msgs = []
    e.setMessageCallback(lambda s, m: msgs.append((s, m)))
    assert e.build(path, w2x.BuildConfig.fixed(3, 64)), msgs
    assert e.load(path, w2x.RenderConfig(batchSize=3, height=64, width=64, scaling=2, overlap=(1 / 16, 1 / 16), tta=tta)), msgs
    return e


def _submit(e, f):
    """w2x_submit / w2x_wait on pinned copies of the frame; None when the engine refuses it."""
    import w2x
    h, w = f.shape[:2]
    pin_in, pin_out = w2x.PinnedArray((h, w, 3)), w2x.PinnedArray((h * e.scaling, w * e.scaling, 3))
    try:
        pin_in.array[...] = f
        t = e.submit(pin_in.ptr, w, h, pin_out.ptr)
        return pin_out.array.copy() if t >= 0 and e.wait(t) else None
    finally:
        pin_in.free()
        pin_out.free()


def _frame(kind, w, h, seed):
    if kind == "bgra_alpha":
        f = masked_frame(w, h, seed)
        assert (f[..., 3] < 255).any()
        return f
    if kind == "bgra_opaque":
        f = masked_frame(w, h, seed)
        f[..., 3] = 255
        return f
    return tiling.synthetic_frame(w, h, seed)


def _run(kind, e, f):
    if kind == "submit":
        return _submit(e, f)
    if kind.startswith("bgra"):
        return e.render_bgra(f)
    return e.render(f)


@pytest.mark.parametrize("kind", ["render", "submit", "bgra_opaque", "bgra_alpha", "tta"])
def test_rejected_frame_does_not_poison_the_engine(kind, built_lib, cunet2x):
    tta = kind == "tta"
    e = _engine(cunet2x, tta)
    assert _run(kind, e, _frame(kind, 120, 80, 1)) is not None, e.last_error
    # 4 columns are no wider than the input overlap of a 64-pixel tile at 1/16 (4 pixels): the tile grid is empty
    assert _run(kind, e, _frame(kind, 4, 80, 2)) is None
    assert "too small" in e.last_error, e.last_error
    f = _frame(kind, 120, 80, 3)
    got = _run(kind, e, f)
    assert got is not None, e.last_error
    fresh = _engine(cunet2x, tta)
    want = _run(kind, fresh, f)
    assert want is not None, fresh.last_error
    assert np.array_equal(got, want)
    fresh.close()
    e.close()


def test_bgr_frames_with_null_pointers_or_short_strides_are_refused_up_front(built_lib, cunet2x):
    """w2x_render, w2x_submit, w2x_render_device and w2x_render_banded refuse a null image pointer and a row stride below 3 bytes per
    pixel with a message, before any copy or launch; the engine then renders what it rendered before."""
    import ctypes as C
    import w2x
    l = w2x.lib()
    e = _engine(cunet2x)
    f = _frame("render", 40, 30, 4)
    want = e.render(f)
    assert want is not None, e.last_error
    msgs = []
    e.setMessageCallback(lambda s, m: msgs.append(m))
    src, dst = np.ascontiguousarray(f), np.zeros_like(want)
    d_src, d_dst = e.device_alloc(src.nbytes), e.device_alloc(dst.nbytes)
    p = lambda a: C.c_void_p(a.ctypes.data)
    banded = lambda h, *args: l.w2x_render_banded((C.c_void_p * 1)(h), 1, *args)
    calls = [(l.w2x_render, p(src), p(dst), 0), (l.w2x_submit, p(src), p(dst), -1),
             (l.w2x_render_device, C.c_void_p(d_src), C.c_void_p(d_dst), 0), (banded, p(src), p(dst), 0)]

    def refusal(fn, bad, *args):
        msgs.clear()
        assert fn(e._h, *args) == bad and len(msgs) == 1, msgs
        return msgs[0]

    n0 = e.launch_count
    for fn, s, d, bad in calls:
        assert "null image pointer" in refusal(fn, bad, None, 40, 30, 120, d, 240)
        assert "null image pointer" in refusal(fn, bad, s, 40, 30, 120, None, 240)
        assert "smaller than 3 bytes per pixel" in refusal(fn, bad, s, 40, 30, 119, d, 240)
        assert "smaller than 3 bytes per pixel" in refusal(fn, bad, s, 40, 30, 120, d, 239)
    assert e.launch_count == n0
    assert np.array_equal(e.render(f), want)
    e.device_free(d_src)
    e.device_free(d_dst)
    e.close()
