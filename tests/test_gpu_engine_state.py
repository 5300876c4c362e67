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
