"""The C-ABI libraries load without a GPU and export every symbol include/*.h declares: include/w2x.h (the drop-in boundary) and
the test hooks of include/w2x_dev.h from the shipped lib/libw2x.so; the w2x_probe_* micro-benchmarks of include/w2x_dev.h from the
development build lib/libw2x_dev.so only."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols(header="w2x.h"):
    hdr = open(os.path.join(ROOT, "include", header)).read()
    return sorted(set(re.findall(r"W2X_API[^;]*?\b(w2x_[a-z0-9_]+)\s*\(", hdr, re.S)))


def test_header_and_binding_agree(built_lib):
    import w2x
    decl = declared_symbols()
    assert len(decl) >= 30
    dev = declared_symbols("w2x_dev.h")
    hooks = [n for n in dev if not n.startswith("w2x_probe_")]
    assert sorted(decl + hooks) == w2x.EXPORTED_SYMBOLS
    assert sorted(n for n in dev if n.startswith("w2x_probe_")) == sorted(w2x._DEV_SIGNATURES)


def test_library_exports_every_declared_symbol(built_lib):
    import w2x
    raw = C.CDLL(w2x.LIB_PATH)
    for name in declared_symbols() + [n for n in declared_symbols("w2x_dev.h") if not n.startswith("w2x_probe_")]:
        assert hasattr(raw, name), name
    # the shipped library carries no micro-benchmarks; the development build carries everything
    for name in w2x._DEV_SIGNATURES:
        assert not hasattr(raw, name), name
    dev = C.CDLL(w2x.DEV_LIB_PATH)
    for name in declared_symbols() + declared_symbols("w2x_dev.h"):
        assert hasattr(dev, name), name


def test_shipped_library_ignores_work_skipping_switches(built_lib):
    """W2X_DBG / W2X_CONV_IMPL / W2X_NO_* alter or skip kernel work: they are compiled out of lib/libw2x.so (csrc/hostutil.h devEnv)."""
    blob = open(__import__("w2x").LIB_PATH, "rb").read()
    for name in (b"W2X_DBG", b"W2X_CONV_IMPL", b"W2X_NO_PATCH", b"W2X_NO_FUSE_FIRST", b"W2X_NO_EPI_GROUPS", b"W2X_NO_HEAD_KERNEL", b"W2X_NO_PDL"):
        assert name + b"\0" not in blob, name


def test_defaults_match_reference_config(built_lib):
    """src/tensorrt/config.h:12-43 defaults."""
    import w2x
    b = w2x._BuildConfig()
    built_lib.w2x_default_build_config(C.byref(b))
    assert [getattr(b, f[0]) for f in b._fields_] == [0, 1, 1, 1, 4, 3, 3, 3, 64, 256, 640, 64, 256, 640]
    r = w2x._RenderConfig()
    built_lib.w2x_default_render_config(C.byref(r))
    assert (r.deviceId, r.precision, r.batchSize, r.channels, r.height, r.width, r.scaling, r.overlapX, r.overlapY, r.tta) == \
        (0, 1, 1, 3, 256, 256, 4, 0.0625, 0.0625, 0)
    d = w2x.BuildConfig()
    assert [getattr(d, f[0]) for f in b._fields_] == [getattr(b, f[0]) for f in b._fields_]


def test_errors_do_not_cross_the_boundary(built_lib):
    """Like the reference's function-try-blocks: failure == false + a message, never an exception/abort."""
    import w2x
    e = w2x.Img2Img()
    msgs = []
    e.setMessageCallback(lambda sev, m: msgs.append((sev, m)))
    assert e.load("/nonexistent/model.onnx", w2x.RenderConfig()) is False
    assert msgs and msgs[-1][0] == 1 and "Failed to find engine file" in msgs[-1][1] and "model file does not exist" in msgs[-1][1]
    assert msgs[-1][1].startswith("[load@")  # "[func@line] msg", logger.cpp:19-22
    assert e.render(__import__("numpy").zeros((8, 8, 3), "uint8")) is None
    assert "no engine loaded" in e.last_error
    e.close()


def test_frame_entry_points_refuse_without_an_engine(built_lib):
    """Every frame entry point of the C ABI fails (0 for the render calls, -1 for the submit calls) on a NULL handle, and on an engine
    that has loaded nothing, with the reason "no engine loaded".  The pool's engines refuse the frame through w2x_pool_wait."""
    import numpy as np
    import w2x
    l = built_lib
    src, dst = np.zeros((8, 8, 4), np.uint8), np.zeros((16, 16, 4), np.uint8)
    src16, dst16 = np.zeros((8, 8, 3), np.uint16), np.zeros((16, 16, 3), np.uint16)
    p = lambda a: C.c_void_p(a.ctypes.data)
    bgr, bgra, u16 = (p(src), 8, 8, 24, p(dst), 48), (p(src), 8, 8, 32, p(dst), 64), (p(src16), 8, 8, 48, p(dst16), 96)
    resized = (p(src), 8, 8, 24, p(dst), 12, 12, 36)
    engine_calls = [("w2x_render", bgr, 0), ("w2x_render_bgra", bgra, 0), ("w2x_render_resized", resized, 0), ("w2x_render_u16", u16, 0),
                    ("w2x_render_device", bgr, 0), ("w2x_submit", bgr, -1), ("w2x_submit_resized", resized, -1), ("w2x_submit_u16", u16, -1)]
    pool_calls = [("w2x_pool_submit", bgr), ("w2x_pool_submit_resized", resized), ("w2x_pool_submit_u16", u16)]

    e = w2x.Img2Img()
    msgs = []
    e.setMessageCallback(lambda sev, m: msgs.append(m))
    for name, args, bad in engine_calls:
        assert getattr(l, name)(None, *args) == bad, name
        msgs.clear()
        assert getattr(l, name)(e._h, *args) == bad, name
        assert len(msgs) == 1 and "no engine loaded" in msgs[0] and "no engine loaded" in e.last_error, (name, msgs)
    assert l.w2x_render_banded(None, 1, *bgr) == 0
    msgs.clear()
    assert l.w2x_render_banded((C.c_void_p * 1)(e._h), 1, *bgr) == 0
    assert len(msgs) == 1 and "no engine loaded" in msgs[0], msgs
    e.close()

    pool = w2x.Img2ImgPool([0])
    msgs = []
    pool.setMessageCallback(lambda sev, m: msgs.append(m))
    for name, args in pool_calls:
        assert getattr(l, name)(None, *args) == -1, name
        msgs.clear()
        ticket = getattr(l, name)(pool._h, *args)
        assert ticket >= 0, name
        assert l.w2x_pool_wait(pool._h, ticket) == 0, name
        assert len(msgs) == 1 and "no engine loaded" in msgs[0], (name, msgs)
    pool.close()
