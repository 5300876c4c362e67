"""Weight packing for --precision tf32 (host-only; no GPU): fp32 GEMM operands rounded to nearest TF32 in the W2XPACK2 layout,
fp16 packs unchanged, SwinUNet refused."""
import hashlib
import os
import struct

import numpy as np
import pytest

from oracle import onnx_io
from oracle.models import make_model

# sha256 of the fp16 packs of the seeded synthetic models (make_synthetic_model / make_model seed 1234), recorded before the tf32
# path existed: a tf32 pack must not change a single byte of an fp16 one
FP16_PACK_SHA256 = {
    ("cunet", 1): "de11cf9a1b4c7a43d443db518c8e8a447dccb66f35bd227a564ba47300cd11c1",
    ("cunet", 2): "34737f15eb042710b881be73a01a5be3dde22dbd09dc7022ea16d8b6a59e9563",
    ("swin_unet", 2): "0e402069c69d02c5e351ab1d9fce114510969e510cc91f1dc7a32fb1a29fce0a",
}


def _onnx(tmp_path, family, scale):
    m = make_model(family, scale, 1234)
    p = str(tmp_path / f"{family}{scale}.onnx")
    (onnx_io.export_cunet if family == "cunet" else onnx_io.export_swin)(m, p)
    return m, p


@pytest.mark.parametrize("family,scale", sorted(FP16_PACK_SHA256))
def test_fp16_packs_are_byte_identical(family, scale, built_lib, tmp_path):
    import w2x
    _, p = _onnx(tmp_path, family, scale)
    q = str(tmp_path / "m.w2x")
    w2x.pack_onnx(p, q, w2x.PRECISION_FP16)
    assert hashlib.sha256(open(q, "rb").read()).hexdigest() == FP16_PACK_SHA256[(family, scale)]


def _tf32(a):
    """round to nearest even TF32: the low 13 bits of the fp32 pattern cleared"""
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).astype(np.uint64)
    u = ((u + 0xFFF + ((u >> 13) & 1)) & 0xFFFFE000).astype(np.uint32)
    return u.view(np.float32)


def _read_pack(path):
    """W2XPACK2: magic | arch scale offset precision dim nlayers | per layer: name, 11 u32 fields, 9 vectors (u32 count + data padded to 4)"""
    b = open(path, "rb").read()
    assert b[:8] == b"W2XPACK2"
    arch, scale, offset, precision, dim, nl = struct.unpack_from("<6I", b, 8)
    off = 32
    wtype = np.float32 if precision == 0 else np.uint16

    def vec(dtype):
        nonlocal off
        n = struct.unpack_from("<I", b, off)[0]
        off += 4
        size = n * np.dtype(dtype).itemsize
        v = np.frombuffer(b, dtype, n, off).copy()
        off += (size + 3) & ~3
        return v

    layers = []
    for _ in range(nl):
        name = vec(np.uint8).tobytes().decode()
        kind, cin, cout, npad, ktot, taps, se_r, heads, window, upscale, eps = struct.unpack_from("<11I", b, off)
        off += 44
        w = vec(wtype)
        bias = vec(np.float32)
        for _ in range(7):
            vec(np.float32)
        layers.append(dict(name=name, kind=kind, cin=cin, cout=cout, npad=npad, ktot=ktot, w=w.reshape(npad, ktot), bias=bias))
    assert off == len(b)
    return dict(arch=arch, scale=scale, offset=offset, precision=precision), layers


def _expected_operand(L, wt):
    """restatement of csrc/model_pack.h's B[npad][ktot] layouts from the torch weight"""
    kind, cin, npad, ktot = L["kind"], L["cin"], L["npad"], L["ktot"]
    B = np.zeros((npad, ktot), np.float32)
    if kind in (0, 1):            # conv3x3 / conv2x2 s2: k = (ky*kw+kx)*cin + ci
        co, ci, kh, kw = wt.shape
        w4 = np.zeros((co, cin, kh, kw), np.float32)
        w4[:, :ci] = wt
        B[:co] = w4.transpose(0, 2, 3, 1).reshape(co, kh * kw * cin)
    elif kind == 2:               # ConvTranspose 2x2 s2: row = (dy*2+dx)*cout + co, k = ci
        B[:] = wt.transpose(2, 3, 1, 0).reshape(4 * wt.shape[1], wt.shape[0])
    else:                         # ConvTranspose 4x4 s2 p3 head: row = (py*2+px)*4 + co, k = (wy*2+wx)*cin + ci
        for py in range(2):
            for px in range(2):
                for co in range(wt.shape[1]):
                    for wy in range(2):
                        for wx in range(2):
                            B[(py * 2 + px) * 4 + co, (wy * 2 + wx) * cin:(wy * 2 + wx + 1) * cin] = wt[:, co, 2 + py - 2 * wy, 2 + px - 2 * wx]
    return B


@pytest.mark.parametrize("scale", [1, 2])
def test_tf32_pack_holds_rounded_fp32_weights(scale, built_lib, tmp_path):
    import w2x
    m, p = _onnx(tmp_path, "cunet", scale)
    q = str(tmp_path / "m.w2x")
    w2x.pack_onnx(p, q, w2x.PRECISION_TF32)
    head, layers = _read_pack(q)
    assert head == dict(arch=scale, scale=scale, offset=36 if scale == 2 else 28, precision=w2x.PRECISION_TF32)
    assert len(layers) == 22
    sd = {k: v.numpy() for k, v in m.state_dict().items()}
    rounded = 0
    for L in layers:
        wt = sd[L["name"] + ".weight"]
        want = _tf32(_expected_operand(L, wt))
        assert np.array_equal(L["w"].view(np.uint32), want.view(np.uint32)), L["name"]
        assert (L["w"].view(np.uint32) & 0x1FFF == 0).all()
        rounded += int((_expected_operand(L, wt) != want).sum())
        if L["kind"] in (0, 1):
            assert np.array_equal(L["bias"][:L["cout"]], sd[L["name"] + ".bias"])
    assert rounded > 0   # the synthetic weights are not TF32 already: rounding really happened
    # the fp16 pack of the same graph has the same records with fp16 operands
    q16 = str(tmp_path / "m16.w2x")
    w2x.pack_onnx(p, q16, w2x.PRECISION_FP16)
    head16, layers16 = _read_pack(q16)
    assert head16["precision"] == w2x.PRECISION_FP16
    for a, b in zip(layers, layers16):
        assert (a["name"], a["kind"], a["npad"], a["ktot"]) == (b["name"], b["kind"], b["npad"], b["ktot"])
        assert np.array_equal(a["bias"], b["bias"])


def test_tf32_pack_refuses_swin_unet(built_lib, tmp_path):
    import w2x
    _, p = _onnx(tmp_path, "swin_unet", 2)
    with pytest.raises(RuntimeError, match="tf32 is not available for swin_unet models"):
        w2x.pack_onnx(p, str(tmp_path / "s.w2x"), w2x.PRECISION_TF32)
    assert not os.path.exists(str(tmp_path / "s.w2x"))
