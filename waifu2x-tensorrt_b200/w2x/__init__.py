"""ctypes binding of libw2x.so (include/w2x.h) + a Python mirror of the reference's operator surface.

`Img2Img` mirrors trt::Img2Img (/root/reference/src/tensorrt/img2img.h:14-50): build / load / render /
setMessageCallback / setProgressCallback with the reference's argument meaning and bool-return error
convention; `BuildConfig` / `RenderConfig` mirror src/tensorrt/config.h:12-43 field-for-field.

There is NO CPU fallback: if the CUDA library is missing, importing `lib()` raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Callable, List, Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libw2x.so")

PRECISION_TF32, PRECISION_FP16 = 0, 1
SEVERITY_NAMES = ["critical", "error", "warn", "info", "debug", "trace"]


class _BuildConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "deviceId", "precision", "minBatchSize", "optBatchSize", "maxBatchSize", "minChannels", "optChannels",
        "maxChannels", "minWidth", "optWidth", "maxWidth", "minHeight", "optHeight", "maxHeight")]


class _RenderConfig(C.Structure):
    _fields_ = [("deviceId", C.c_int), ("precision", C.c_int), ("batchSize", C.c_int), ("channels", C.c_int),
                ("height", C.c_int), ("width", C.c_int), ("scaling", C.c_int), ("overlapX", C.c_double),
                ("overlapY", C.c_double), ("tta", C.c_int)]


class _Rect(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("width", C.c_int), ("height", C.c_int)]


MESSAGE_CB = C.CFUNCTYPE(None, C.c_int, C.c_char_p, C.c_void_p)
PROGRESS_CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.c_double, C.c_void_p)


@dataclass
class BuildConfig:  # src/tensorrt/config.h:12-31
    deviceId: int = 0
    precision: int = PRECISION_FP16
    minBatchSize: int = 1
    optBatchSize: int = 1
    maxBatchSize: int = 4
    minChannels: int = 3
    optChannels: int = 3
    maxChannels: int = 3
    minWidth: int = 64
    optWidth: int = 256
    maxWidth: int = 640
    minHeight: int = 64
    optHeight: int = 256
    maxHeight: int = 640

    @staticmethod
    def fixed(batch: int, tile: int, device: int = 0, precision: int = PRECISION_FP16) -> "BuildConfig":
        """The config the reference CLI builds with (src/main.cpp:276-291): min = opt = max."""
        return BuildConfig(device, precision, batch, batch, batch, 3, 3, 3, tile, tile, tile, tile, tile, tile)

    def _c(self) -> _BuildConfig:
        return _BuildConfig(*[getattr(self, f[0]) for f in _BuildConfig._fields_])


@dataclass
class RenderConfig:  # src/tensorrt/config.h:33-43
    deviceId: int = 0
    precision: int = PRECISION_FP16
    batchSize: int = 1
    channels: int = 3
    height: int = 256
    width: int = 256
    scaling: int = 4
    overlap: Tuple[float, float] = (0.0625, 0.0625)
    tta: bool = False

    def _c(self) -> _RenderConfig:
        return _RenderConfig(self.deviceId, self.precision, self.batchSize, self.channels, self.height, self.width,
                             self.scaling, float(self.overlap[0]), float(self.overlap[1]), int(self.tta))


_lib = None

_SIGNATURES = {
    "w2x_default_build_config": (None, [C.POINTER(_BuildConfig)]),
    "w2x_default_render_config": (None, [C.POINTER(_RenderConfig)]),
    "w2x_create": (C.c_void_p, []),
    "w2x_destroy": (None, [C.c_void_p]),
    "w2x_set_message_callback": (None, [C.c_void_p, MESSAGE_CB, C.c_void_p]),
    "w2x_set_progress_callback": (None, [C.c_void_p, PROGRESS_CB, C.c_void_p]),
    "w2x_build": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(_BuildConfig)]),
    "w2x_load": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(_RenderConfig)]),
    "w2x_render": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_render_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_render_bgra": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_render_resized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_size_t]),
    "w2x_submit_resized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_size_t]),
    "w2x_render_u16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_submit_u16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_render_banded": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_wait": (C.c_int, [C.c_void_p, C.c_int]),
    "w2x_pool_create": (C.c_void_p, [C.POINTER(C.c_int), C.c_int]),
    "w2x_pool_destroy": (None, [C.c_void_p]),
    "w2x_pool_size": (C.c_int, [C.c_void_p]),
    "w2x_pool_engine": (C.c_void_p, [C.c_void_p, C.c_int]),
    "w2x_pool_set_message_callback": (None, [C.c_void_p, MESSAGE_CB, C.c_void_p]),
    "w2x_pool_build": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(_BuildConfig)]),
    "w2x_pool_load": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(_RenderConfig)]),
    "w2x_pool_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_pool_submit_resized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_size_t]),
    "w2x_pool_submit_u16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "w2x_pool_wait": (C.c_int, [C.c_void_p, C.c_int]),
    "w2x_pool_sync": (C.c_int, [C.c_void_p]),
    "w2x_sync": (C.c_int, [C.c_void_p]),
    "w2x_host_alloc": (C.c_void_p, [C.c_size_t]),
    "w2x_host_free": (None, [C.c_void_p]),
    "w2x_device_alloc": (C.c_void_p, [C.c_void_p, C.c_size_t]),
    "w2x_device_free": (None, [C.c_void_p, C.c_void_p]),
    "w2x_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "w2x_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "w2x_last_error": (C.c_char_p, [C.c_void_p]),
    "w2x_output_tile_size": (C.c_int, [C.c_void_p]),
    "w2x_launch_count": (C.c_longlong, [C.c_void_p]),
    "w2x_model_flops_per_tile": (C.c_double, [C.c_void_p]),
    "w2x_last_stage_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.c_int]),
    "w2x_timer_mark": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "w2x_timer_elapsed_ms": (C.c_float, [C.c_void_p, C.c_int, C.c_int]),
    "w2x_layer_kernel": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_int]),
    "w2x_profile_layers": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_double), C.c_int]),
    "w2x_calculate_tiles": (C.c_int, [C.c_int] * 9 + [C.c_double, C.c_double, C.POINTER(_Rect), C.POINTER(_Rect), C.c_int, C.POINTER(C.c_int)]),
    "w2x_blend_ramp": (C.c_int, [C.c_int, C.POINTER(C.c_float)]),
    "w2x_unpack_tiles": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.POINTER(_Rect), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_void_p]),
    "w2x_stitch_tiles": (C.c_int, [C.c_int, C.c_void_p] + [C.c_int] * 8 + [C.c_void_p, C.c_size_t]),
    "w2x_unpack_tiles_u16": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.POINTER(_Rect), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_void_p]),
    "w2x_stitch_tiles_u16": (C.c_int, [C.c_int, C.c_void_p] + [C.c_int] * 8 + [C.c_void_p, C.c_size_t]),
    "w2x_tta_reduce": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "w2x_alpha_bleed": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_void_p]),
    "w2x_resample": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_size_t]),
    "w2x_resample_table": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "w2x_infer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "w2x_layer_tensor": (C.c_longlong, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "w2x_selftest_conv": (C.c_double, [C.c_int] * 7 + [C.c_uint]),
    "w2x_run_conv_layer": (C.c_int, [C.c_int] * 8 + [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.c_void_p, C.c_void_p]),
    "w2x_run_conv_layer_f32": (C.c_int, [C.c_int] * 7 + [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.c_void_p, C.c_void_p]),
    "w2x_swin_attn_prepare": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "w2x_compose_up_to_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "w2x_run_swin_attn": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_float)]),
    "w2x_run_swin_mlp": (C.c_int, [C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int, C.POINTER(C.c_float)]),
    "w2x_select_engine": (C.c_int, [C.c_char_p, C.POINTER(_RenderConfig), C.c_char_p, C.c_char_p, C.c_size_t]),
    "w2x_config_hash": (None, [C.c_char_p, C.POINTER(_BuildConfig), C.c_char_p]),
    "w2x_pack_onnx": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_int]),
    "w2x_pack_info": (C.c_int, [C.c_char_p] + [C.POINTER(C.c_int)] * 4),
}

EXPORTED_SYMBOLS = sorted(_SIGNATURES)

# development build only (lib/libw2x_dev.so, -DW2X_DEV): micro-benchmarks declared in include/w2x_dev.h
_DEV_SIGNATURES = {
    "w2x_probe_umma": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "w2x_probe_mma_rate": (C.c_float, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "w2x_probe_hmma_rate": (C.c_float, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "w2x_probe_mma_tiles": (C.c_float, [C.c_int, C.c_int, C.c_int]),
    "w2x_probe_mma_rate_stream": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "w2x_probe_l2_stream": (C.c_float, [C.c_int, C.c_int, C.c_int]),
}
DEV_LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libw2x_dev.so")
_dev_lib = None


def dev_lib() -> C.CDLL:
    """lib/libw2x_dev.so: the same sources built with -DW2X_DEV (probes + the W2X_* switches that alter kernel work).
    Only scripts/ use it; tests and bench.py run the shipped library."""
    global _dev_lib
    if _dev_lib is None:
        l = C.CDLL(DEV_LIB_PATH)
        for name, (res, args) in {**_SIGNATURES, **_DEV_SIGNATURES}.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _dev_lib = l
    return _dev_lib


def use_dev_lib() -> None:
    """Route this process's w2x calls through lib/libw2x_dev.so (scripts/ only: kernel timing experiments)."""
    global _lib
    _lib = dev_lib()


def lib() -> C.CDLL:
    """Load libw2x.so (built in-tree by `make -C waifu2x-tensorrt_b200/csrc` / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with __graft_entry__.build(); there is no CPU fallback")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError here == the library does not export what w2x.h declares
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def _ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


# ---- host-only helpers ------------------------------------------------------------------------------
def calculate_tiles(in_w, in_h, out_w, out_h, tile_w, tile_h, out_tile_w, out_tile_h, scaling, overlap_x, overlap_y):
    """calculateTiles (img2img_render.cpp:7-66) -> (count, grid[8], in_rects, out_rects)."""
    l = lib()
    grid = (C.c_int * 8)()
    n = l.w2x_calculate_tiles(in_w, in_h, out_w, out_h, tile_w, tile_h, out_tile_w, out_tile_h, scaling,
                              overlap_x, overlap_y, None, None, 0, grid)
    if n < 0:
        raise ValueError("calculate_tiles failed")
    ir = (_Rect * max(n, 1))()
    orr = (_Rect * max(n, 1))()
    l.w2x_calculate_tiles(in_w, in_h, out_w, out_h, tile_w, tile_h, out_tile_w, out_tile_h, scaling,
                          overlap_x, overlap_y, ir, orr, n, grid)
    conv = lambda rs: [(r.x, r.y, r.width, r.height) for r in rs[:n]]
    return n, list(grid), conv(ir), conv(orr)


def blend_ramp(overlap: int) -> np.ndarray:
    out = np.zeros(max(overlap, 1), np.float32)
    n = lib().w2x_blend_ramp(overlap, out.ctypes.data_as(C.POINTER(C.c_float)))
    return out[:n]


def config_hash(device_name: str, cfg: BuildConfig) -> str:
    buf = C.create_string_buffer(65)
    lib().w2x_config_hash(device_name.encode(), C.byref(cfg._c()), buf)
    return buf.value.decode()


def pack_onnx(onnx_path: str, out_path: str, precision: int = PRECISION_FP16) -> None:
    err = C.create_string_buffer(512)
    if not lib().w2x_pack_onnx(onnx_path.encode(), out_path.encode(), precision, err, 512):
        raise RuntimeError(err.value.decode())


def select_engine(model_path: str, cfg: "RenderConfig", device_name: str) -> str:
    """img2img_load.cpp:79-114 without a GPU: the engine artefact `load` would pick on a device called device_name."""
    buf = C.create_string_buffer(4096)
    if not lib().w2x_select_engine(model_path.encode(), C.byref(cfg._c()), device_name.encode(), buf, 4096):
        raise RuntimeError(buf.value.decode())
    return buf.value.decode()


def pack_info(path: str):
    v = [C.c_int() for _ in range(4)]
    if not lib().w2x_pack_info(path.encode(), *[C.byref(x) for x in v]):
        raise RuntimeError("not a pack file: " + path)
    return dict(arch=v[0].value, scale=v[1].value, offset=v[2].value, layers=v[3].value)


# ---- stage entry points (GPU) ------------------------------------------------------------------------
def unpack_tiles(src_bgr: np.ndarray, rects: List[Tuple[int, int, int, int]], aug: List[int], tile: int, device: int = 0) -> np.ndarray:
    """-> float16 [n, tile, tile, 4] (RGB0)."""
    src = np.ascontiguousarray(src_bgr)
    n = len(rects)
    cr = (_Rect * n)(*[_Rect(*r) for r in rects])
    ca = (C.c_int * n)(*aug)
    out = np.empty((n, tile, tile, 4), np.float16)
    ok = lib().w2x_unpack_tiles(device, _ptr(src), src.shape[1], src.shape[0], src.strides[0], cr, ca, n, tile, _ptr(out))
    if not ok:
        raise RuntimeError("w2x_unpack_tiles failed")
    return out


def stitch_tiles(tiles_f16: np.ndarray, nx: int, ny: int, ov_x: int, ov_y: int, canvas_w: int, canvas_h: int, device: int = 0) -> np.ndarray:
    t = np.ascontiguousarray(tiles_f16, dtype=np.float16)
    count, out_tile = t.shape[0], t.shape[1]
    dst = np.empty((canvas_h, canvas_w, 3), np.uint8)
    ok = lib().w2x_stitch_tiles(device, _ptr(t), count, out_tile, nx, ny, ov_x, ov_y, canvas_w, canvas_h, _ptr(dst), dst.strides[0])
    if not ok:
        raise RuntimeError("w2x_stitch_tiles failed")
    return dst


def unpack_tiles_u16(src_bgr: np.ndarray, rects: List[Tuple[int, int, int, int]], aug: List[int], tile: int, device: int = 0) -> np.ndarray:
    """uint16 [H, W, 3] BGR (rows may be strided) -> float16 [n, tile, tile, 4] (RGB0), each sample x as fp16(f32(x) * f32(1/65535))."""
    src = src_bgr if _rows_of_pixels(src_bgr, 3, np.uint16) else np.ascontiguousarray(src_bgr, dtype=np.uint16)
    n = len(rects)
    cr = (_Rect * n)(*[_Rect(*r) for r in rects])
    ca = (C.c_int * n)(*aug)
    out = np.empty((n, tile, tile, 4), np.float16)
    ok = lib().w2x_unpack_tiles_u16(device, _ptr(src), src.shape[1], src.shape[0], src.strides[0], cr, ca, n, tile, _ptr(out))
    if not ok:
        raise RuntimeError("w2x_unpack_tiles_u16 failed")
    return out


def stitch_tiles_u16(tiles_f16: np.ndarray, nx: int, ny: int, ov_x: int, ov_y: int, canvas_w: int, canvas_h: int, device: int = 0) -> np.ndarray:
    """stitch_tiles with a uint16 [canvas_h, canvas_w, 3] BGR canvas: saturate(rint(65535 v)) of the same fp32 blend."""
    t = np.ascontiguousarray(tiles_f16, dtype=np.float16)
    count, out_tile = t.shape[0], t.shape[1]
    dst = np.empty((canvas_h, canvas_w, 3), np.uint16)
    ok = lib().w2x_stitch_tiles_u16(device, _ptr(t), count, out_tile, nx, ny, ov_x, ov_y, canvas_w, canvas_h, _ptr(dst), dst.strides[0])
    if not ok:
        raise RuntimeError("w2x_stitch_tiles_u16 failed")
    return dst


def tta_reduce(outs_f16: np.ndarray, device: int = 0) -> np.ndarray:
    t = np.ascontiguousarray(outs_f16, dtype=np.float16)  # [tiles, 8, T, T, 4]
    tiles, _, ot = t.shape[0], t.shape[1], t.shape[2]
    mean = np.empty((tiles, ot, ot, 4), np.float32)
    if not lib().w2x_tta_reduce(device, _ptr(t), tiles, ot, _ptr(mean)):
        raise RuntimeError("w2x_tta_reduce failed")
    return mean


def _rows_of_pixels(a: np.ndarray, channels: int, dtype) -> bool:
    """a is [H, W, channels] of dtype with contiguous pixels (rows may be strided, by whole samples from an aligned start)."""
    n = np.dtype(dtype).itemsize
    return (a.dtype == dtype and a.ndim == 3 and a.shape[2] == channels and a.strides[2] == n and a.strides[1] == channels * n
            and a.strides[0] % n == 0 and a.ctypes.data % n == 0)


def _call_packed(owner, fn, src_ptr: int, w: int, h: int, dst_ptr: int, pixel_bytes: int, size: Optional[Tuple[int, int]] = None) -> int:
    """fn, a frame entry point of owner (Img2Img or Img2ImgPool), on packed rows: src_ptr holds h rows of w pixels, dst_ptr the
    canvas (w * scaling x h * scaling), or with size = (dst_w, dst_h), dst_h rows of dst_w pixels."""
    src, dst = C.c_void_p(src_ptr), C.c_void_p(dst_ptr)
    if size is None:
        return int(fn(owner._h, src, w, h, w * pixel_bytes, dst, w * owner.scaling * pixel_bytes))
    dw, dh = int(size[0]), int(size[1])
    return int(fn(owner._h, src, w, h, w * pixel_bytes, dst, dw, dh, dw * pixel_bytes))


def alpha_bleed(src_bgra: np.ndarray, rounds: int, device: int = 0) -> np.ndarray:
    """The colour bleed of w2x_render_bgra (include/w2x_dev.h: w2x_alpha_bleed): uint8 [H, W, 4] BGRA -> uint8 [H, W, 4], alpha unchanged."""
    src = src_bgra if _rows_of_pixels(src_bgra, 4, np.uint8) else np.ascontiguousarray(src_bgra, dtype=np.uint8)
    h, w = src.shape[:2]
    out = np.empty((h, w, 4), np.uint8)
    if not lib().w2x_alpha_bleed(device, _ptr(src), w, h, src.strides[0], int(rounds), _ptr(out)):
        raise RuntimeError("w2x_alpha_bleed failed")
    return out


def resample_table(n_in: int, n_out: int):
    """The resample's table of one axis n_in -> n_out (include/w2x_dev.h: w2x_resample_table; no GPU needed): (first int32 [n_out],
    count int32 [n_out], weights float32 [n_out, taps]); output i reads inputs first[i] .. first[i] + count[i] - 1."""
    l = lib()
    taps = l.w2x_resample_table(int(n_in), int(n_out), None, None, None, 0)
    if taps <= 0:
        raise ValueError(f"resample_table: need 1 <= n_out <= n_in, got {n_in} -> {n_out}")
    first, count = np.empty(n_out, np.int32), np.empty(n_out, np.int32)
    weights = np.empty((n_out, taps), np.float32)
    if l.w2x_resample_table(int(n_in), int(n_out), _ptr(first), _ptr(count), _ptr(weights), weights.size) != taps:
        raise RuntimeError("w2x_resample_table failed")
    return first, count, weights


def resample(src_bgr: np.ndarray, size: Tuple[int, int], dst: Optional[np.ndarray] = None, device: int = 0) -> np.ndarray:
    """The resample of Img2Img.render_resized alone (include/w2x_dev.h: w2x_resample): uint8 [H, W, 3] BGR -> uint8 [dst_h, dst_w, 3],
    size = (dst_w, dst_h) with 1 <= dst_w <= W, 1 <= dst_h <= H.  src and a caller's dst may have strided rows."""
    src = src_bgr if _rows_of_pixels(src_bgr, 3, np.uint8) else np.ascontiguousarray(src_bgr, dtype=np.uint8)
    h, w = src.shape[:2]
    dw, dh = int(size[0]), int(size[1])
    if dst is None:
        dst = np.empty((dh, dw, 3), np.uint8)
    elif not _rows_of_pixels(dst, 3, np.uint8) or dst.shape[:2] != (dh, dw):
        raise ValueError("dst must be uint8 [dst_h, dst_w, 3] with contiguous pixels")
    if not lib().w2x_resample(device, _ptr(src), w, h, src.strides[0], _ptr(dst), dw, dh, dst.strides[0]):
        raise RuntimeError("w2x_resample failed")
    return dst


def run_conv_layer(kind: int, x: np.ndarray, w_packed: np.ndarray, bias: np.ndarray, cout: int, skip: Optional[np.ndarray] = None,
                   head: bool = False, device: int = 0) -> np.ndarray:
    """One layer of the dense path on host data (include/w2x_dev.h: w2x_run_conv_layer).  x: fp16 NHWC [n][h][w][cin];
    w_packed: fp16 [npad][ktot]; bias f32 [npad]; returns fp16 NHWC."""
    x = np.ascontiguousarray(x, np.float16)
    n, h, w, cin = x.shape
    shape = {0: (n, h - 2, w - 2, cout), 1: (n, h // 2, w // 2, cout), 2: (n, 2 * h, 2 * w, cout), 3: (n, 2 * h - 4, 2 * w - 4, 4),
             4: (n, h - 2, w - 2, 4)}[kind]
    out = np.zeros(shape, np.float16)
    wp = np.ascontiguousarray(w_packed, np.float16)
    b = np.ascontiguousarray(bias, np.float32)
    sk = np.ascontiguousarray(skip, np.float16) if skip is not None else None
    ok = lib().w2x_run_conv_layer(device, kind, int(head), n, h, w, cin, cout, _ptr(x), _ptr(wp), b.ctypes.data_as(C.POINTER(C.c_float)),
                                  _ptr(sk) if sk is not None else None, _ptr(out))
    if not ok:
        raise RuntimeError("w2x_run_conv_layer failed")
    return out


def run_conv_layer_f32(kind: int, x: np.ndarray, w_packed: np.ndarray, bias: np.ndarray, cout: int, skip: Optional[np.ndarray] = None,
                       device: int = 0) -> np.ndarray:
    """run_conv_layer through the tf32 kernel of --precision tf32 engines (include/w2x_dev.h: w2x_run_conv_layer_f32): x, skip and the
    result are float32 NHWC, w_packed float32 [npad][ktot] (the tensor core uses its TF32 part)."""
    x = np.ascontiguousarray(x, np.float32)
    n, h, w, cin = x.shape
    shape = {0: (n, h - 2, w - 2, cout), 1: (n, h // 2, w // 2, cout), 2: (n, 2 * h, 2 * w, cout), 3: (n, 2 * h - 4, 2 * w - 4, 4),
             4: (n, h - 2, w - 2, 4)}[kind]
    out = np.zeros(shape, np.float32)
    wp = np.ascontiguousarray(w_packed, np.float32)
    b = np.ascontiguousarray(bias, np.float32)
    sk = np.ascontiguousarray(skip, np.float32) if skip is not None else None
    ok = lib().w2x_run_conv_layer_f32(device, kind, n, h, w, cin, cout, _ptr(x), _ptr(wp), b.ctypes.data_as(C.POINTER(C.c_float)),
                                      _ptr(sk) if sk is not None else None, _ptr(out))
    if not ok:
        raise RuntimeError("w2x_run_conv_layer_f32 failed")
    return out


def run_swin_mlp(x: np.ndarray, gamma: np.ndarray, beta: np.ndarray, eps: float, w1: np.ndarray, b1: np.ndarray, w2: np.ndarray, b2: np.ndarray,
                 reps: int = 0, device: int = 0, variant: int = 0):
    """x + fc2(GELU(fc1(LayerNorm(x)))) through the fused MLP kernel (include/w2x_dev.h: w2x_run_swin_mlp).  x: fp16 [tokens][c],
    c = 96 or 192; w1 fp16 [2c][c], w2 fp16 [c][2c].  Returns (fp16 [tokens][c], average ms of `reps` extra launches or None)."""
    out = np.ascontiguousarray(x, np.float16).copy()
    assert out.ndim == 2 and out.shape[1] in (96, 192)
    c = out.shape[1]
    f32 = [np.ascontiguousarray(a, np.float32) for a in (gamma, beta, b1, b2)]
    f16 = [np.ascontiguousarray(a, np.float16) for a in (w1, w2)]
    assert f16[0].shape == (2 * c, c) and f16[1].shape == (c, 2 * c)
    ms = C.c_float(0)
    ok = lib().w2x_run_swin_mlp(device, out.shape[0], c, int(variant), _ptr(out), _ptr(f32[0]), _ptr(f32[1]), float(eps), _ptr(f16[0]), _ptr(f32[2]), _ptr(f16[1]), _ptr(f32[3]),
                                int(reps), C.byref(ms))
    if not ok:
        raise RuntimeError("w2x_run_swin_mlp failed")
    return out, (ms.value if reps > 0 else None)


def swin_attn_prepare(wqkv: np.ndarray, bqkv: np.ndarray, relpos: np.ndarray, heads: int = 6):
    """Host-side operand preparation of the fused attention kernel (include/w2x_dev.h: w2x_swin_attn_prepare; no GPU needed).
    Returns (w' fp16 [3c][c], b' f32 [3c], bias tables f32 [heads][36][pitch])."""
    wq = np.ascontiguousarray(wqkv, dtype=np.float16)
    c = wq.shape[1]
    b = np.ascontiguousarray(bqkv, dtype=np.float32)
    r = np.ascontiguousarray(relpos, dtype=np.float32)
    w_out, b_out, rel_out = np.zeros((3 * c, c), np.float16), np.zeros(3 * c, np.float32), np.zeros((heads, 36, 64), np.float32)
    pitch = lib().w2x_swin_attn_prepare(_ptr(wq), _ptr(b), _ptr(r), c, int(heads), _ptr(w_out), _ptr(b_out), _ptr(rel_out))
    if pitch <= 0 or pitch > 64:
        raise RuntimeError("w2x_swin_attn_prepare failed")
    return w_out, b_out, rel_out.reshape(-1)[: heads * 36 * pitch].reshape(heads, 36, pitch)


def compose_up_to_image(w_up: np.ndarray, b_up: np.ndarray, w_img: np.ndarray, b_img: np.ndarray):
    """PatchUp + ToImage(pixel shuffle 2) -> one linear map with a pixel shuffle of 4, from the PACKED layer operands
    (include/w2x_dev.h: w2x_compose_up_to_image; no GPU needed).  Returns (w fp16 [64][k], b f32 [64])."""
    wu, wi = np.ascontiguousarray(w_up, dtype=np.float16), np.ascontiguousarray(w_img, dtype=np.float16)
    bu, bi = np.ascontiguousarray(b_up, dtype=np.float32), np.ascontiguousarray(b_img, dtype=np.float32)
    cmid, k = wu.shape[0] // 4, wu.shape[1]
    if wi.shape != (16, cmid) or bu.shape != (4 * cmid,) or bi.shape != (16,):
        raise ValueError("compose_up_to_image: operand shapes")
    w_out, b_out = np.zeros((64, k), np.float16), np.zeros(64, np.float32)
    if not lib().w2x_compose_up_to_image(_ptr(wu), _ptr(bu), _ptr(wi), _ptr(bi), cmid, k, _ptr(w_out), _ptr(b_out)):
        raise RuntimeError("w2x_compose_up_to_image failed")
    return w_out, b_out


def run_swin_attn(x: np.ndarray, gamma: np.ndarray, beta: np.ndarray, eps: float, wqkv: np.ndarray, bqkv: np.ndarray, wproj, bproj,
                  relpos: np.ndarray, heads: int = 6, shift: int = 0, reps: int = 0, device: int = 0):
    """The fused attention kernel (include/w2x_dev.h: w2x_run_swin_attn).  x: fp16 [n][h][w][c]; wqkv [3c][c] fp16; relpos [heads][36][36] f32.
    c = 96: returns x + proj(window attention(LayerNorm(x))) (wproj [c][c] fp16, bproj [c]); c = 192: returns window attention(LayerNorm(x)),
    the kernel's output before the projection (wproj / bproj ignored).  Second value: ms per launch over `reps` extra launches, or None."""
    out = np.ascontiguousarray(x, dtype=np.float16).copy()
    n, h, w, c = out.shape
    wq = np.ascontiguousarray(wqkv, dtype=np.float16)
    f32 = [np.ascontiguousarray(a, dtype=np.float32) for a in (gamma, beta, bqkv, relpos)]
    if wq.shape != (3 * c, c) or f32[3].shape != (heads, 36, 36):
        raise ValueError("run_swin_attn: operand shapes")
    wp = bp = None
    if c == 96:
        wp, bp = np.ascontiguousarray(wproj, dtype=np.float16), np.ascontiguousarray(bproj, dtype=np.float32)
        if wp.shape != (c, c) or bp.shape != (c,):
            raise ValueError("run_swin_attn: operand shapes")
    ms = C.c_float(0.0)
    ok = lib().w2x_run_swin_attn(device, n, h, w, c, int(heads), int(shift), _ptr(out), _ptr(f32[0]), _ptr(f32[1]), float(eps), _ptr(wq), _ptr(f32[2]),
                                 _ptr(wp) if wp is not None else None, _ptr(bp) if bp is not None else None, _ptr(f32[3]), int(reps), C.byref(ms))
    if not ok:
        raise RuntimeError("w2x_run_swin_attn failed")
    return out, (ms.value if reps > 0 else None)


def selftest_conv(kind: int, n: int, h: int, w: int, cin: int, cout: int, seed: int = 1, device: int = 0) -> float:
    return float(lib().w2x_selftest_conv(device, kind, n, h, w, cin, cout, seed))


# ---- the operator surface ---------------------------------------------------------------------------
class Img2Img:
    """Python mirror of trt::Img2Img (src/tensorrt/img2img.h:14-50)."""

    def __init__(self):
        self._l = lib()
        self._h = self._l.w2x_create()
        if not self._h:
            raise RuntimeError("w2x_create failed")
        self._msg_cb = None
        self._prog_cb = None
        self.scaling = 1

    def close(self):
        if getattr(self, "_h", None):
            self._l.w2x_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def setMessageCallback(self, cb: Optional[Callable[[int, str], None]]):
        self._msg_cb = MESSAGE_CB(lambda sev, msg, user: cb(sev, msg.decode(errors="replace"))) if cb else MESSAGE_CB()
        self._l.w2x_set_message_callback(self._h, self._msg_cb, None)

    def setProgressCallback(self, cb: Optional[Callable[[int, int, float], None]]):
        self._prog_cb = PROGRESS_CB(lambda cur, tot, speed, user: cb(cur, tot, speed)) if cb else PROGRESS_CB()
        self._l.w2x_set_progress_callback(self._h, self._prog_cb, None)

    def build(self, path: str, config: BuildConfig) -> bool:
        return bool(self._l.w2x_build(self._h, path.encode(), C.byref(config._c())))

    def load(self, path: str, config: RenderConfig) -> bool:
        ok = bool(self._l.w2x_load(self._h, path.encode(), C.byref(config._c())))
        if ok:
            self.scaling = config.scaling
        return ok

    def render(self, src: np.ndarray, dst: Optional[np.ndarray] = None) -> Optional[np.ndarray]:
        """src: uint8 [H, W, 3] BGR.  Returns dst (uint8 [H*s, W*s, 3] BGR) or None on failure."""
        src = np.ascontiguousarray(src, dtype=np.uint8)
        h, w = src.shape[:2]
        if dst is None:
            dst = np.empty((h * self.scaling, w * self.scaling, 3), np.uint8)
        ok = self._l.w2x_render(self._h, _ptr(src), w, h, src.strides[0], _ptr(dst), dst.strides[0])
        return dst if ok else None

    # extensions
    def _render_frame(self, fn, src: np.ndarray, dst: Optional[np.ndarray], channels: int, dtype, size: Optional[Tuple[int, int]] = None):
        """fn (w2x_render_bgra / _resized / _u16) from src, whose rows may be strided (else it is copied), into the caller's dst, which
        must have contiguous pixels, or a new one: the canvas (H*s x W*s), or size = (dst_w, dst_h) (at least 1 x 1).  Returns dst, or None
        on failure (the reason in last_error)."""
        if not _rows_of_pixels(src, channels, dtype):
            src = np.ascontiguousarray(src, dtype=dtype)
        h, w = src.shape[:2]
        if dst is None:
            shape = (h * self.scaling, w * self.scaling) if size is None else (max(int(size[1]), 1), max(int(size[0]), 1))
            dst = np.empty(shape + (channels,), dtype)
        elif not _rows_of_pixels(dst, channels, dtype):
            raise ValueError(f"dst must be {np.dtype(dtype).name} [H, W, {channels}] with contiguous pixels")
        out_size = () if size is None else (int(size[0]), int(size[1]))
        ok = fn(self._h, _ptr(src), w, h, src.strides[0], _ptr(dst), *out_size, dst.strides[0])
        return dst if ok else None

    def render_bgra(self, src: np.ndarray, dst: Optional[np.ndarray] = None) -> Optional[np.ndarray]:
        """src: uint8 [H, W, 4] BGRA (rows may be strided).  Returns dst (uint8 [H*s, W*s, 4] BGRA; a caller's dst may have strided rows)
        or None on failure (the reason in last_error)."""
        return self._render_frame(self._l.w2x_render_bgra, src, dst, 4, np.uint8)

    def render_resized(self, src: np.ndarray, size: Tuple[int, int], dst: Optional[np.ndarray] = None) -> Optional[np.ndarray]:
        """src: uint8 [H, W, 3] BGR (rows may be strided); size = (dst_w, dst_h) with 1 <= dst_w <= W * scaling, 1 <= dst_h <= H * scaling.
        Returns dst (uint8 [dst_h, dst_w, 3] BGR: render(src) reduced by an antialiased bicubic resample, include/w2x.h w2x_render_resized;
        a caller's dst may have strided rows) or None on failure (the reason in last_error)."""
        return self._render_frame(self._l.w2x_render_resized, src, dst, 3, np.uint8, size)

    def submit_resized(self, src_ptr: int, w: int, h: int, dst_ptr: int, size: Tuple[int, int]) -> int:
        """submit with the output of render_resized: dst_ptr holds size[1] rows of 3 * size[0] bytes.  Returns a ticket for wait, or -1."""
        return _call_packed(self, self._l.w2x_submit_resized, src_ptr, w, h, dst_ptr, 3, size)

    def render_u16(self, src: np.ndarray, dst: Optional[np.ndarray] = None) -> Optional[np.ndarray]:
        """src: uint16 [H, W, 3] BGR (rows may be strided).  Returns dst (uint16 [H*s, W*s, 3] BGR, include/w2x.h w2x_render_u16; a
        caller's dst may have strided rows) or None on failure (the reason in last_error)."""
        return self._render_frame(self._l.w2x_render_u16, src, dst, 3, np.uint16)

    def submit_u16(self, src_ptr: int, w: int, h: int, dst_ptr: int) -> int:
        """submit with the frames of render_u16: src_ptr holds h rows of 6 * w bytes, dst_ptr h * s rows of 6 * w * s bytes.  Returns
        a ticket for wait, or -1."""
        return _call_packed(self, self._l.w2x_submit_u16, src_ptr, w, h, dst_ptr, 6)

    def infer(self, x_nchw: np.ndarray) -> Optional[np.ndarray]:
        x = np.ascontiguousarray(x_nchw, dtype=np.float32)
        n = x.shape[0]
        ot = self.output_tile_size
        out = np.empty((n, 3, ot, ot), np.float32)
        return out if self._l.w2x_infer(self._h, _ptr(x), n, _ptr(out)) else None

    @property
    def output_tile_size(self) -> int:
        return int(self._l.w2x_output_tile_size(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._l.w2x_launch_count(self._h))

    @property
    def flops_per_tile(self) -> float:
        return float(self._l.w2x_model_flops_per_tile(self._h))

    @property
    def last_error(self) -> str:
        return (self._l.w2x_last_error(self._h) or b"").decode(errors="replace")

    def last_stage_ms(self):
        buf = (C.c_float * 5)()
        n = self._l.w2x_last_stage_ms(self._h, buf, 5)
        return dict(zip(["unpack", "model", "stitch", "total", "tta_reduce"], list(buf)[:n]))

    def render_into(self, src: np.ndarray, dst: np.ndarray) -> bool:
        """w2x_render on caller-owned (pageable) arrays, no allocation: the literal drop-in call, used for timing."""
        h, w = src.shape[:2]
        return bool(self._l.w2x_render(self._h, _ptr(src), w, h, src.strides[0], _ptr(dst), dst.strides[0]))

    def timer_mark(self, idx: int, which: int = 0) -> bool:
        return bool(self._l.w2x_timer_mark(self._h, idx, which))

    def timer_elapsed_ms(self, i0: int, i1: int) -> float:
        return float(self._l.w2x_timer_elapsed_ms(self._h, i0, i1))

    def profile_layers(self, repeats: int = 5):
        cap = 256
        names = ((C.c_char * 48) * cap)()
        ms = (C.c_float * cap)()
        fl = (C.c_double * cap)()
        n = self._l.w2x_profile_layers(self._h, repeats, names, ms, fl, cap)
        if n < 0:
            raise RuntimeError(self.last_error)
        return [(names[i].value.decode(), ms[i], fl[i]) for i in range(n)]

    def layer_kernel(self, index: int) -> Optional[str]:
        buf = C.create_string_buffer(256)
        return buf.value.decode() if self._l.w2x_layer_kernel(self._h, index, buf, 256) else None

    # which: 0 layer output, 1 model input, 2 SE sums, 3 SE gate, 4 per-image folded weights (include/w2x_dev.h: w2x_layer_tensor)
    _LAYER_TENSOR_RANK = {0: 4, 1: 4, 2: 2, 3: 2, 4: 3}

    def layer_tensor(self, index: int, which: int = 0) -> Optional[np.ndarray]:
        """A copy of one tensor of plan layer `index` of a loaded CUNet engine, as the last batch left it: float16 or float32 (the
        engine's elements) for which 0, 1 and 4, int64 for 2, float32 for 3.  None when the layer has no such tensor."""
        dims = (C.c_int * 4)()
        n = self._l.w2x_layer_tensor(self._h, index, which, None, 0, dims)
        if n < 0:
            raise RuntimeError(self.last_error)
        if n == 0:
            return None
        shape = tuple(dims[:self._LAYER_TENSOR_RANK[which]])
        count = int(np.prod(shape))
        dtype = np.int64 if which == 2 else np.float32 if which == 3 else np.float16 if n == 2 * count else np.float32
        out = np.empty(shape, dtype)
        if out.nbytes != n or self._l.w2x_layer_tensor(self._h, index, which, _ptr(out), out.nbytes, dims) != n:
            raise RuntimeError(self.last_error or "w2x_layer_tensor: unexpected size")
        return out

    def render_device(self, d_src: int, w: int, h: int, d_dst: int) -> bool:
        return bool(_call_packed(self, self._l.w2x_render_device, d_src, w, h, d_dst, 3))

    def submit(self, src_ptr: int, w: int, h: int, dst_ptr: int) -> int:
        return _call_packed(self, self._l.w2x_submit, src_ptr, w, h, dst_ptr, 3)

    def wait(self, ticket: int) -> bool:
        return bool(self._l.w2x_wait(self._h, ticket))

    def sync(self) -> bool:
        return bool(self._l.w2x_sync(self._h))

    def device_alloc(self, nbytes: int) -> int:
        p = self._l.w2x_device_alloc(self._h, nbytes)
        if not p:
            raise MemoryError("w2x_device_alloc")
        return int(p)

    def device_free(self, p: int):
        self._l.w2x_device_free(self._h, C.c_void_p(p))

    def h2d(self, dptr: int, arr: np.ndarray):
        a = np.ascontiguousarray(arr)
        if not self._l.w2x_memcpy_h2d(self._h, C.c_void_p(dptr), _ptr(a), a.nbytes):
            raise RuntimeError("h2d failed")

    def d2h(self, arr: np.ndarray, dptr: int):
        if not self._l.w2x_memcpy_d2h(self._h, _ptr(arr), C.c_void_p(dptr), arr.nbytes):
            raise RuntimeError("d2h failed")


def render_banded(engines: List["Img2Img"], src: np.ndarray, dst: Optional[np.ndarray] = None) -> Optional[np.ndarray]:
    """One image over several engines (one per GPU): bands of tile rows + P2P seam exchange (SURVEY 8e).  Pass pinned arrays
    (PinnedArray.array) for src / dst to let the per-band copies of all GPUs overlap."""
    src = np.ascontiguousarray(src, dtype=np.uint8)
    h, w = src.shape[:2]
    s = engines[0].scaling
    if dst is None:
        dst = np.empty((h * s, w * s, 3), np.uint8)
    arr = (C.c_void_p * len(engines))(*[e._h for e in engines])
    ok = lib().w2x_render_banded(arr, len(engines), _ptr(src), w, h, src.strides[0], _ptr(dst), dst.strides[0])
    return dst if ok else None


class PinnedArray:
    """uint8 ndarray over cudaHostAlloc memory (for the pipelined submit path)."""

    def __init__(self, shape):
        self.nbytes = int(np.prod(shape))
        self.ptr = lib().w2x_host_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError("w2x_host_alloc")
        buf = (C.c_uint8 * self.nbytes).from_address(self.ptr)
        self.array = np.frombuffer(buf, np.uint8).reshape(shape)

    def free(self):
        if self.ptr:
            self.array = None
            lib().w2x_host_free(self.ptr)
            self.ptr = None


def model_path(models_dir: str, model: str, noise: int, scale: int) -> str:
    """models/<model>/[noiseN_][scaleSx].onnx, src/main.cpp:201-204 (trailing underscore for scale 1 kept, SURVEY q7)."""
    return os.path.join(models_dir, model, ("" if noise == -1 else f"noise{noise}_") + ("" if scale == 1 else f"scale{scale}x") + ".onnx")


class Img2ImgPool:
    """Frame-parallel multi-GPU rendering in one process (w2x_pool_*, include/w2x.h): frame f -> devices[f % len(devices)], one
    worker thread + engine + weight replica per device, frames retired by ticket."""

    def __init__(self, devices):
        self._l = lib()
        ids = (C.c_int * len(devices))(*devices)
        self._h = self._l.w2x_pool_create(ids, len(devices))
        if not self._h:
            raise RuntimeError("w2x_pool_create failed")
        self.devices = list(devices)
        self.scaling = 1
        self._msg_cb = None

    def close(self):
        if getattr(self, "_h", None):
            self._l.w2x_pool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def setMessageCallback(self, cb):
        """cb may be called from the pool's worker threads."""
        self._msg_cb = MESSAGE_CB(lambda sev, msg, user: cb(sev, msg.decode(errors="replace"))) if cb else MESSAGE_CB()
        self._l.w2x_pool_set_message_callback(self._h, self._msg_cb, None)

    def build(self, path: str, config: BuildConfig) -> bool:
        return bool(self._l.w2x_pool_build(self._h, path.encode(), C.byref(config._c())))

    def load(self, path: str, config: RenderConfig) -> bool:
        ok = bool(self._l.w2x_pool_load(self._h, path.encode(), C.byref(config._c())))
        if ok:
            self.scaling = config.scaling
        return ok

    def submit(self, src_ptr: int, w: int, h: int, dst_ptr: int) -> int:
        return _call_packed(self, self._l.w2x_pool_submit, src_ptr, w, h, dst_ptr, 3)

    def submit_resized(self, src_ptr: int, w: int, h: int, dst_ptr: int, size: Tuple[int, int]) -> int:
        """submit with the output of Img2Img.render_resized: dst_ptr holds size[1] rows of 3 * size[0] bytes."""
        return _call_packed(self, self._l.w2x_pool_submit_resized, src_ptr, w, h, dst_ptr, 3, size)

    def submit_u16(self, src_ptr: int, w: int, h: int, dst_ptr: int) -> int:
        """submit with the frames of Img2Img.render_u16: src_ptr holds h rows of 6 * w bytes, dst_ptr h * s rows of 6 * w * s bytes."""
        return _call_packed(self, self._l.w2x_pool_submit_u16, src_ptr, w, h, dst_ptr, 6)

    def wait(self, ticket: int) -> bool:
        return bool(self._l.w2x_pool_wait(self._h, ticket))

    def sync(self) -> bool:
        return bool(self._l.w2x_pool_sync(self._h))

    def launch_counts(self):
        return [int(self._l.w2x_launch_count(self._l.w2x_pool_engine(self._h, i))) for i in range(len(self.devices))]
