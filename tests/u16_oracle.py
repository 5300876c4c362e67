"""NumPy restatement of the 16-bit contract of w2x_render_u16 (include/w2x.h) for the tests, on top of oracle/tiling.py.

The input side is tiling.render with each sample x taken as f32(x) * f32(1/65535) instead of f32(x) * f32(1/255); the output side packs
the same fp32 canvas with saturate_u16(rint(65535 v)).  tiling.render is wrapped, not restated: its normaliser is swapped for the call
and its canvas taken where it packs, as tests/alpha_oracle.py does.
"""
from __future__ import annotations

import numpy as np

from oracle import tiling

K16 = np.float32(1.0 / 65535.0)


def normalize_u16(tile_u16: np.ndarray) -> np.ndarray:
    """f32(u16) * f32(1/65535), one rounded fp32 multiply."""
    return tile_u16.astype(np.float32) * K16


def pack_u16(canvas: np.ndarray) -> np.ndarray:
    """saturate_u16(rint(f32(v) * 65535)): round to nearest even, then clamp to [0, 65535]."""
    v = np.asarray(canvas, np.float32) * np.float32(65535.0)
    return np.clip(np.rint(v), 0, 65535).astype(np.uint16)


def canvas_u16(src_bgr_u16: np.ndarray, model, *args, **kwargs) -> np.ndarray:
    """The fp32 RGB canvas of tiling.render run on a uint16 [H, W, 3] BGR frame with the 16-bit normaliser (same arguments as
    tiling.render after the frame)."""
    captured = []
    norm, pack = tiling.normalize_u8, tiling.pack_u8

    def keep(canvas):
        captured.append(np.array(canvas, np.float32))
        return pack(canvas)

    tiling.normalize_u8, tiling.pack_u8 = normalize_u16, keep
    try:
        tiling.render(np.asarray(src_bgr_u16, np.uint16), model, *args, **kwargs)
    finally:
        tiling.normalize_u8, tiling.pack_u8 = norm, pack
    return captured[-1]


def render_u16(src_bgr_u16: np.ndarray, model, *args, **kwargs) -> np.ndarray:
    """w2x_render_u16: uint16 [H, W, 3] BGR -> uint16 [H*s, W*s, 3] BGR."""
    return pack_u16(canvas_u16(src_bgr_u16, model, *args, **kwargs))[..., ::-1].copy()
