"""NumPy restatement of the BGRA contract of w2x_render_bgra (include/w2x.h) for the tests, on top of oracle/tiling.py.

alpha_bleed: the colour bleed in integers, so the GPU must match it bit for bit.  render_bgra: opaque frames are tiling.render of the
B, G, R planes with alpha 255; otherwise the colour is tiling.render of the bled frame and the alpha is packed from the mean of the three
channels of the fp32 canvas that tiling.render accumulates for the grey frame B = G = R = alpha.
"""
from __future__ import annotations

import numpy as np

from oracle import tiling

# the model's input-side border (pack header offset / scale): the bleed rounds of each model the tests use
BLEED_ROUNDS = {("cunet", 1): 28, ("cunet", 2): 18, ("swin_unet", 4): 8}


def alpha_bleed(src_bgra: np.ndarray, rounds: int) -> np.ndarray:
    """A pixel is known when alpha > 0.  Each round (Jacobi: it reads the previous round's state only), every unknown pixel with n > 0
    known pixels in its 3 x 3 window (clipped to the image) takes (2 * sum + n) // (2 * n) per channel and becomes known.  Pixels still
    unknown at the end are (0, 0, 0).  Alpha is copied."""
    a = np.asarray(src_bgra, np.uint8)
    h, w = a.shape[:2]
    known = a[..., 3] > 0
    col = np.where(known[..., None], a[..., :3], 0).astype(np.int64)
    for _ in range(rounds):
        kp = np.pad(known, 1).astype(np.int64)
        cp = np.pad(col * known[..., None], ((1, 1), (1, 1), (0, 0)))
        n = np.zeros((h, w), np.int64)
        s = np.zeros((h, w, 3), np.int64)
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                if dy == 0 and dx == 0:
                    continue
                n += kp[1 + dy:1 + dy + h, 1 + dx:1 + dx + w]
                s += cp[1 + dy:1 + dy + h, 1 + dx:1 + dx + w]
        grow = ~known & (n > 0)
        nn = n[grow][:, None]
        col[grow] = (2 * s[grow] + nn) // (2 * nn)
        known = known | grow
    col[~known] = 0
    out = np.empty_like(a)
    out[..., :3] = col
    out[..., 3] = a[..., 3]
    return out


def render_canvas(src_bgr: np.ndarray, model, *args, **kwargs) -> np.ndarray:
    """The fp32 RGB canvas tiling.render packs into its result (same arguments as tiling.render).  tiling.render ends with
    pack_u8(canvas); the canvas is taken there, so the loop is not restated."""
    captured = []
    pack = tiling.pack_u8

    def keep(canvas):
        captured.append(np.array(canvas, np.float32))
        return pack(canvas)

    tiling.pack_u8 = keep
    try:
        tiling.render(src_bgr, model, *args, **kwargs)
    finally:
        tiling.pack_u8 = pack
    return captured[-1]


def render_bgra(src_bgra: np.ndarray, model, tile: int, out_tile: int, scaling: int, overlap: float, batch: int = 1, tta: bool = False,
                rounds: int = 0) -> np.ndarray:
    """w2x_render_bgra: uint8 [H, W, 4] BGRA -> uint8 [H*s, W*s, 4] BGRA.  rounds: the model's BLEED_ROUNDS."""
    src = np.asarray(src_bgra, np.uint8)
    alpha = src[..., 3]
    args = (model, tile, out_tile, scaling, overlap, batch)
    h, w = src.shape[:2]
    out = np.empty((h * scaling, w * scaling, 4), np.uint8)
    colour = alpha_bleed(src, rounds) if (alpha == 0).any() else src
    out[..., :3] = tiling.render(np.ascontiguousarray(colour[..., :3]), *args, tta=tta)
    if (alpha == 255).all():
        out[..., 3] = 255
        return out
    c = render_canvas(np.repeat(alpha[..., None], 3, axis=2), *args, tta=tta)
    out[..., 3] = tiling.pack_u8((c[..., 0] + c[..., 1] + c[..., 2]) / np.float32(3))
    return out


def masked_frame(w: int, h: int, seed: int) -> np.ndarray:
    """A synthetic BGRA frame: tiling.synthetic_frame colour under soft-edged ellipses on a transparent background (about half of the
    pixels at alpha 0), with random colour under the transparent pixels."""
    rng = np.random.default_rng(seed)
    bgr = tiling.synthetic_frame(w, h, seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    a = np.zeros((h, w), np.float32)
    for _ in range(6):
        cx, cy = rng.uniform(0, w), rng.uniform(0, h)
        rx, ry = rng.uniform(0.1, 0.3) * w, rng.uniform(0.1, 0.3) * h
        d = np.sqrt(((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2)
        a = np.maximum(a, np.clip((1.15 - d) / 0.3, 0, 1))
    out = np.empty((h, w, 4), np.uint8)
    out[..., :3] = np.where((a > 0)[..., None], bgr, rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
    out[..., 3] = np.rint(a * 255).astype(np.uint8)
    return out
