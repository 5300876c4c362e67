"""Resized output without a GPU: the host-built resample tables (w2x.resample_table) against a float64 NumPy restatement of the contract in
include/w2x.h (w2x_render_resized), that restatement against torch's antialiased bicubic interpolate, and the CLI's --outputScale checks."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_alpha import BASE, _cli

SIZES = [(3840, 2880), (2160, 1620), (256, 64), (97, 13), (1000, 999), (7, 1), (5, 3), (10, 10), (1, 1)]


def cubic(x, a=-0.5):
    x = abs(x)
    if x < 1:
        return ((a + 2) * x - (a + 3)) * x * x + 1
    if x < 2:
        return a * (((x - 5) * x + 8) * x - 4)
    return 0.0


def resample_matrix(n_in, n_out):
    """float64 [n_out, n_in]: row i holds the weights of output i (the formula of include/w2x.h)."""
    r = n_in / n_out
    s = max(r, 1.0)
    m = np.zeros((n_out, n_in))
    for i in range(n_out):
        c = r * (i + 0.5)
        lo, hi = max(math.floor(c - 2 * s + 0.5), 0), min(math.floor(c + 2 * s + 0.5), n_in)
        w = np.array([cubic((j - c + 0.5) / s) for j in range(lo, hi)])
        m[i, lo:hi] = w / w.sum()
    return m


def torch_resample(img, size):
    """The contract's reference: clamp(rint(R_y(R_x(img)))) of a u8 [H, W, 3] image to size = (dst_w, dst_h), R being torch's float64
    interpolate(mode="bicubic", antialias=True, align_corners=False).  Each axis is its own call along the width (R_y on the transposed
    image): torch 2.11's CPU kernel, asked for both axes at once, returns the first row for every output row when the output is one column
    wide and the height shrinks."""
    def along_w(t, n):
        return F.interpolate(t, size=(t.shape[2], n), mode="bicubic", antialias=True, align_corners=False)
    t = torch.from_numpy(np.ascontiguousarray(img, dtype=np.float64)).permute(2, 0, 1)[None]
    t = along_w(along_w(t, size[0]).transpose(2, 3), size[1]).transpose(2, 3)
    return np.clip(np.rint(t[0].permute(1, 2, 0).numpy()), 0, 255).astype(np.uint8)


def table_matrix(n_in, n_out):
    import w2x
    first, count, weights = w2x.resample_table(n_in, n_out)
    assert first.shape == count.shape == (n_out,) and weights.shape[0] == n_out
    m = np.zeros((n_out, n_in))
    for i in range(n_out):
        assert count[i] >= 1 and first[i] >= 0 and first[i] + count[i] <= n_in
        m[i, first[i]:first[i] + count[i]] = weights[i, :count[i]]
        assert not weights[i, count[i]:].any()
    return m, first, count


@pytest.mark.parametrize("n_in,n_out", SIZES)
def test_formula_is_torch_interpolate(n_in, n_out):
    eye = torch.eye(n_in, dtype=torch.float64).reshape(1, 1, n_in, n_in)
    t = F.interpolate(eye, size=(n_out, n_in), mode="bicubic", antialias=True, align_corners=False)[0, 0].numpy()
    assert np.abs(t - resample_matrix(n_in, n_out)).max() <= 1e-12


@pytest.mark.parametrize("w,h,dw,dh", [(1, 300, 1, 113), (300, 1, 113, 1), (2, 300, 1, 113), (97, 65, 13, 9), (7, 7, 1, 1), (640, 360, 427, 360),
                                       (640, 360, 640, 240), (1, 1, 1, 1)])
def test_torch_reference_is_the_formula(w, h, dw, dh):
    """torch_resample, which the GPU tests hold the kernels to, equals the float64 formula applied to a random image, before rounding."""
    img = np.random.default_rng(w * 7 + h).random((h, w, 3)) * 255
    want = np.einsum("ij,jkc->ikc", resample_matrix(h, dh), np.einsum("kl,jlc->jkc", resample_matrix(w, dw), img))
    got = torch_resample(img, (dw, dh))
    assert np.array_equal(got, np.clip(np.rint(want), 0, 255).astype(np.uint8))


def _check_table(n_in, n_out):
    want = resample_matrix(n_in, n_out)
    got, first, count = table_matrix(n_in, n_out)
    assert np.abs(got - want).max() <= 2 ** -24 * max(1.0, np.abs(want).max()) * 1.01, (n_in, n_out)
    # the window of every output covers each of its non-zero weights, and the windows are monotone (the engine's band rule needs both)
    for i in range(n_out):
        nz = np.flatnonzero(want[i])
        assert first[i] <= nz.min() and nz.max() < first[i] + count[i], (n_in, n_out, i)
    assert (np.diff(first) >= 0).all() and (np.diff(first + count) >= 0).all()
    return count


@pytest.mark.parametrize("n_in,n_out", SIZES)
def test_table_matches_formula(n_in, n_out, built_lib):
    count = _check_table(n_in, n_out)
    assert count.max() <= 4 * n_in / n_out + 3


def test_table_matches_formula_on_every_small_reduction(built_lib):
    for n in range(1, 41):
        for m in range(1, n + 1):
            _check_table(n, m)


def test_identity_axis_is_one_tap_of_weight_one(built_lib):
    import w2x
    for n in (1, 2, 7, 640):
        first, count, weights = w2x.resample_table(n, n)
        assert (first == np.arange(n)).all() and (count == 1).all() and (weights[:, 0] == 1).all()


@pytest.mark.parametrize("n_in,n_out", [(10, 11), (0, 1), (5, 0), (-3, -4)])
def test_table_refuses_enlargement_and_empty_axes(n_in, n_out, built_lib):
    import w2x
    with pytest.raises(ValueError):
        w2x.resample_table(n_in, n_out)


# ---- CLI -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("extra", [["--outputScale", "0"], ["--outputScale", "-1"], ["--outputScale=-0.5"], ["--outputScale", "2.01"],
                                   ["--outputScale", "4"], ["--outputScale", "abc"], ["--outputScale", "1.5x"], ["--outputScale", "nan"],
                                   ["--outputScale", "inf"], ["--outputScale", ""], ["--outputScale", "1.5", "--alpha"],
                                   ["--alpha", "--outputScale", "1"]])
def test_cli_output_scale_refusals(extra, tmp_path, built_lib):
    r = _cli(*BASE, "render", "-i", str(tmp_path), *extra, cwd=str(tmp_path))
    assert r.returncode == 106, r.stdout + r.stderr
    assert "--outputScale" in r.stderr


def test_cli_output_scale_flag(tmp_path, built_lib):
    assert "--outputScale" in _cli("--help").stdout
    assert _cli(*BASE, "build", "--outputScale", "1.5").returncode == 106      # render-only flag, like --tta
    # accepted by render up to --scale: parsing passes and the run stops at the missing model (-1), not at the arguments (106)
    for f in ("1.5", "2", "0.25", "1.3333"):
        r = _cli(*BASE, "render", "-i", str(tmp_path), "--outputScale", f, cwd=str(tmp_path))
        assert r.returncode == 255, r.stdout + r.stderr
        assert "not expected" not in r.stderr
