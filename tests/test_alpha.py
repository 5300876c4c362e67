"""BGRA rendering without a GPU: the colour-bleed oracle (tests/alpha_oracle.py), the CLI's --alpha flag, and host/videoio.hpp at four
channels with fake ffprobe / ffmpeg scripts that pass raw frames through."""
import os
import stat
import subprocess

import numpy as np
import pytest

from alpha_oracle import alpha_bleed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "waifu2x-tensorrt_b200")
CLI = os.path.join(PKG, "bin", "waifu2x-b200")


def _blobs(w, h, seed, p_visible=0.3):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    a[..., 3] = np.where(rng.random((h, w)) < p_visible, rng.integers(1, 256, (h, w)), 0)
    return a


@pytest.mark.parametrize("rounds", [1, 8, 18])
def test_bleed_is_identity_without_transparent_pixels(rounds):
    a = _blobs(40, 30, 1)
    a[..., 3] = np.maximum(a[..., 3], 1)
    assert np.array_equal(alpha_bleed(a, rounds), a)


def test_bleed_ignores_colour_under_alpha_zero():
    a = _blobs(50, 37, 2)
    b = a.copy()
    hidden = a[..., 3] == 0
    b[..., :3][hidden] = np.random.default_rng(3).integers(0, 256, (int(hidden.sum()), 3), dtype=np.uint8)
    assert not np.array_equal(a, b)
    assert np.array_equal(alpha_bleed(a, 8), alpha_bleed(b, 8))


def test_bleed_fill_lies_between_known_neighbours():
    """Each filled channel of a round lies between the min and max of the known neighbours it was computed from."""
    a = _blobs(64, 48, 4, p_visible=0.01)
    h, w = a.shape[:2]
    known = a[..., 3] > 0      # known after round r - 1
    for r in range(1, 6):
        prev, cur = alpha_bleed(a, r - 1), alpha_bleed(a, r)
        checked = 0
        for y, x in np.argwhere(~known):
            ys, xs = slice(max(y - 1, 0), y + 2), slice(max(x - 1, 0), x + 2)
            nb = known[ys, xs]
            if not nb.any():
                assert (cur[y, x, :3] == 0).all()
                continue
            vals = prev[ys, xs, :3][nb].astype(int)
            assert (vals.min(0) <= cur[y, x, :3]).all() and (cur[y, x, :3] <= vals.max(0)).all(), (r, y, x)
            checked += 1
        assert checked > 0
        kp = np.pad(known, 1)
        known = np.any([kp[1 + dy:1 + dy + h, 1 + dx:1 + dx + w] for dy in (-1, 0, 1) for dx in (-1, 0, 1)], axis=0)


@pytest.mark.parametrize("rounds", [0, 1, 5, 18])
@pytest.mark.parametrize("y,x,w,h", [(0, 0, 40, 30), (13, 21, 40, 30), (29, 39, 40, 30), (2, 3, 7, 5)])
def test_single_visible_pixel_fills_its_square(rounds, y, x, w, h):
    a = np.zeros((h, w, 4), np.uint8)
    a[..., :3] = 77
    a[y, x] = (10, 200, 31, 9)
    out = alpha_bleed(a, rounds)
    sq = np.zeros((h, w), bool)
    sq[max(y - rounds, 0):y + rounds + 1, max(x - rounds, 0):x + rounds + 1] = True
    assert (out[sq][:, :3] == (10, 200, 31)).all()
    assert (out[~sq][:, :3] == 0).all()
    assert np.array_equal(out[..., 3], a[..., 3])


def test_all_transparent_frame_becomes_zero():
    a = _blobs(20, 10, 5)
    a[..., 3] = 0
    assert not alpha_bleed(a, 18).any()


# ---- CLI -------------------------------------------------------------------------------------------------------------------------
BASE = ["--model", "cunet/art", "--scale", "2", "--noise", "0", "--batchSize", "2", "--tileSize", "64"]


def _cli(*args, cwd=None):
    return subprocess.run([CLI, *args], capture_output=True, text=True, cwd=cwd)


def test_cli_alpha_flag(tmp_path, built_lib):
    assert "--alpha" in _cli("--help").stdout
    assert _cli(*BASE, "build", "--alpha").returncode == 106            # render-only flag, like --tta
    # accepted by render: parsing passes and the run stops at the missing model (-1), not at the arguments (106)
    r = _cli(*BASE, "render", "-i", str(tmp_path), "--alpha", cwd=str(tmp_path))
    assert r.returncode == 255, r.stdout + r.stderr
    assert "not expected" not in r.stderr


# ---- videoio.hpp at four channels ----------------------------------------------------------------------------------------------
FAKE_FFPROBE = """#!/bin/bash
# prints the <input>.meta file the test wrote (key=value lines as `-of default=noprint_wrappers=1` would)
for last; do :; done
cat "$last.meta"
"""

FAKE_FFMPEG = """#!/bin/bash
# reader (`-f image2pipe`): records its command line as <input>.read_cmd and streams the input file, which holds raw frames;
# writer (`-i -`): records its command line as <output>.cmd and copies stdin to the output path
args=("$@")
for last; do :; done
if [[ " $* " == *" image2pipe "* ]]; then
  for ((i = 0; i < ${#args[@]}; i++)); do
    if [[ "${args[$i]}" == "-i" ]]; then echo "$@" > "${args[$((i + 1))]}.read_cmd"; exec cat "${args[$((i + 1))]}"; fi
  done
else
  echo "$@" > "$last.cmd"
  exec cat > "$last"
fi
"""

PROG = r"""
#include "videoio.hpp"
#include <cstdio>
#include <cstdlib>
#include <vector>
int main(int argc, char** argv) {
    // argv: ffmpegDir input output channels
    try {
        const int ch = std::atoi(argv[4]);
        VideoCapture cap;
        cap.setFfmpegDir(argv[1]).setChannels(ch);
        cap.open(argv[2]);
        const FrameSize sz = cap.getFrameSize();
        VideoWriter wr;
        wr.setFfmpegDir(argv[1]).setFrameSize(sz).setFrameRate(cap.getFrameRate()).setOutputFile(argv[3]).setCodec("libx264")
            .setPixelFormat("yuv420p").setConstantRateFactor(23).setChannels(ch);
        wr.open();
        std::vector<uint8_t> buf(sz.bytes(ch));
        int n = 0;
        while (cap.read(buf.data())) {
            for (auto& b : buf) b = 255 - b;
            wr.write(buf.data(), sz);
            ++n;
        }
        std::printf("%d %d %d\n", n, cap.getChannels(), wr.getChannels());
        cap.release();
        wr.release();
        try { cap.setChannels(2); return 7; } catch (const std::invalid_argument&) {}
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
"""


def _tools(d):
    for name, body in (("ffprobe", FAKE_FFPROBE), ("ffmpeg", FAKE_FFMPEG)):
        p = os.path.join(d, name)
        with open(p, "w") as f:
            f.write(body)
        os.chmod(p, os.stat(p).st_mode | stat.S_IXUSR)
    return d + "/"


def test_videoio_bgra_roundtrip_and_command_lines(tmp_path):
    d = str(tmp_path)
    tools = _tools(d)
    src = os.path.join(d, "prog.cpp")
    with open(src, "w") as f:
        f.write(PROG)
    exe = os.path.join(d, "prog")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(PKG, "host"), src, "-o", exe])
    rng = np.random.default_rng(0)
    cmds = {}
    for ch in (3, 4):
        frames = rng.integers(0, 256, (4, 12, 20, ch), dtype=np.uint8)
        vid = os.path.join(d, f"clip{ch}.mp4")
        frames.tofile(vid)
        with open(vid + ".meta", "w") as f:
            f.write("width=20\nheight=12\nr_frame_rate=30000/1001\nnb_frames=4\n")
        outp = os.path.join(d, f"out{ch}.mp4")
        r = subprocess.run([exe, tools, vid, outp, str(ch)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert r.stdout.split() == ["4", str(ch), str(ch)]
        assert np.array_equal(np.fromfile(outp, np.uint8).reshape(frames.shape), 255 - frames)
        cmds[ch] = (open(vid + ".read_cmd").read().strip().replace(vid, "IN"), open(outp + ".cmd").read().strip().replace(outp, "OUT"))
    assert "-pix_fmt bgr24" in cmds[3][0] and "-pix_fmt bgr24" in cmds[3][1]
    assert cmds[4][0] == cmds[3][0].replace("bgr24", "bgra")
    assert cmds[4][1] == cmds[3][1].replace("bgr24", "bgra")


@pytest.mark.parametrize("model,scale,rounds", [("cunet/art", 1, 28), ("cunet/art", 2, 18), ("swin_unet/art", 4, 8)])
def test_bleed_rounds_are_the_model_border(model, scale, rounds, tmp_path, built_lib):
    """The engine bleeds offset / scale rounds (the pack header's input-side border); BLEED_ROUNDS restates them."""
    import w2x
    import __graft_entry__
    from alpha_oracle import BLEED_ROUNDS
    _, path = __graft_entry__.make_synthetic_model(str(tmp_path), scale, 0, model=model)
    w2x.pack_onnx(path, str(tmp_path / "m.pack"))
    info = w2x.pack_info(str(tmp_path / "m.pack"))
    assert info["offset"] // info["scale"] == rounds == BLEED_ROUNDS[(model.split("/")[0], scale)]
