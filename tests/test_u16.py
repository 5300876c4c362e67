"""16 bits per channel without a GPU: the normalisation identity that ties w2x_render_u16 to w2x_render on fp16 engines, the u16 pack of
tests/u16_oracle.py, the CLI's --bitDepth flag, and host/videoio.hpp at 16 bits with the fake ffprobe / ffmpeg of tests/test_alpha.py."""
import os
import subprocess

import numpy as np
import pytest

from oracle import tiling
from u16_oracle import K16, canvas_u16, normalize_u16, pack_u16

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "waifu2x-tensorrt_b200")


def test_normalisation_identity_for_every_u8_value():
    """fp16(f32(257 x) * f32(1/65535)) == fp16(f32(x) * f32(1/255)) for all 256 u8 values, so render_u16(257 F) feeds an fp16 engine the
    tiles render(F) does.  At fp32 the two differ by one ulp for some values (tf32 engines get no such identity)."""
    x = np.arange(256, dtype=np.uint16)
    wide = normalize_u16(x * np.uint16(257))
    narrow = tiling.normalize_u8(x.astype(np.uint8))
    assert np.array_equal(wide.astype(np.float16).view(np.uint16), narrow.astype(np.float16).view(np.uint16))
    assert (wide != narrow).sum() > 0


def test_normaliser_is_one_rounded_multiply():
    x = np.arange(65536, dtype=np.uint16)
    assert np.array_equal(normalize_u16(x), x.astype(np.float32) * np.float32(1.0 / 65535.0))
    assert K16 == np.float32(1 / 65535) and normalize_u16(np.uint16(65535)) == np.float32(1.0)


def test_pack_u16_rounds_to_nearest_even_and_saturates():
    k = np.float32(65535)
    v = np.array([0.5 / k, 1.5 / k, 2.5 / k, -3.0, 7.0, -0.0, 1.0, 0.0, np.float32(65534.5) / k], np.float32)
    got = pack_u16(v)
    want = np.clip(np.rint(v * k), 0, 65535).astype(np.uint16)
    assert np.array_equal(got, want)
    assert got[3] == 0 and got[4] == 65535 and got[6] == 65535


def test_pack_u16_is_within_129_of_257_times_pack_u8():
    """The bound of the u8 relation: for any fp32 canvas value, |pack_u16(v) - 257 pack_u8(v)| <= 129."""
    v = np.linspace(-0.01, 1.01, 2_000_003, dtype=np.float32)
    d = np.abs(pack_u16(v).astype(np.int64) - 257 * tiling.pack_u8(v).astype(np.int64))
    assert d.max() <= 129


def test_u16_oracle_on_widened_u8_frame_matches_u8_canvas_at_fp16():
    """With a model that rounds its input to fp16 (as an fp16 engine does), the 16-bit oracle of 257 F blends the canvas of F."""
    f = tiling.synthetic_frame(40, 30, 3)

    def model(x):
        x = x.astype(np.float16).astype(np.float32)
        return np.repeat(np.repeat(x * np.float32(0.9) + np.float32(0.05), 2, axis=2), 2, axis=3)

    from alpha_oracle import render_canvas
    a = canvas_u16(f.astype(np.uint16) * np.uint16(257), model, 16, 32, 2, 1 / 16, 3)
    b = render_canvas(f, model, 16, 32, 2, 1 / 16, 3)
    assert np.array_equal(a, b)


# ---- CLI -------------------------------------------------------------------------------------------------------------------------
def test_cli_bit_depth_flag(tmp_path, built_lib):
    from test_alpha import BASE, _cli
    assert "--bitDepth" in _cli("--help").stdout
    for args in (["render", "-i", str(tmp_path), "--bitDepth", "12"], ["render", "-i", str(tmp_path), "--bitDepth", "x"],
                 ["build", "--bitDepth", "16"], ["build", "--bitDepth", "8"],
                 ["render", "-i", str(tmp_path), "--bitDepth", "16", "--alpha"],
                 ["render", "-i", str(tmp_path), "--bitDepth", "16", "--outputScale", "1.5"]):
        r = _cli(*BASE, *args)
        assert r.returncode == 106, (args, r.stdout + r.stderr)
        assert "--bitDepth" in r.stderr, (args, r.stderr)
    # accepted by render: parsing passes and the run stops at the missing model (-1), not at the arguments (106)
    for depth in ("8", "16"):
        r = _cli(*BASE, "render", "-i", str(tmp_path), "--bitDepth", depth, cwd=str(tmp_path))
        assert r.returncode == 255, r.stdout + r.stderr
        assert "not expected" not in r.stderr


# ---- videoio.hpp at 16 bits ------------------------------------------------------------------------------------------------------
PROG16 = r"""
#include "videoio.hpp"
#include <cstdio>
#include <cstdlib>
#include <vector>
int main(int argc, char** argv) {
    // argv: ffmpegDir input output bitDepth
    try {
        const int depth = std::atoi(argv[4]);
        VideoCapture cap;
        cap.setFfmpegDir(argv[1]).setBitDepth(depth);
        cap.open(argv[2]);
        const FrameSize sz = cap.getFrameSize();
        VideoWriter wr;
        wr.setFfmpegDir(argv[1]).setFrameSize(sz).setFrameRate(cap.getFrameRate()).setOutputFile(argv[3]).setCodec("libx264")
            .setPixelFormat("yuv420p").setConstantRateFactor(23).setBitDepth(depth);
        wr.open();
        std::vector<uint8_t> buf(sz.bytes(3, depth));
        int n = 0;
        while (cap.read(buf.data())) {
            for (auto& b : buf) b = 255 - b;
            wr.write(buf.data(), sz);
            ++n;
        }
        std::printf("%d %d %d %zu\n", n, cap.getBitDepth(), wr.getBitDepth(), sz.bytes(3, depth));
        cap.release();
        wr.release();
        int refused = 0;
        try { cap.setBitDepth(12); } catch (const std::invalid_argument&) { ++refused; }
        try { VideoCapture c; c.setBitDepth(16).setChannels(4); } catch (const std::invalid_argument&) { ++refused; }
        try { VideoWriter w; w.setChannels(4).setBitDepth(16); } catch (const std::invalid_argument&) { ++refused; }
        try { rawPixelFormat(4, 16); } catch (const std::invalid_argument&) { ++refused; }
        if (refused != 4) return 7;
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
"""


def test_videoio_16bit_roundtrip_and_command_lines(tmp_path):
    from test_alpha import _tools
    d = str(tmp_path)
    tools = _tools(d)
    src = os.path.join(d, "prog.cpp")
    with open(src, "w") as f:
        f.write(PROG16)
    exe = os.path.join(d, "prog")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(PKG, "host"), src, "-o", exe])
    rng = np.random.default_rng(0)
    cmds = {}
    for depth, dtype in ((8, np.uint8), (16, np.uint16)):
        frames = rng.integers(0, np.iinfo(dtype).max + 1, (4, 12, 20, 3), dtype=dtype)
        vid = os.path.join(d, f"clip{depth}.mp4")
        frames.astype("<" + np.dtype(dtype).str[1:]).tofile(vid)
        with open(vid + ".meta", "w") as f:
            f.write("width=20\nheight=12\nr_frame_rate=30000/1001\nnb_frames=4\n")
        outp = os.path.join(d, f"out{depth}.mp4")
        r = subprocess.run([exe, tools, vid, outp, str(depth)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert r.stdout.split() == ["4", str(depth), str(depth), str(12 * 20 * 3 * depth // 8)]
        # every byte inverted: for u16 samples that is 65535 - x as well
        got = np.fromfile(outp, "<" + np.dtype(dtype).str[1:]).reshape(frames.shape)
        assert np.array_equal(got, np.iinfo(dtype).max - frames)
        cmds[depth] = (open(vid + ".read_cmd").read().strip().replace(vid, "IN"), open(outp + ".cmd").read().strip().replace(outp, "OUT"))
    assert "-pix_fmt bgr24" in cmds[8][0] and "-pix_fmt bgr24" in cmds[8][1]
    assert cmds[16][0] == cmds[8][0].replace("bgr24", "bgr48le")
    assert cmds[16][1] == cmds[8][1].replace("bgr24", "bgr48le")
