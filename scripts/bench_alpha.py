"""bench_alpha.py -- cost of BGRA rendering (w2x_render_bgra) on cfg2 (cunet/art 2x, tile 256, batch 8, 1920x1080 -> 3840x2160) and cfg4
(swin_unet/art 4x, tile 256, batch 4, 1920x1080 -> 7680x4320), in one process on one GPU.

Per workload, three synchronous host-buffer paths, alternating frame by frame so that clock and neighbour drift hit all three alike:
  bgr        w2x_render on a BGR frame (pageable buffers)
  opaque     w2x_render_bgra on the same frame with alpha 255 everywhere (alpha scan, no alpha pass)
  masked     w2x_render_bgra on a seeded mask: soft-edged ellipses on a transparent background, about half of the pixels at alpha 0
             (alpha scan, colour bleed, alpha model pass)
Reported: the median wall-clock ms per frame and output Mpx/s over the timed frames, and the median of each w2x_last_stage_ms stage (CUDA
events on the engine's stream; the scan and bleed count as unpack).  The card's name, power limit and max SM clock are read with
nvidia-smi in the same run.

    python scripts/bench_alpha.py [--steps 32] [--warmup 3] [--out profiles/r04_alpha.txt]
"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "waifu2x-tensorrt_b200"), os.path.join(ROOT, "tests")]

FRAME_W, FRAME_H, BLEND = 1920, 1080, 1 / 16
WORKLOADS = {
    "cfg2": dict(model="cunet/art", scale=2, tile=256, batch=8),
    "cfg4": dict(model="swin_unet/art", scale=4, tile=256, batch=4),
}
STAGES = ["unpack", "model", "stitch", "total"]


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "nvidia-smi unavailable"


def run(wl, steps, warmup, path, say):
    import w2x
    from alpha_oracle import masked_frame
    from oracle import tiling
    s = wl["scale"]
    eng = w2x.Img2Img()
    msgs = []
    eng.setMessageCallback(lambda sev, m: msgs.append(m))
    if not eng.build(path, w2x.BuildConfig.fixed(wl["batch"], wl["tile"])):
        raise SystemExit(f"build failed: {msgs}")
    if not eng.load(path, w2x.RenderConfig(batchSize=wl["batch"], height=wl["tile"], width=wl["tile"], scaling=s, overlap=(BLEND, BLEND))):
        raise SystemExit(f"load failed: {msgs}")
    bgr = tiling.synthetic_frame(FRAME_W, FRAME_H, 1)
    opaque = np.empty((FRAME_H, FRAME_W, 4), np.uint8)
    opaque[..., :3] = bgr
    opaque[..., 3] = 255
    masked = masked_frame(FRAME_W, FRAME_H, 2)
    out3 = np.empty((FRAME_H * s, FRAME_W * s, 3), np.uint8)
    out4 = np.empty((FRAME_H * s, FRAME_W * s, 4), np.uint8)
    paths = {
        "bgr": lambda: eng.render_into(bgr, out3),
        "opaque": lambda: eng.render_bgra(opaque, out4) is not None,
        "masked": lambda: eng.render_bgra(masked, out4) is not None,
    }
    ms = {k: [] for k in paths}
    stages = {k: {st: [] for st in STAGES} for k in paths}
    for i in range(warmup + steps):
        for k, fn in paths.items():
            t0 = time.perf_counter()
            assert fn(), eng.last_error
            dt = (time.perf_counter() - t0) * 1e3
            if i >= warmup:
                ms[k].append(dt)
                st = eng.last_stage_ms()
                for name in STAGES:
                    stages[k][name].append(st[name])
    out_mpx = FRAME_W * s * FRAME_H * s / 1e6
    say(f"   transparent pixels of the mask: {100 * (masked[..., 3] == 0).mean():.1f} %, partly transparent: "
        f"{100 * ((masked[..., 3] > 0) & (masked[..., 3] < 255)).mean():.1f} %")
    say(f"   {'path':8s} {'ms/frame':>9s} {'Mpx/s':>8s} {'x bgr':>6s}   device stages, median ms: " + "  ".join(f"{n:>7s}" for n in STAGES))
    base = float(np.median(ms["bgr"]))
    for k in paths:
        m = float(np.median(ms[k]))
        say(f"   {k:8s} {m:9.2f} {out_mpx / (m / 1e3):8.1f} {m / base:6.2f}                                " +
            "  ".join(f"{float(np.median(stages[k][n])):7.3f}" for n in STAGES))
    um = float(np.median(stages["masked"]["unpack"]))
    tm = float(np.median(stages["masked"]["total"]))
    say(f"   masked: unpack stage (alpha scan + colour bleed + unpack of both passes) {um:.3f} ms = {100 * um / tm:.2f} % of its device time")
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import __graft_entry__
    lines = []
    say = lambda s="": (print(s, flush=True), lines.append(s))
    say(f"card (name, power limit, max SM clock): {card()}")
    say(f"{FRAME_W}x{FRAME_H} input frames, blend {BLEND}, {args.steps} timed frames per path after {args.warmup} warm-up frames, "
        "paths alternating frame by frame; wall clock around each synchronous call (pageable host buffers)")
    with tempfile.TemporaryDirectory() as d:
        for name, wl in WORKLOADS.items():
            _, path = __graft_entry__.make_synthetic_model(d, scale=wl["scale"], noise=0, model=wl["model"])
            say()
            say(f"== {name}: {wl['model']} {wl['scale']}x, tile {wl['tile']}, batch {wl['batch']}, -> {FRAME_W * wl['scale']}x{FRAME_H * wl['scale']}")
            run(wl, args.steps, args.warmup, path, say)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
