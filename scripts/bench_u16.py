"""bench_u16.py -- cost of 16-bit rendering (w2x_render_u16 / w2x_submit_u16) on cfg2 (cunet/art 2x, tile 256, batch 8, 1920x1080 ->
3840x2160) and cfg4 (swin_unet/art 4x, tile 256, batch 4, 1920x1080 -> 7680x4320), in one process on one GPU.

Per workload, four paths, alternating step by step so that clock and neighbour drift hit all of them alike:
  render       w2x_render on a BGR frame (pageable buffers), one synchronous call per frame
  render_u16   w2x_render_u16 on the same frame widened to 16 bits (257 x), one synchronous call per frame
  submit       w2x_submit / w2x_wait on pinned buffers: three frames in flight, then all three waited for (ms per frame)
  submit_u16   the same with w2x_submit_u16
Reported: the median wall-clock ms per frame and output Mpx/s over the timed frames, the frame bytes each path copies in and out, and for
the synchronous paths the median of each w2x_last_stage_ms stage (CUDA events on the engine's stream).  The card's name, power limit and
max SM clock are read with nvidia-smi in the same run.

    python scripts/bench_u16.py [--steps 32] [--warmup 3] [--out profiles/r05_u16.txt]
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
IN_FLIGHT = 3


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "nvidia-smi unavailable"


def run(wl, steps, warmup, path, say):
    import w2x
    from oracle import tiling
    s = wl["scale"]
    eng = w2x.Img2Img()
    msgs = []
    eng.setMessageCallback(lambda sev, m: msgs.append(m))
    if not eng.build(path, w2x.BuildConfig.fixed(wl["batch"], wl["tile"])):
        raise SystemExit(f"build failed: {msgs}")
    if not eng.load(path, w2x.RenderConfig(batchSize=wl["batch"], height=wl["tile"], width=wl["tile"], scaling=s, overlap=(BLEND, BLEND))):
        raise SystemExit(f"load failed: {msgs}")
    ow, oh = FRAME_W * s, FRAME_H * s
    bgr = tiling.synthetic_frame(FRAME_W, FRAME_H, 1)
    bgr16 = bgr.astype(np.uint16) * np.uint16(257)
    out8 = np.empty((oh, ow, 3), np.uint8)
    out16 = np.empty((oh, ow, 3), np.uint16)
    pins = []

    def pinned(shape, dtype):
        p = w2x.PinnedArray(tuple(shape[:-1]) + (shape[-1] * np.dtype(dtype).itemsize,))
        pins.append(p)
        return p, p.array.view(dtype).reshape(shape)

    sub = {}
    for k, frame, dtype in (("submit", bgr, np.uint8), ("submit_u16", bgr16, np.uint16)):
        ins = [pinned((FRAME_H, FRAME_W, 3), dtype) for _ in range(IN_FLIGHT)]
        outs = [pinned((oh, ow, 3), dtype) for _ in range(IN_FLIGHT)]
        for _, a in ins:
            a[...] = frame
        sub[k] = (ins, outs)

    def burst(k):
        ins, outs = sub[k]
        fn = eng.submit if k == "submit" else eng.submit_u16
        tickets = [fn(pi.ptr, FRAME_W, FRAME_H, po.ptr) for (pi, _), (po, _) in zip(ins, outs)]
        return all(t >= 0 for t in tickets) and all([eng.wait(t) for t in tickets])

    paths = {
        "render": (lambda: eng.render_into(bgr, out8), 1),
        "render_u16": (lambda: eng.render_u16(bgr16, out16) is not None, 1),
        "submit": (lambda: burst("submit"), IN_FLIGHT),
        "submit_u16": (lambda: burst("submit_u16"), IN_FLIGHT),
    }
    ms = {k: [] for k in paths}
    stages = {k: {st: [] for st in STAGES} for k in ("render", "render_u16")}
    for i in range(warmup + steps):
        for k, (fn, frames) in paths.items():
            t0 = time.perf_counter()
            assert fn(), eng.last_error
            dt = (time.perf_counter() - t0) * 1e3 / frames
            if i >= warmup:
                ms[k].append(dt)
                if k in stages:
                    st = eng.last_stage_ms()
                    for name in STAGES:
                        stages[k][name].append(st[name])
    d = np.abs(out16.astype(np.int64) - 257 * out8.astype(np.int64))
    say(f"   |render_u16(257 F) - 257 render(F)| max {int(d.max())} (contract: <= 129)")
    out_mpx = ow * oh / 1e6
    say(f"   {'path':10s} {'ms/frame':>9s} {'Mpx/s':>8s} {'x u8':>6s} {'MB in':>7s} {'MB out':>7s}   device stages, median ms: " +
        "  ".join(f"{n:>7s}" for n in STAGES))
    for k in paths:
        m = float(np.median(ms[k]))
        base = float(np.median(ms["render" if k.startswith("render") else "submit"]))
        b = 2 if k.endswith("u16") else 1
        line = (f"   {k:10s} {m:9.2f} {out_mpx / (m / 1e3):8.1f} {m / base:6.2f} {FRAME_W * FRAME_H * 3 * b / 1e6:7.1f} "
                f"{ow * oh * 3 * b / 1e6:7.1f}   ")
        if k in stages:
            line += "                             " + "  ".join(f"{float(np.median(stages[k][n])):7.3f}" for n in STAGES)
        say(line)
    for p in pins:
        p.free()
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
    say(f"{FRAME_W}x{FRAME_H} input frames, blend {BLEND}, {args.steps} timed steps per path after {args.warmup} warm-up steps, paths "
        f"alternating step by step; wall clock around each synchronous call (pageable host buffers) or around {IN_FLIGHT} pipelined "
        "submits and their waits (pinned host buffers); medians")
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
