"""bench_tf32.py -- --precision tf32 against fp16 on cfg2's shape (cunet/art 2x, tile 256, batch 8, 1920x1080 -> 3840x2160), both in
the same process on one GPU.

Per precision:
  value     output Mpx/s of whole frames already resident in HBM (w2x_render_device), CUDA events on the engine's stream
  e2e_sync  output Mpx/s of the synchronous drop-in call (w2x_render, pageable host buffers), wall clock
  layers    profile_layers: per-layer device time of one batch, achieved TFLOP/s and share of the data-sheet dense peak of that precision
            (B200: 1,125 TFLOP/s TF32, 2,250 TFLOP/s FP16); the RGB first layers' share of the model time
The card's name, power limit and max SM clock are read with nvidia-smi in the same run.

    python scripts/bench_tf32.py [--steps 20] [--warmup 3] [--out profiles/r03_tf32_cfg2.txt]
"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "waifu2x-tensorrt_b200")]

FRAME_W, FRAME_H, TILE, BATCH, SCALE, BLEND = 1920, 1080, 256, 8, 2, 1 / 16
PEAK_TFLOPS = {"tf32": 1125.0, "fp16": 2250.0}


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "nvidia-smi unavailable"


def run(precision_name, steps, warmup, path):
    import w2x
    from oracle import tiling
    precision = w2x.PRECISION_TF32 if precision_name == "tf32" else w2x.PRECISION_FP16
    eng = w2x.Img2Img()
    msgs = []
    eng.setMessageCallback(lambda s, m: msgs.append(m))
    if not eng.build(path, w2x.BuildConfig.fixed(BATCH, TILE, precision=precision)):
        raise SystemExit(f"build failed: {msgs}")
    if not eng.load(path, w2x.RenderConfig(precision=precision, batchSize=BATCH, height=TILE, width=TILE, scaling=SCALE, overlap=(BLEND, BLEND))):
        raise SystemExit(f"load failed: {msgs}")
    frames = [tiling.synthetic_frame(FRAME_W, FRAME_H, s) for s in range(4)]
    out_mpx = FRAME_W * SCALE * FRAME_H * SCALE / 1e6
    d_in = [eng.device_alloc(FRAME_W * FRAME_H * 3) for _ in frames]
    for d, f in zip(d_in, frames):
        eng.h2d(d, f)
    d_out = eng.device_alloc(FRAME_W * SCALE * FRAME_H * SCALE * 3)
    for i in range(warmup):
        assert eng.render_device(d_in[i % 4], FRAME_W, FRAME_H, d_out), eng.last_error
    eng.sync()
    eng.timer_mark(0)
    for i in range(steps):
        assert eng.render_device(d_in[i % 4], FRAME_W, FRAME_H, d_out), eng.last_error
    eng.timer_mark(1)
    eng.sync()
    ms = eng.timer_elapsed_ms(0, 1)
    value = steps * out_mpx / (ms / 1e3)
    page_out = np.empty((FRAME_H * SCALE, FRAME_W * SCALE, 3), np.uint8)
    for i in range(2):
        assert eng.render_into(frames[i % 4], page_out), eng.last_error
    t0 = time.perf_counter()
    for i in range(steps):
        assert eng.render_into(frames[i % 4], page_out), eng.last_error
    sync_ms = (time.perf_counter() - t0) * 1e3
    e2e_sync = steps * out_mpx / (sync_ms / 1e3)
    last = page_out.copy()
    layers = eng.profile_layers(10)
    kernels = [eng.layer_kernel(i) for i in range(len(layers))]
    eng.close()
    return dict(value=value, ms_per_frame=ms / steps, e2e_sync=e2e_sync, sync_ms_per_frame=sync_ms / steps, layers=layers, kernels=kernels, last=last)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import __graft_entry__
    lines = []
    say = lambda s="": (print(s, flush=True), lines.append(s))
    with tempfile.TemporaryDirectory() as d:
        _, path = __graft_entry__.make_synthetic_model(d, scale=SCALE, noise=0)
        say(f"card (name, power limit, max SM clock): {card()}")
        say(f"workload: cunet/art {SCALE}x, tile {TILE}, batch {BATCH}, {FRAME_W}x{FRAME_H} -> {FRAME_W * SCALE}x{FRAME_H * SCALE}, "
            f"blend {BLEND}, {args.steps} timed frames after {args.warmup} warm-up frames")
        res = {}
        for name in ("tf32", "fp16"):
            r = run(name, args.steps, args.warmup, path)
            res[name] = r
            say()
            say(f"== {name}: value {r['value']:.1f} Mpx/s ({r['ms_per_frame']:.2f} ms/frame, w2x_render_device, CUDA events) | "
                f"e2e_sync {r['e2e_sync']:.1f} Mpx/s ({r['sync_ms_per_frame']:.2f} ms/frame, w2x_render, wall clock)")
            say(f"   per layer, one batch of {BATCH} tiles (profile_layers, 10 repeats); % of the data-sheet dense {name.upper()} peak "
                f"({PEAK_TFLOPS[name]:.0f} TFLOP/s)")
            total = sum(ms for _, ms, _ in r["layers"])
            first = 0.0
            for (lname, ms, fl), k in zip(r["layers"], r["kernels"]):
                tf = fl / (ms * 1e-3) / 1e12 if ms > 0 and fl > 0 else 0.0
                if k and k.startswith("first-layer"):
                    first += ms
                say(f"   {lname:28s} {ms:8.4f} ms {100 * ms / total:5.1f} %  {tf:7.1f} TFLOP/s {100 * tf / PEAK_TFLOPS[name]:5.1f} %  {k}")
            say(f"   model total {total:.3f} ms per batch; RGB first layers {first:.4f} ms = {100 * first / total:.2f} % of it")
        diff = np.abs(res["tf32"]["last"].astype(np.int32) - res["fp16"]["last"].astype(np.int32))
        say()
        say(f"tf32 / fp16 frame time: {res['tf32']['ms_per_frame'] / res['fp16']['ms_per_frame']:.2f}x; last frame tf32 vs fp16: "
            f"max |diff| {int(diff.max())} LSB, {100 * (diff <= 1).mean():.3f} % within +-1")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
