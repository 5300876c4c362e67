"""bench_resize.py -- cost of resized output (w2x_render_resized / w2x_submit_resized) on cfg2 (cunet/art 2x, tile 256, batch 8) and cfg4
(swin_unet/art 4x, tile 256, batch 4), 1920x1080 input frames, in one process on one GPU.

Per workload, output scales F (the first is the model's scale: plain w2x_render / w2x_submit; the others resample the canvas to
lround(1920 F) x lround(1080 F)):
  sync     w2x_render (F = scale) or w2x_render_resized, pageable host buffers, wall clock around each synchronous call; the output scales
           alternate frame by frame.  Also the median w2x_last_stage_ms stage 2 (stitch, plus the resample when resized).
  submit   w2x_submit / w2x_submit_resized on pinned buffers, three frames in flight; ms/frame = the interval between consecutive completed
           waits in steady state (the first three completions of each chunk of 11 frames are not counted); the output scales alternate
           chunk by chunk.
Then, in a separate profiled pass (torch.profiler, CUDA activities), the device time of the two resample kernels (resample_h_kernel,
resample_v_kernel) per frame, and their algorithmic bytes (canvas read + output write) over that time as a share of 7.7 TB/s.  The
kernels also write and read an fp32 intermediate (canvas rows x output columns x 3 x 4 bytes), listed beside it.  The card's name, power
limit and max SM clock are read with nvidia-smi in the same run.

    python scripts/bench_resize.py [--steps 32] [--warmup 3] [--out profiles/r05_resize.txt]
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
HBM_TBPS = 7.7
WORKLOADS = {
    "cfg2": dict(model="cunet/art", scale=2, tile=256, batch=8, factors=(2, 1.5, 1.0)),
    "cfg4": dict(model="swin_unet/art", scale=4, tile=256, batch=4, factors=(4, 3, 2)),
}
CHUNK, FILL = 11, 3


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "nvidia-smi unavailable"


def out_size(f):
    return max(1, round(FRAME_W * f)), max(1, round(FRAME_H * f))


def run(wl, steps, warmup, path, say):
    import torch
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
    src = tiling.synthetic_frame(FRAME_W, FRAME_H, 1)
    factors = wl["factors"]
    sizes = {f: out_size(f) for f in factors}
    outs = {f: np.empty((sizes[f][1], sizes[f][0], 3), np.uint8) for f in factors}

    def sync(f):
        if f == s:
            return eng.render_into(src, outs[f])
        return eng.render_resized(src, sizes[f], outs[f]) is not None

    # sync path, output scales alternating frame by frame
    ms = {f: [] for f in factors}
    st2 = {f: [] for f in factors}
    for i in range(warmup + steps):
        for f in factors:
            t0 = time.perf_counter()
            assert sync(f), eng.last_error
            dt = (time.perf_counter() - t0) * 1e3
            if i >= warmup:
                ms[f].append(dt)
                st2[f].append(eng.last_stage_ms()["stitch"])
    # the resized frames equal the resample of the full canvas (the same kernels, so byte for byte)
    full = eng.render(src)
    for f in factors[1:]:
        assert np.array_equal(eng.render_resized(src, sizes[f]), w2x.resample(full, sizes[f])), f

    # submit path: three frames in flight on pinned buffers, output scales alternating chunk by chunk
    pin_in = w2x.PinnedArray((FRAME_H, FRAME_W, 3))
    pin_in.array[...] = src
    pin_out = {f: [w2x.PinnedArray((sizes[f][1], sizes[f][0], 3)) for _ in range(3)] for f in factors}
    iv = {f: [] for f in factors}

    def chunk(f, record):
        tickets, done = [], []
        for k in range(CHUNK):
            if len(tickets) == 3:
                assert eng.wait(tickets.pop(0)), eng.last_error
                done.append(time.perf_counter())
            dst = pin_out[f][k % 3]
            t = (eng.submit(pin_in.ptr, FRAME_W, FRAME_H, dst.ptr) if f == s
                 else eng.submit_resized(pin_in.ptr, FRAME_W, FRAME_H, dst.ptr, sizes[f]))
            assert t >= 0, eng.last_error
            tickets.append(t)
        for t in tickets:
            assert eng.wait(t), eng.last_error
            done.append(time.perf_counter())
        if record:
            iv[f].extend(np.diff(done[FILL - 1:]) * 1e3)

    rounds = -(-steps // (CHUNK - FILL))
    for r in range(1 + rounds):
        for f in factors:
            chunk(f, r > 0)
    pin_in.free()
    for lst in pin_out.values():
        for p in lst:
            p.free()

    base = float(np.median(ms[s]))
    say(f"   {'F':>4s} {'output':>10s}   {'sync ms':>8s} {'Mpx/s':>8s} {'x F=' + str(s):>7s} {'stage2 ms':>9s}   {'submit ms':>9s} {'Mpx/s':>8s}  "
        f"(medians over {steps} sync frames and {len(iv[s])} submit intervals)")
    sbase = float(np.median(iv[s]))
    for f in factors:
        w, h = sizes[f]
        m, sm = float(np.median(ms[f])), float(np.median(iv[f]))
        say(f"   {f:4g} {f'{w}x{h}':>10s}   {m:8.2f} {w * h / 1e3 / m:8.1f} {m / base:7.3f} {float(np.median(st2[f])):9.3f}   {sm:9.2f} "
            f"{w * h / 1e3 / sm:8.1f}   submit x F={s}: {sm / sbase:.3f}")
    say(f"   sync ms/frame spread (p10..p90): " + ", ".join(f"F={f:g} {np.percentile(ms[f], 10):.2f}..{np.percentile(ms[f], 90):.2f}" for f in factors))

    # profiled pass: the resample kernels' own device time
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    reps = 8
    for f in factors[1:]:
        eng.render_resized(src, sizes[f], outs[f])
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                assert eng.render_resized(src, sizes[f], outs[f]) is not None, eng.last_error
        kern = {"resample_h_kernel": [0.0, 0], "resample_v_kernel": [0.0, 0]}
        total = 0.0
        for ev in prof.key_averages():
            t = float(getattr(ev, "device_time_total", 0.0) or 0.0)
            if not ev.key.startswith(("Memcpy", "Memset")):
                total += t
            for k in kern:
                if k in ev.key:
                    kern[k][0] += t
                    kern[k][1] += ev.count
        w, h = sizes[f]
        if kern["resample_v_kernel"][1] == 0:
            say(f"   F={f:g}: the profiler captured no resample kernel ({len(prof.key_averages())} kernels in the trace): not measured")
            continue
        us = (kern["resample_h_kernel"][0] + kern["resample_v_kernel"][0]) / reps
        cw, ch = FRAME_W * s, FRAME_H * s
        algo = cw * ch * 3 + w * h * 3
        tmp = 2 * ch * w * 3 * 4
        say(f"   F={f:g} profiled ({reps} frames): resample_h {kern['resample_h_kernel'][0] / reps:.1f} us + resample_v "
            f"{kern['resample_v_kernel'][0] / reps:.1f} us = {us:.1f} us/frame ({kern['resample_h_kernel'][1] // reps} + "
            f"{kern['resample_v_kernel'][1] // reps} launches), {100 * us / (total / reps):.2f} % of the frame's kernel time "
            f"({total / reps / 1e3:.2f} ms)")
        say(f"        canvas read + output write {algo / 1e6:.1f} MB -> {algo / (us * 1e-6) / 1e12:.2f} TB/s = "
            f"{100 * algo / (us * 1e-6) / (HBM_TBPS * 1e12):.1f} % of {HBM_TBPS} TB/s; with the fp32 intermediate (write + read, "
            f"{tmp / 1e6:.1f} MB) {(algo + tmp) / (us * 1e-6) / 1e12:.2f} TB/s")
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
    say(f"{FRAME_W}x{FRAME_H} input frames, blend {BLEND}, {args.steps} timed frames per path after {args.warmup} warm-up frames; "
        "Mpx/s counts output pixels")
    with tempfile.TemporaryDirectory() as d:
        for name, wl in WORKLOADS.items():
            _, path = __graft_entry__.make_synthetic_model(d, scale=wl["scale"], noise=0, model=wl["model"])
            say()
            say(f"== {name}: {wl['model']} {wl['scale']}x, tile {wl['tile']}, batch {wl['batch']}, canvas "
                f"{FRAME_W * wl['scale']}x{FRAME_H * wl['scale']}")
            run(wl, args.steps, args.warmup, path, say)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
