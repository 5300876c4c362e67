"""bench.py --dump-outputs: float32 row samples at fixed, seeded rows, within 64 MB for all three workloads together; on the GPU,
the dumps are the last timed frame of every workload and --steps sets every timed loop."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench


def _out_shape(wl):
    return (bench.FRAME_H * wl["scale"], bench.FRAME_W * wl["scale"], 3)


def test_dump_outputs_format_size_and_rows(tmp_path):
    rng = np.random.default_rng(5)
    outputs = {k: rng.integers(0, 256, size=_out_shape(wl), dtype=np.uint8) for k, wl in bench.WORKLOADS.items()}
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), outputs)
    bench.dump_outputs(str(b), outputs)
    total = 0
    for key, frame in outputs.items():
        got = np.load(a / f"{key}.npy")
        rows = np.load(a / f"{key}_rows.npy")
        assert got.dtype == np.float32 and rows.dtype == np.float64
        assert got.shape == (bench.DUMP_ROWS, frame.shape[1], 3)
        idx = rows.astype(np.int64)
        assert np.array_equal(idx, rows) and np.all(np.diff(idx) > 0) and idx[-1] < frame.shape[0]
        assert np.array_equal(got, frame[idx].astype(np.float32))
        assert np.array_equal(np.load(b / f"{key}.npy"), got) and np.array_equal(np.load(b / f"{key}_rows.npy"), rows)
        total += os.path.getsize(a / f"{key}.npy") + os.path.getsize(a / f"{key}_rows.npy")
    assert total <= 64 << 20


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_frame_of_every_workload(tmp_path, built_lib):
    import __graft_entry__
    import w2x
    from oracle import tiling
    steps, out = 3, tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(os.path.dirname(os.path.abspath(bench.__file__)), "bench.py"), "--gpus", "1",
                        "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["e2e_sync"]["steps"] == steps
    assert sorted(line["workloads"]) == sorted(k for k in bench.WORKLOADS if k != "cunet")
    for key, x in line["workloads"].items():
        assert x["steps"] == steps and x["e2e_sync"]["steps"] == steps, key
    # the device-resident loop renders input frame i % 4 at step i; rank 0's frame s is synthetic_frame(seed s)
    src = tiling.synthetic_frame(bench.FRAME_W, bench.FRAME_H, (steps - 1) % 4)
    for key, wl in bench.WORKLOADS.items():
        _, onnx = __graft_entry__.make_synthetic_model(str(tmp_path / key), scale=wl["scale"], noise=wl["noise"], model=wl["model"])
        eng = w2x.Img2Img()
        assert eng.build(onnx, w2x.BuildConfig.fixed(wl["batch"], wl["tile"]))
        assert eng.load(onnx, w2x.RenderConfig(batchSize=wl["batch"], height=wl["tile"], width=wl["tile"], scaling=wl["scale"],
                                               overlap=(bench.BLEND, bench.BLEND), tta=wl["tta"]))
        want = eng.render(src)
        eng.close()
        assert want is not None and want.shape == _out_shape(wl), key
        rows = np.load(out / f"{key}_rows.npy").astype(np.int64)
        assert np.array_equal(np.load(out / f"{key}.npy"), want[rows].astype(np.float32)), key
