"""bench.py --dump-outputs: the writer keeps float64 as float64, stores everything else as float32, and refuses a dump
over its size limit before writing anything."""
import os

import numpy as np
import pytest

import bench


def test_write_dump_dtypes_and_names(tmp_path):
    d = str(tmp_path / "out")
    bench.write_dump(d, {"a": np.arange(6, dtype=np.float64).reshape(2, 3), "m": np.array([3, -2], np.int32),
                         "h": np.ones(4, np.float16)})
    assert sorted(os.listdir(d)) == ["a.npy", "h.npy", "m.npy"]
    a, m, h = (np.load(os.path.join(d, n + ".npy")) for n in ("a", "m", "h"))
    assert a.dtype == np.float64 and a.shape == (2, 3) and a[1, 2] == 5.0
    assert m.dtype == np.float32 and m.tolist() == [3.0, -2.0]
    assert h.dtype == np.float32 and h.tolist() == [1.0] * 4


def test_write_dump_refuses_oversized_output(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 16)
    with pytest.raises(AssertionError):
        bench.write_dump(str(tmp_path / "out"), {"x": np.zeros(5, np.float32)})
    assert not os.path.exists(tmp_path / "out")


def _run_bench(out_dir, *args):
    import json
    import subprocess
    import sys
    cmd = [sys.executable, os.path.join(bench.ROOT, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "1",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir)] + list(args)
    r = subprocess.run(cmd, cwd=bench.ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_dump_outputs_end_to_end(tmp_path):
    """bench.py --dump-outputs on the B200: the training run dumps the 4 metrics its last timed step returned, the
    inference run the float64 patch_wise_prediction of the 256x256x64 volume - bit-identical in a second run with the
    same arguments - and every record times exactly --steps iterations."""
    line = _run_bench(tmp_path / "train", "--workload", "train")
    assert line["steps"] == 1
    assert sorted(os.listdir(tmp_path / "train")) == ["train_metrics.npy"]
    m = np.load(tmp_path / "train" / "train_metrics.npy")
    assert m.dtype == np.float32 and m.shape == (4,) and np.isfinite(m).all()
    assert m[0] == -m[3] and 0.0 <= m[1] <= 1.0            # soft-Dice loss = -dice; binary accuracy
    runs = []
    for k in range(2):
        line = _run_bench(tmp_path / ("infer%d" % k), "--workload", "infer")
        assert line["steps"] == 1
        assert sorted(os.listdir(tmp_path / ("infer%d" % k))) == ["infer_prediction.npy"]
        runs.append(np.load(tmp_path / ("infer%d" % k) / "infer_prediction.npy"))
    p = runs[0]
    assert p.dtype == np.float64 and p.shape == (256, 256, 64, 1)
    assert np.isfinite(p).all() and p.min() >= 0.0 and p.max() <= 1.0
    assert np.array_equal(runs[0], runs[1])
