"""CPU: the reference arm of bench.py (the reference's own modules compiled into oracle/_ref, else the oracle port, on
the host cores) prints one JSON line with the contract's keys; the b200 arm refuses to run without a CUDA device (no CPU
fallback)."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--nodes", "96",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
                "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    from baseline import ref_arm
    have_ref = ref_arm.available()
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert line["cpu_baseline"]["nproc"] >= line["cpu_baseline"]["cores"] >= 1
    assert set(line["config"]) == {"workload", "parallelism", "l2", "superpoints", "embedded_superpoints",
                                   "points", "edges"}
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0
    assert line["config"]["superpoints"] == 96
    assert line["config"]["workload"].startswith("configs[1]")  # same workload string as the b200 arm
    r, c = line["rates"], line["config"]
    assert abs(r["points_per_s"] + r["edges_per_s"] - line["value"]) <= 1e-6 * line["value"]
    assert abs(r["edge_iterations_per_s"] - 10 * r["edges_per_s"]) <= 1e-9 * r["edge_iterations_per_s"]
    assert abs(r["superpoints_per_s"] * c["points"] - r["points_per_s"] * c["superpoints"]) \
        <= 1e-6 * r["points_per_s"] * c["superpoints"]


def test_dump_outputs_float_arrays_within_budget(tmp_path):
    """--dump-outputs: float32/float64 .npy files; past the byte budget the logits keep a fixed seeded row sample."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(1)
    small = {"logits": rng.standard_normal((100, 13)).astype(np.float32), "loss": np.ones(1, np.float32)}
    bench.dump_outputs(str(tmp_path / "small"), small)
    assert sorted(os.listdir(tmp_path / "small")) == ["logits.npy", "loss.npy"]
    assert np.array_equal(np.load(tmp_path / "small" / "logits.npy"), small["logits"])
    big = {"logits": rng.standard_normal((50000, 13)).astype(np.float32), "loss": np.ones(1, np.float32)}
    for d in ("big1", "big2"):
        bench.dump_outputs(str(tmp_path / d), big, budget=10 ** 6)
        files = sorted(os.listdir(tmp_path / d))
        assert files == ["logits.npy", "logits_rows.npy", "loss.npy"]
        assert sum(os.path.getsize(tmp_path / d / f) for f in files) <= 10 ** 6
        got = {f: np.load(tmp_path / d / f) for f in files}
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        assert np.array_equal(got["logits.npy"], big["logits"][got["logits_rows.npy"].astype(np.int64)])
    assert np.array_equal(np.load(tmp_path / "big1" / "logits_rows.npy"), np.load(tmp_path / "big2" / "logits_rows.npy"))


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=300)
    assert out.returncode != 0 and "--steps must be >= 1" in out.stderr


def test_b200_arm_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
