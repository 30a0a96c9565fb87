"""bench.py contract checks that need no GPU: the CPU reference arm prints one JSON line with the
keys the driver reads (impl, metric, unit, value, cpu_baseline, e2e ...)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, B200_REF_SECONDS="0.5")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=600, check=True)
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "MS/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["scaling"] == "weak" and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, env=env, timeout=120)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_dump_outputs_writes_a_fixed_bounded_sample(tmp_path):
    """--dump-outputs: whole outputs while they fit the budget, then the same seeded rows on every run."""
    import importlib.util

    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    small = torch.arange(6 * 4, dtype=torch.float32).view(6, 4)
    big = torch.arange(50 * 10, dtype=torch.float32).view(50, 10)
    for run in ("a", "b"):
        got = bench.dump_outputs(str(tmp_path / run), [("small", small), ("big", big)], budget=6 * 16 + 12 * 40)
        assert got == {"small": 6, "big": 12}
    a_small, a_big = (np.load(tmp_path / "a" / f"{n}.npy") for n in ("small", "big"))
    assert a_small.dtype == a_big.dtype == np.float32 and np.array_equal(a_small, small.numpy())
    rows = a_big[:, 0].astype(int) // 10
    assert a_big.shape == (12, 10) and list(rows) == sorted(set(rows)) and np.array_equal(a_big, big.numpy()[rows])
    assert np.array_equal(a_big, np.load(tmp_path / "b" / "big.npy"))
    assert bench.DUMP_BYTES <= 64_000_000
