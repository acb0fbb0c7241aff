"""CPU-only: the reference arm of bench.py (the one leg that runs without a GPU) prints one JSON line with the
keys the driver reads, on a bounded sample."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


@pytest.mark.parametrize("workload", ["c2", "c4"])
def test_reference_arm_json(workload):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload,
                          "--steps", "1", "--warmup", "0", "--ref-seconds", "0.3", "--sweeps", "4"],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert KEYS <= set(line), KEYS - set(line)
    assert line["impl"] == "reference" and line["metric"] == "spin-updates/sec" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["vs_baseline"] is None
    assert "workload" in line["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def test_tensor_roofline_denominator_follows_the_timed_region():
    """MEASURED_PEAKS.json holds a burst and a sustained cuBLAS bf16 rate; bench.py divides by the burst rate for a short
    timed region and by the sustained rate for regions of 2 s and more, and always reports both fractions."""
    b = _bench_module()
    pk = {"tc_burst": 1617.1, "tc_sustained": 1355.9, "src": "test"}
    p_short, s_short = b.tensor_peak(pk, 0.4)
    p_long, s_long = b.tensor_peak(pk, 2.5)
    assert p_short == 1617.1 and "BURST" in s_short
    assert p_long == 1355.9 and "SUSTAINED" in s_long


def test_dump_outputs_types_budget_and_sample(tmp_path):
    """--dump-outputs writes spins as float32 and counts as float64; at most 64 MB in all, every array keeping the same
    seeded sample of replicas, so two runs (or two builds) write identical files for identical results."""
    import numpy as np
    b = _bench_module()
    rng = np.random.default_rng(1)
    small = {"spins": rng.choice(np.array([-1, 1], dtype=np.int8), (64, 32)), "flips": rng.integers(0, 10**6, 64)}
    b.dump_outputs(str(tmp_path / "small"), small)
    s, f = np.load(tmp_path / "small" / "spins.npy"), np.load(tmp_path / "small" / "flips.npy")
    assert s.dtype == np.float32 and f.dtype == np.float64
    assert np.array_equal(s, small["spins"]) and np.array_equal(f, small["flips"])

    R, n = 8192, 4096                      # the C3 shape: 2 x 128 MiB as float32
    big = {"spins": np.repeat(np.arange(R, dtype=np.int64)[:, None] % 2 * 2 - 1, n, 1).astype(np.int8),
           "hidden": np.ones((R, n), dtype=np.int8), "flips": np.arange(R)}
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), big)
    total = sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in big)
    assert total <= 64 * 10**6
    fa, fb = np.load(tmp_path / "a" / "flips.npy"), np.load(tmp_path / "b" / "flips.npy")
    assert np.array_equal(fa, fb) and np.all(np.diff(fa) > 0) and 1000 < fa.size < R
    keep = fa.astype(np.int64)              # flips[r] == r: the kept replica ids, the same rows in every array
    assert np.array_equal(np.load(tmp_path / "a" / "spins.npy"), big["spins"][keep].astype(np.float32))
