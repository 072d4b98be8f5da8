"""bench.py contract: on a machine without a GPU the reference arm prints one JSON line with the required keys, and the GPU arm
refuses to run without a device (no CPU fallback); on the B200, --dump-outputs writes what the timed path computed."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMP_GOLDEN = os.path.join(ROOT, "tests", "golden", "bench_dump_log2n12.json")


def test_reference_arm_json_line():
    env = dict(os.environ, PG_BENCH_CPU_BUDGET_S="0.5")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=300)
    assert res.returncode == 0, res.stderr
    line = json.loads(res.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "port" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and line["vs_baseline"] is None


def test_gpu_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert res.returncode != 0 and "no CPU path" in (res.stderr + res.stdout)


def _digest(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.gpu
def test_dump_outputs_are_the_recorded_ones(tmp_path, oracle):
    """--dump-outputs at a batch of 2^12: float arrays within 64 MiB, the in-range (even) instances give 1 and the others 0, the
    verdict is "satisfied", and every array equals, byte for byte, what this benchmark wrote when the digests in
    tests/golden/bench_dump_log2n12.json were recorded."""
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--log2n", "12", "--steps", "2", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == 2
    got = {f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)}
    with open(DUMP_GOLDEN) as f:
        golden = json.load(f)
    assert set(got) == set(golden)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    idx = got["range_check_results_index"]
    assert (idx == np.arange(1 << 12)).all()
    one = oracle.from_ints([1]).view(np.uint32).astype(np.float64)
    results = got["range_check_results"]
    assert (results[0::2] == one).all() and (results[1::2] == 0).all()
    assert got["verdict"].tolist() == [0, -1]
    assert got["variables"].shape == (256, 653, 8)
    for name, a in got.items():
        assert [list(a.shape), _digest(a)] == golden[name], name
