"""bench.py's JSON contract, as far as it can be exercised without a GPU: the reference arm (the CPU
restatement on the host cores) prints ONE line with every key the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import bits_equal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=600, cwd=ROOT)


def synth_inputs(grid):
    """bench.synth_inputs() at grid x grid: pressure and divergence from seed 42."""
    rng = np.random.default_rng(42)
    d = rng.uniform(-1, 1, (grid, grid)).astype(np.float32)
    return rng.standard_normal((grid, grid)).astype(np.float32), d


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--grid", "512", "--iters", "50"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    want = json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    assert d["impl"] == "reference" and d["metric"] == want and d["unit"] == "cell-updates/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "f32"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["gpu_launches"] == 0


def test_gpu_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU path" in (out.stderr + out.stdout)


@pytest.mark.parametrize("grid,sampled", [(512, False), (4096, True)])
def test_reference_arm_dumps_its_last_timed_step(oracle, tmp_path, grid, sampled):
    """--dump-outputs on the CPU arm: 3 warm-up steps of 2 sweeps and 2 timed steps of 10 sweeps leave the
    oracle's 26 sweeps of the seeded inputs; a 4096^2 field is over the budget and cut to seeded rows."""
    out = bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--grid", str(grid),
                "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    p, d = synth_inputs(grid)
    want = oracle.jacobi(p, d, 2 * 3 + 10 * 2)
    got = np.load(tmp_path / "pressure.npy")
    assert got.dtype == np.float32
    if sampled:
        rows = np.load(tmp_path / "pressure_rows.npy")
        assert rows.dtype == np.float64 and np.all(np.diff(rows) > 0) and got.nbytes <= 32 << 20
        want = want[rows.astype(np.int64)]
    else:
        assert not (tmp_path / "pressure_rows.npy").exists()
    assert bits_equal(got, want)


def test_steps_below_one_are_refused():
    out = bench("--impl", "reference", "--steps", "0", "--grid", "512")
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_timed_step(oracle, tmp_path):
    """--dump-outputs on the timed path: 3 warm-up and 4 timed solves (each clear + 50 Jacobi sweeps), so the
    dump is the oracle's 7th solve of the seeded inputs, bit for bit."""
    out = bench("--steps", "4", "--warmup", "3", "--grid", "512", "--iters", "50", "--quick",
                "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])["steps"] == 4
    p, d = synth_inputs(512)
    for _ in range(3 + 4):
        p = oracle.jacobi(oracle.clear(p, 0.8), d, 50)
    assert bits_equal(np.load(tmp_path / "pressure.npy"), p)
