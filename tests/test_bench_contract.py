"""bench.py's contract with the driver, checked on the CPU: the reference arm (`--impl reference`: the oracle's arkworks-shaped
Pippenger on the host cores) prints ONE JSON line with the agreed keys, on the same `config` the GPU arm builds, and its
result passes its own self-check; under a multi-rank launch only rank 0 prints.  The GPU arm itself needs a B200 (its line
is exercised by the driver and by `profiles/r02_bench_*.json`)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=(), impl="reference"):
    env = dict(os.environ)
    env.pop("RANK", None), env.pop("WORLD_SIZE", None), env.pop("LOCAL_RANK", None)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--log-n", "12", "--steps", "2", "--warmup", "1", *args],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_prints_one_contract_line():
    sys.path.insert(0, ROOT)
    import bench

    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["config"] == bench.make_config(12, 1)  # the same workload description as the GPU arm's
    assert d["value"] > 0 and abs(d["value"] - (1 << 12) / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    assert d["self_check"] is True and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, ("--gpus", "2")) == []
    lines = _run({"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"}, ("--gpus", "2"))
    assert len(lines) == 1 and json.loads(lines[0])["n_gpus"] == 2


def test_bench_scalars_are_valid_montgomery_residues():
    sys.path.insert(0, ROOT)
    import bench

    a = bench.bench_scalars(1000, 3)
    assert a.shape == (1000, 4) and int(a[:, 3].max()) < (1 << 62)  # below 2^254 < r: every value is a residue
    assert (a == bench.bench_scalars(1000, 3)).all() and not (a == bench.bench_scalars(1000, 4)).all()


def test_reference_arm_dumps_the_result_of_its_last_step(tmp_path, oracle):
    sys.path.insert(0, ROOT)
    import bench

    assert len(_run(args=("--dump-outputs", str(tmp_path / "out")))) == 1
    assert os.listdir(tmp_path / "out") == ["msm_result.npy"]
    got = np.load(tmp_path / "out" / "msm_result.npy")
    assert got.dtype == np.float64 and got.shape == (2, 8) and (got == np.floor(got)).all() and got.max() < 2**32
    x, y = (sum(int(w) << (32 * i) for i, w in enumerate(row)) for row in got)
    n = 1 << 12
    assert (x, y) == oracle.pt_to_affine_ints(oracle.msm_affine(oracle.derive_points(2, n), bench.bench_scalars(n, 0)))


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


@pytest.mark.gpu
def test_gpu_arm_dumps_what_the_reference_arm_dumps(tmp_path):
    """Same arguments, same inputs: the GPU arm's last timed MSM and the reference arm's are the same point."""
    assert len(_run(args=("--dump-outputs", str(tmp_path / "ref")))) == 1
    quick = ("--no-cpu-baseline", "--no-secondary", "--no-strong", "--dump-outputs", str(tmp_path / "gpu"))
    lines = _run(args=quick, impl="ours")
    assert len(lines) == 1 and json.loads(lines[0])["oracle_match"] is True
    assert np.array_equal(np.load(tmp_path / "gpu" / "msm_result.npy"), np.load(tmp_path / "ref" / "msm_result.npy"))
