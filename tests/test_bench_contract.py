"""bench.py's JSON contract, exercised on the CPU through the reference arm, and the GPU arm's timed steps and output
dump (those need a B200)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-batch", "256"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _gpu_arm(dump_dir):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "20", "--warmup", "3", "--batch", "4096",
                          "--no-cpu", "--dump-outputs", str(dump_dir)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(dump_dir, f)) for f in os.listdir(dump_dir)}


@pytest.mark.gpu
def test_gpu_arm_times_exactly_the_given_steps_and_dumps_the_last_one(tmp_path):
    """--steps 20 is 20 timed steps (the library's step counter agrees), cut into sync-interval blocks of 8, 8 and 4;
    --dump-outputs writes the last timed step's per-env outputs and the weights as float32 / float64 .npy files, and a
    second run with the same arguments starts from the same inputs."""
    d, a = _gpu_arm(tmp_path / "a")
    tr = d["timed_region"]
    assert d["steps"] == 20 and tr["steps"] == 20 and tr["steps_run"] == 20 and tr["blocks"] == 3
    assert sorted(a) == ["action", "flags", "option", "reward", "state", "td_error", "weights"]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) == d["dump_outputs"]["bytes"] <= 64 * 10 ** 6
    assert a["state"].shape == (4096, 4) and a["weights"].shape == (4, 5, 256)
    assert set(np.unique(a["action"])) <= set(range(5)) and np.isfinite(a["td_error"]).all()
    _, b = _gpu_arm(tmp_path / "b")
    # the weight-delta sums use floating-point atomics: an env may only leave the other run's path at an arg-max near-tie
    assert (a["state"] == b["state"]).all(axis=1).mean() > 0.99
    assert np.abs(a["weights"] - b["weights"]).max() <= 1e-4 * np.abs(a["weights"]).max()


def test_gpu_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
