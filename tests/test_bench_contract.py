"""bench.py --impl reference (CPU arm) prints one JSON line with the contract's keys (CPU only, tiny sample); on a GPU,
--dump-outputs writes the last timed step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--T", "8", "--cpu-envs", "8", "--update-epoch", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["higher_is_better"] is True
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert "workload" in line["config"]


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    B, T, obs, act = 256, 16, 32, 2
    out_dir = tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--B", str(B), "--T", str(T), "--obs", str(obs),
                          "--act", str(act), "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-kernel-bench",
                          "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    arrays = {f.name[:-len(".npy")]: np.load(f) for f in out_dir.iterdir()}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert arrays["rollout.states"].shape == (T, B, obs) and arrays["rollout.prev_values"].shape == (T + 1, B, 1)
    assert arrays["train.advantages"].shape == (T * B, 1) and np.isfinite(arrays["train.returns"]).all()
    assert arrays["param.actor_logstd"].shape == (1, act)
    assert float(arrays["metric.actor.policy_loss"]) == line["train_metrics"]["actor/policy_loss"]
