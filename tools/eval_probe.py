"""Cost of one EmbodiedRunner.evaluate (CUDA-graph replay) beside a training rollout_phase at the same shape.

    python tools/eval_probe.py [--out RESULTS.json]

Shapes: B = 4096 envs, T = 512 steps, obs 128, act 8 (the benchmark's configuration), and the example eval size of
examples/embodiment/config/maniskill_ppo_mlp.yaml (32 envs, 50 steps).  Per shape: ms per evaluate (host clock around
the call, which ends in its one device-to-host read), us per chunk step, kernels per chunk step (rb200_launch_count
while the graph was captured), and ms per training rollout_phase (CUDA events, the production rollout kernel).  The
card's name, power limit and SM clock are printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rlinf_b200.config import synthetic_ppo_config  # noqa: E402
from rlinf_b200.runner import EmbodiedRunner  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                               "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def probe(B, T, reps):
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=128, action_dim=8)
    cfg["env"]["eval"] = {"total_num_envs": B, "max_steps_per_rollout_epoch": T, "max_episode_steps": max(T // 4, 1),
                          "auto_reset": True, "ignore_terminations": True, "rollout_epoch": 1}
    r = EmbodiedRunner(cfg)
    for _ in range(3):  # eager, capture + replay, replay
        m = r.evaluate()
    torch.cuda.synchronize()
    ev = []
    for _ in range(reps):
        t0 = time.perf_counter()
        m = r.evaluate()
        ev.append((time.perf_counter() - t0) * 1e3)
    for _ in range(2):
        r.rollout_phase()
    torch.cuda.synchronize()
    ro = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r.rollout_phase()
        e1.record()
        torch.cuda.synchronize()
        ro.append(e0.elapsed_time(e1))
    w = r.eval_worker
    steps = w.epochs * w.n_chunk_steps
    ev.sort()
    ro.sort()
    return {"B": B, "T": T, "eval_ms_median": ev[len(ev) // 2], "eval_ms_min": ev[0],
            "eval_us_per_chunk_step": ev[len(ev) // 2] * 1e3 / steps,
            "eval_launches_per_chunk_step": w.graph_kernel_count / steps, "eval_graph_launches": w.graph_kernel_count,
            "rollout_phase_ms_median": ro[len(ro) // 2], "rollout_phase_ms_min": ro[0],
            "rollout_impl": "tc" if r.rollout._tc else ("fused" if r.rollout._fused else "graph"),
            "eval_metrics": m}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    res = {"gpu": gpu_info(), "shapes": [probe(4096, 512, a.reps), probe(32, 50, a.reps)], "gpu_after": gpu_info()}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
