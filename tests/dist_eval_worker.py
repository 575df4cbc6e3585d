"""2-rank evaluation worker (launched by tests/test_gpu_eval.py::test_two_rank_evaluate_matches_oracle with torchrun).

Each rank evaluates its half of the eval envs with injected noise; the ranks' metric sums meet in one all-reduce.  Every
rank replays both halves with the CPU oracle and compares the device metrics with compute_evaluate_metrics over the
concatenated episodes of both ranks."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from oracle.eval_oracle import EvalRunnerOracle, compute_evaluate_metrics
    from rlinf_b200.runner import EmbodiedRunner
    from test_oracle_eval import eval_case

    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_r7.npz"))
    cfg, params, noise, init = eval_case(g, "ar_term", 64, 128, 8)
    cfg["env"]["train"]["total_num_envs"] = 64
    per = 64 // world
    cfg["actor"]["micro_batch_size"] = cfg["actor"]["global_batch_size"] // world
    r = EmbodiedRunner(cfg)
    r.actor.model.load_state_dict({k: v.detach() for k, v in params.items()})
    sl = slice(rank * per, (rank + 1) * per)
    out = {}
    for _ in range(2):  # eager, then the captured graph
        out = r.evaluate(env_noise=noise[:, sl].contiguous().cuda(), init_states=init[:, sl].contiguous().cuda())
    eps = []
    for q in range(world):
        s = slice(q * per, (q + 1) * per)
        _, e = EvalRunnerOracle(cfg, params=params).evaluate(noise[:, s], init[:, s], num_envs=per)
        eps.append(e)
    want = compute_evaluate_metrics(eps)
    ok = sorted(out) == sorted(want) and out["num_trajectories"] == want["num_trajectories"] and all(
        abs(out[k] - v) <= 1e-4 * max(1.0, abs(v)) for k, v in want.items())
    if rank == 0:
        with open(os.environ["RB200_DIST_OUT"], "w") as fh:
            json.dump({"ok": bool(ok), "device": out, "oracle": want}, fh)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
