"""EvalRunnerOracle.evaluate (oracle/eval_oracle.py) against executed reference code (tests/golden/make_golden_r7.py):
EnvWorker.evaluate / env_evaluate_step, MultiStepRolloutWorker.evaluate, ManiskillEnv's episode bookkeeping, compute_evaluate_metrics and
check_progress.  Also the product's own check_progress / metrics_from_sums (host code) against the same goldens."""
import numpy as np
import pytest
import torch

from oracle import rl_oracle as O
from oracle.eval_oracle import EvalRunnerOracle
from rlinf_b200.config import synthetic_ppo_config
from rlinf_b200.evaluation import SUM_KEYS, check_progress, metrics_from_sums

CASES = ["ar_ign", "ar_term", "noreset", "chunk2", "none"]


def fixture_params(seed, obs_dim, act_dim, chunks):
    """Initial parameters of the r7 cases (same lines as make_golden_r5.fixture_params)."""
    p = O.mlp_init(obs_dim, act_dim, chunks, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    for n in p:
        if p[n].dim() == 1 or n == "actor_logstd":
            p[n] = p[n] + 0.05 * torch.randn(p[n].shape, generator=g)
    return {n: v.detach().clone() for n, v in p.items()}


def eval_case(g, name, B=None, obs=None, A=None):
    """(cfg, params, env_noise, init_states) of one r7 case.  B / obs / A override the fixture's shape (GPU tests reuse
    the case's flags and schedule at other shapes, with fresh noise)."""
    k = name + "_"
    fB, T, C, fobs, fA, auto_reset, ign, epochs, mes = (int(x) for x in g[k + "meta"])
    B, obs, A = B or fB, obs or fobs, A or fA
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=A, **{
        "actor.model.num_action_chunks": C, "env.train.seed": int(g[k + "sim_seed"]),
        "env.train.max_episode_steps": mes, "env.train.auto_reset": auto_reset})
    cfg["env"]["eval"] = {"total_num_envs": B, "max_steps_per_rollout_epoch": T, "max_episode_steps": mes,
                          "auto_reset": auto_reset, "ignore_terminations": ign, "rollout_epoch": epochs,
                          "p_term": float(g[k + "p_term"])}
    params = fixture_params(int(g[k + "param_seed"]), obs, A, C)
    if (B, obs, A) == (fB, fobs, fA):
        noise, init = torch.from_numpy(g[k + "env_noise"]), torch.from_numpy(g[k + "init_states"])
    else:
        gen = torch.Generator().manual_seed(int(g[k + "param_seed"]))
        R = epochs * (T // C)
        parts = []
        for _ in range(C):
            parts += [torch.randn(R, B, obs + 1, generator=gen), torch.rand(R, B, 1, generator=gen)]
        parts.append(torch.randn(R, B, obs, generator=gen))
        noise = torch.cat(parts, dim=-1)
        init = torch.randn(epochs if not auto_reset else 1, B, obs, generator=gen)
    return cfg, params, noise, init


@pytest.mark.parametrize("case", CASES)
def test_r7_evaluate_vs_reference_workers(golden, case):
    g = golden("r7")
    nt = torch.get_num_threads()
    torch.set_num_threads(1)  # the fixture was generated single-threaded: same init and GEMM blocking, same roundings
    try:
        cfg, params, noise, init = eval_case(g, case)
        metrics, eps = EvalRunnerOracle(cfg, params=params).evaluate(noise, init)
    finally:
        torch.set_num_threads(nt)
    k = case + "_"
    assert sorted(eps) == sorted(str(x) for x in g[k + "ep_keys"])
    for key in eps:
        want = torch.from_numpy(g[k + "ep_" + key])
        assert eps[key].dtype == want.dtype, key
        assert torch.equal(eps[key], want), key  # bit-exact per-episode records, reference order
    agg = dict(zip((str(x) for x in g[k + "agg_keys"]), g[k + "agg_vals"].tolist()))
    assert sorted(metrics) == sorted(agg)
    assert metrics["num_trajectories"] == agg["num_trajectories"]
    for key, v in agg.items():
        assert abs(metrics[key] - v) <= 1e-6 * max(1.0, abs(v)), key


@pytest.mark.parametrize("case", CASES)
def test_r7_metrics_from_sums_matches_reference_aggregation(golden, case):
    """The product's host-side aggregation of the fp64 sums (what rb200_eval_metrics returns) gives the reference's
    compute_evaluate_metrics dict."""
    g = golden("r7")
    k = case + "_"
    keys = [str(x) for x in g[k + "ep_keys"]]
    n = len(g[k + "ep_return"]) if "return" in keys else 0
    sums = [float(np.sum(g[k + "ep_" + key].astype(np.float64))) if key in keys else 0.0 for key in SUM_KEYS] + [n]
    got = metrics_from_sums(sums, bool(g[k + "meta"][6]))
    agg = dict(zip((str(x) for x in g[k + "agg_keys"]), g[k + "agg_vals"].tolist()))
    assert sorted(got) == sorted(agg)
    for key, v in agg.items():
        assert abs(got[key] - v) <= 1e-6 * max(1.0, abs(v)), key


def test_r7_check_progress_grid(golden):
    grid = golden("r7")["check_progress_grid"]
    for step, max_steps, vci, save, run_val, save_model, end in grid.tolist():
        assert check_progress(step, max_steps, vci, save, 1.0) == (bool(run_val), bool(save_model), bool(end))
