"""Policy evaluation on the device (EmbodiedRunner.evaluate) against EvalRunnerOracle.evaluate, which
tests/test_oracle_eval.py pins to executed reference code (golden_r7.npz)."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_oracle_eval import eval_case

pytestmark = pytest.mark.gpu

SHAPES = [(1000, 128, 8), (1000, 10, 8)]  # fp16-split GEMMs with a partial last tile; SIMT first layer (frankasim-like)


def _runner(cfg, params):
    from rlinf_b200.runner import EmbodiedRunner

    r = EmbodiedRunner(cfg)
    r.actor.model.load_state_dict({k: v.detach() for k, v in params.items()})
    return r


def _check(metrics, eps, o_metrics, o_eps):
    assert sorted(metrics) == sorted(o_metrics)
    assert metrics["num_trajectories"] == o_metrics["num_trajectories"]
    assert sorted(eps) == sorted(o_eps)
    for k in ("episode_len", "success_once", "success_at_end"):
        if k in o_eps:
            assert torch.equal(eps[k], o_eps[k]), k
    for k in ("return", "reward"):
        torch.testing.assert_close(eps[k], o_eps[k], rtol=1e-4, atol=1e-5, msg=k)
    for k, v in o_metrics.items():
        assert abs(metrics[k] - v) <= 1e-4 * max(1.0, abs(v)), (k, metrics[k], v)


def test_mean_bit_identical_to_training_head():
    from rlinf_b200 import _lib as L
    from rlinf_b200.policy import MLPPolicy

    for obs, act in ((128, 8), (10, 8)):
        pol = MLPPolicy(obs, act, seed=3)
        with torch.no_grad():
            pol.flat_params.add_(0.01 * torch.randn(pol.flat_params.shape, device=pol.device))
        pol.mark_params_changed()
        n = 1000
        states = torch.randn(n, obs, device=pol.device)
        pol.forward_train(states, torch.zeros(n, act, device=pol.device))
        acts = pol._last[4]
        want = acts[6 * n * 256: 6 * n * 256 + n * act].view(n, act).clone()
        lib = L.load()
        mean = torch.empty(n, act, device=pol.device)
        work = torch.empty(int(lib.rb200_mlp_fwd_scratch_floats(C.byref(pol.layout), n)), device=pol.device)
        L.check(lib.rb200_mlp_mean(C.byref(pol.layout), L.ptr(pol.flat_params), pol._ws(), L.ptr(states), n,
                                   L.ptr(mean), L.ptr(work), L.stream_ptr()), "mlp_mean")
        assert torch.equal(mean, want), (obs, (mean - want).abs().max().item())


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("case", ["ar_ign", "ar_term", "noreset", "chunk2"])
def test_evaluate_matches_oracle(golden, case, shape):
    from oracle.eval_oracle import EvalRunnerOracle

    cfg, params, noise, init = eval_case(golden("r7"), case, *shape)
    o_metrics, o_eps = EvalRunnerOracle(cfg, params=params).evaluate(noise, init)
    r = _runner(cfg, params)
    for _ in range(3):  # eager, graph capture + replay, replay
        metrics, eps = r.evaluate(return_episodes=True, env_noise=noise.cuda(), init_states=init.cuda())
        _check(metrics, eps, o_metrics, o_eps)
    assert r.eval_worker.graph_kernel_count > 0


def test_evaluate_repeatable_with_device_noise(golden):
    cfg, params, _, _ = eval_case(golden("r7"), "ar_ign", 1000, 128, 8)
    cfg["env"]["eval"]["max_steps_per_rollout_epoch"] = 40
    cfg["env"]["eval"]["max_episode_steps"] = 16
    r = _runner(cfg, params)
    runs = [r.evaluate(return_episodes=True) for _ in range(3)]  # eager, captured, replayed
    assert runs[0][0]["num_trajectories"] > 0
    for m, e in runs[1:]:
        assert m == runs[0][0]
        for k in e:
            assert torch.equal(e[k], runs[0][1][k]), k


def test_evaluation_does_not_disturb_training():
    from rlinf_b200.config import synthetic_ppo_config

    def run(with_eval):
        cfg = synthetic_ppo_config(B=256, T=16, obs_dim=128, action_dim=8, update_epoch=1, num_minibatches=2,
                                   seed=7, **{"runner.max_epochs": 3})
        cfg["env"]["eval"] = {"total_num_envs": 64, "max_steps_per_rollout_epoch": 24, "max_episode_steps": 10,
                              "auto_reset": True, "ignore_terminations": True, "rollout_epoch": 1}
        if with_eval:
            cfg["runner"]["val_check_interval"] = 1
        from rlinf_b200.runner import EmbodiedRunner

        r = EmbodiedRunner(cfg)
        out = r.run(3)
        return out, r.actor.model.flat_params.clone()

    m0, p0 = run(False)
    m1, p1 = run(True)
    assert torch.equal(p0, p1)
    for a, b in zip(m0, m1):
        assert any(k.startswith("eval/") for k in b)
        assert not any(k.startswith("eval/") for k in a)
        np.testing.assert_equal({k: v for k, v in b.items() if not k.startswith("eval/")}, a)  # NaN == NaN here


def test_evaluate_sees_fresh_weights_after_update(golden):
    from oracle.eval_oracle import EvalRunnerOracle

    cfg, params, noise, init = eval_case(golden("r7"), "ar_term", 1000, 128, 8)
    cfg["env"]["train"]["total_num_envs"] = 256
    cfg["actor"]["global_batch_size"] = cfg["actor"]["micro_batch_size"] = 256 * 10 // 2
    r = _runner(cfg, params)
    for _ in range(2):  # eager, then the captured graph
        _, before = r.evaluate(return_episodes=True, env_noise=noise.cuda(), init_states=init.cuda())
    r.run_iteration()
    r.update_rollout_weights()
    metrics, eps = r.evaluate(return_episodes=True, env_noise=noise.cuda(), init_states=init.cuda())
    new = {k: v.detach().cpu().clone() for k, v in r.actor.model.named_parameters()}
    assert any(not torch.equal(new[k], params[k]) for k in params)
    o_metrics, o_eps = EvalRunnerOracle(cfg, params=new).evaluate(noise, init)
    _check(metrics, eps, o_metrics, o_eps)
    assert not torch.equal(eps["return"], before["return"])  # the replay read the updated weights


def test_two_rank_evaluate_matches_oracle(tmp_path):
    import json
    import os
    import socket
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    env = dict(os.environ, RB200_DIST_OUT=str(tmp_path / "out.json"))
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "dist_eval_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), worker], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    res = json.loads((tmp_path / "out.json").read_text())
    assert res["ok"], res
