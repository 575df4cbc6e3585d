"""GPU end-to-end parity: device rollout buffer alignment, synthetic env, and the PPO update
(shuffle -> micro-batches -> fused loss -> backward -> clip+AdamW) against the CPU oracle."""
import os

import numpy as np
import pytest
import torch

from oracle import rl_oracle as O
from oracle.runner_oracle import RunnerOracle, SyntheticEnvCPU

pytestmark = pytest.mark.gpu


def _cpu_batch(b):
    return {k: (_cpu_batch(v) if isinstance(v, dict) else v.detach().cpu().clone()) for k, v in b.items()}


def test_env_step_given_noise_matches_cpu():
    from rlinf_b200.envs import SyntheticVectorEnv

    B, obs, act = 300, 24, 3
    env = SyntheticVectorEnv(B, obs, act, max_episode_steps=5, p_term=0.2, seed=7)
    ref = SyntheticEnvCPU(B, obs, act, max_episode_steps=5, p_term=0.2, seed=7)
    assert torch.equal(env.w_s.cpu(), ref.w_s) and torch.equal(env.w_a.cpu(), ref.w_a)
    g = torch.Generator().manual_seed(0)
    state = torch.randn(B, obs, generator=g)
    env.state.copy_(state)
    ref.state = state.clone()
    for step in range(12):
        action = torch.randn(B, act, generator=g)
        noise = torch.cat([torch.randn(B, obs + 1, generator=g), torch.rand(B, 1, generator=g),
                           torch.randn(B, obs, generator=g)], 1)
        obs_l, r, te, tr, infos = env.chunk_step(action.cuda().view(B, 1, act), noise=noise.cuda())
        robs, rr, rte, rtr, rinf = ref.chunk_step(action.view(B, 1, act), noise)
        assert torch.equal(te.cpu(), rte) and torch.equal(tr.cpu(), rtr), step
        torch.testing.assert_close(r.cpu(), rr, rtol=1e-4, atol=1e-6)
        torch.testing.assert_close(obs_l[-1]["states"].cpu(), robs[-1]["states"], rtol=1e-4, atol=1e-6)
        torch.testing.assert_close(infos[-1]["final_observation"]["states"].cpu(),
                                   rinf[-1]["final_observation"]["states"], rtol=1e-4, atol=1e-6)
        # keep the two copies in lock-step (tanh differs by ulps between libm and CUDA)
        env.state.copy_(ref.state)
    assert (ref.elapsed == env.elapsed.cpu()).all()


@pytest.mark.parametrize("bootstrap_type", ["always", "standard"])
def test_rollout_buffer_alignment_vs_oracle(bootstrap_type):
    """Rows of the on-device [T(+1),B,...] buffer equal what the reference's trajectory builder would
    stack, for the same injected policy/env noise (incl. truncation bootstrap folded into rewards)."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    B, T, obs, act = 64, 24, 6, 2
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=act, **{"algorithm.bootstrap_type": bootstrap_type,
                                                                          "env.train.p_term": 0.05,
                                                                          "rollout.enable_cuda_graph": False})
    run = EmbodiedRunner(cfg)
    orc = RunnerOracle(cfg, params={n: p.detach().cpu().clone() for n, p in run.actor.model.named_parameters()})
    g = torch.Generator().manual_seed(3)
    pn = torch.randn(T + 1, B, act, generator=g)
    en = torch.cat([torch.randn(T, B, obs + 1, generator=g), torch.rand(T, B, 1, generator=g),
                    torch.randn(T, B, obs, generator=g)], -1)
    s0 = torch.randn(B, obs, generator=g)
    orc.env.state = s0.clone()
    orc.obs = {"states": orc.env.state}
    ob = orc.rollout(policy_noise=pn, env_noise=en)
    run.rollout.started = True
    run.buffer.states[0].copy_(s0)
    run.rollout._one_rollout(policy_noise=pn.cuda(), env_noise=en.cuda())
    b = _cpu_batch(run.buffer.as_batch())
    for k in ("dones", "terminations", "truncations"):
        assert torch.equal(b[k], ob[k]), k
    assert bool(ob["dones"].any()) and ob["dones"].shape == (T + 1, B, 1) and ob["rewards"].shape == (T, B, 1)
    for k in ("rewards", "prev_values", "prev_logprobs"):
        torch.testing.assert_close(b[k], ob[k], rtol=1e-4, atol=2e-5, msg=k)
    torch.testing.assert_close(b["forward_inputs"]["states"], ob["forward_inputs"]["states"], rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(b["forward_inputs"]["action"], ob["forward_inputs"]["action"], rtol=1e-4, atol=2e-5)


@pytest.mark.parametrize("bootstrap_type", ["always", "standard"])
def test_fused_rollout_kernel_vs_oracle(bootstrap_type):
    """The persistent fused rollout kernel (rb200_rollout_fused) fills the same buffer rows as the reference's
    loop for the same injected noise: flags bit-exact, floats within 1e-4."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    B, T, obs, act = 64, 24, 8, 2
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=act, **{"algorithm.bootstrap_type": bootstrap_type,
                                                                          "env.train.p_term": 0.05,
                                                                          "env.train.max_episode_steps": 10})
    run = EmbodiedRunner(cfg)
    assert run.rollout._fused
    orc = RunnerOracle(cfg, params={n: p.detach().cpu().clone() for n, p in run.actor.model.named_parameters()})
    g = torch.Generator().manual_seed(5)
    pn = torch.randn(T + 1, B, act, generator=g)
    en = torch.cat([torch.randn(T, B, obs + 1, generator=g), torch.rand(T, B, 1, generator=g),
                    torch.randn(T, B, obs, generator=g)], -1)
    s0 = torch.randn(B, obs, generator=g)
    orc.env.state = s0.clone()
    orc.obs = {"states": orc.env.state}
    ob = orc.rollout(policy_noise=pn, env_noise=en)
    run.rollout.started = True
    run.buffer.states[0].copy_(s0)
    run.rollout._one_rollout(policy_noise=pn[:T].cuda(), env_noise=en.cuda())
    b = _cpu_batch(run.buffer.as_batch())
    for k in ("dones", "terminations", "truncations"):
        assert torch.equal(b[k], ob[k]), k
    assert bool(ob["truncations"].any()) and bool(ob["terminations"].any())
    for k in ("rewards", "prev_values", "prev_logprobs"):
        torch.testing.assert_close(b[k], ob[k], rtol=1e-4, atol=2e-5, msg=k)
    torch.testing.assert_close(b["forward_inputs"]["states"], ob["forward_inputs"]["states"], rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(b["forward_inputs"]["action"], ob["forward_inputs"]["action"], rtol=1e-4, atol=2e-5)


@pytest.mark.parametrize("B", [300, 1000, 2000, 4096])
def test_fused_rollout_matches_per_kernel_path(B):
    """Device RNG: the fused kernel and the per-kernel CUDA-graph loop consume the same Philox streams, so two
    consecutive rollouts agree (flags exactly, floats up to fp32 summation order). Covers E = 3, 7, 14, 28
    environments per CTA (all four template instances)."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    T, obs, act = 6, 8, 3
    bufs = []
    for fused in (True, False):
        cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=act, **{"rollout.fused_kernel": fused,
                                                                              "env.train.p_term": 0.03,
                                                                              "env.train.max_episode_steps": 5,
                                                                              "algorithm.bootstrap_type": "always"})
        run = EmbodiedRunner(cfg)
        assert run.rollout._fused == fused
        out = []
        for _ in range(3):  # eager, graph capture, graph replay on the per-kernel path
            run.rollout_phase()
            torch.cuda.synchronize()
            out.append(_cpu_batch(run.buffer.as_batch()))
            out[-1]["elapsed"] = run.env.elapsed.cpu().clone()
        bufs.append(out)
    for r in range(3):
        a, b = bufs[0][r], bufs[1][r]
        for k in ("dones", "terminations", "truncations"):
            assert torch.equal(a[k], b[k]), (r, k)
        assert torch.equal(a["elapsed"], b["elapsed"]), r
        for k in ("rewards", "prev_values", "prev_logprobs"):
            torch.testing.assert_close(a[k], b[k], rtol=2e-3, atol=2e-4, msg=f"{r} {k}")
        torch.testing.assert_close(a["forward_inputs"]["states"], b["forward_inputs"]["states"], rtol=2e-3, atol=2e-4)
        torch.testing.assert_close(a["forward_inputs"]["action"], b["forward_inputs"]["action"], rtol=2e-3, atol=2e-4)
    assert bool(bufs[0][2]["dones"].any())


@pytest.mark.skipif(os.environ.get("RB200_EXPERIMENTAL", "0") != "1",
                    reason="experimental CUDA-graphed optimiser step: RB200_EXPERIMENTAL=1 to run")
@pytest.mark.parametrize("accum", [1, 2])
def test_experimental_graphed_update_matches_eager(accum):
    """actor.cuda_graph_update replays the same kernels: parameters after 3 iterations agree with the eager loop
    (atomics in the weight-gradient kernels make it allclose, not bit-equal)."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    B, T, obs, act = 256, 16, 8, 2
    n = B * T
    finals = []
    for graphed in (False, True):
        cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=act, update_epoch=2, num_minibatches=4,
                                   micro_batch_size=n // 4 // accum, **{"actor.cuda_graph_update": graphed})
        run = EmbodiedRunner(cfg)
        ms = [run.run_iteration() for _ in range(3)]
        torch.cuda.synchronize()
        finals.append((run.actor.model.flat_params.cpu().clone(), ms[-1]))
    torch.testing.assert_close(finals[0][0], finals[1][0], rtol=1e-4, atol=2e-5)
    for k, v in finals[0][1].items():
        if k != "critic/explained_variance" and np.isfinite(v):
            assert abs(v - finals[1][1][k]) <= 1e-3 * abs(v) + 1e-5, k


@pytest.mark.parametrize("accum", [1, 2])
def test_update_matches_oracle_after_k_steps(accum):
    """Same rollout batch -> advantages -> shuffled mini/micro-batches -> k optimiser steps: parameters,
    metrics within 1e-4 rel (fp32) of the oracle."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    B, T, obs, act = 64, 32, 4, 2  # BASELINE config 1
    n = B * T
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=act, update_epoch=2, num_minibatches=4,
                               micro_batch_size=n // 4 // accum)
    run = EmbodiedRunner(cfg)
    run.rollout_phase()
    torch.cuda.synchronize()
    batch = _cpu_batch(run.buffer.as_batch())
    orc = RunnerOracle(cfg, params={k: p.detach().cpu().clone() for k, p in run.actor.model.named_parameters()})
    om = orc.update(batch)
    m = run.update_phase()
    # Parameters after k = 8 optimiser steps. Adam's update lr*m/(sqrt(v)+eps) is sign-like for |g| >> eps and
    # amplifies ABSOLUTE gradient differences by lr/eps for |g| <~ eps = 1e-8: the fp16-split tensor-core GEMMs
    # (~2e-6 relative on each dot product) therefore move a few near-zero-gradient entries by up to ~1e-5 (0.4 % of
    # the 2.4e-3 total travel k*lr); everything else agrees to 1e-4 relative.
    worst = 0.0
    for name, p in run.actor.model.named_parameters():
        ref = orc.params[name].detach()
        torch.testing.assert_close(p.cpu(), ref, rtol=1e-4, atol=2e-5, msg=name)
        worst = max(worst, (p.cpu() - ref).abs().max().item())
        frac_tight = ((p.cpu() - ref).abs() <= 1e-4 * ref.abs() + 1e-6).float().mean().item()
        assert frac_tight > 0.99, (name, frac_tight)
    print("max |param - oracle| after 8 steps:", worst)
    for k, v in om.items():
        if k in ("critic/value_clip_ratio",):
            continue
        assert k in m, k
        np.testing.assert_allclose(m[k], v, rtol=2e-4, atol=1e-6, err_msg=k)
    assert run.actor.optimizer.state[0].item() == 8


def test_full_iterations_with_cuda_graph_rollout():
    """3 iterations (eager rollout, graph capture, graph replay): finite metrics, fresh noise per replay,
    value loss decreasing on the synthetic task."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    cfg = synthetic_ppo_config(B=256, T=16, obs_dim=8, action_dim=2, update_epoch=2, num_minibatches=2,
                               **{"rollout.fused_kernel": False})
    run = EmbodiedRunner(cfg)
    ms, acts = [], []
    for _ in range(3):
        ms.append(run.run_iteration())
        acts.append(run.buffer.actions.clone())
    assert all(np.isfinite(v) for m in ms for k, v in m.items() if k != "critic/explained_variance")
    assert not torch.equal(acts[1], acts[2])
    assert run.rollout._graph is not None


def test_host_batch_e2e_equals_device_batch():
    """recv_rollout_trajectories accepts HOST tensors (as the reference's channel delivers them)."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    cfg = synthetic_ppo_config(B=64, T=16, obs_dim=4, action_dim=2, update_epoch=1, num_minibatches=2)
    a, b = EmbodiedRunner(cfg), EmbodiedRunner(cfg)
    a.rollout_phase()
    torch.cuda.synchronize()
    host = _cpu_batch(a.buffer.as_batch())
    ma = a.update_phase()
    mb = b.update_phase(batch=host)
    # obs_dim 4 is not a multiple of 32: the first layer's weight gradient goes through the SIMT GEMM, whose per-split
    # partial sums are added with float atomics (order not deterministic): equal to rounding, not bitwise
    torch.testing.assert_close(a.actor.model.flat_params, b.actor.model.flat_params, rtol=1e-5, atol=1e-7)
    for k in ma:
        np.testing.assert_allclose(ma[k], mb[k], rtol=1e-4, atol=1e-7, err_msg=k)
