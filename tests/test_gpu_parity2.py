"""Round-2 GPU parity: branches of already-tested kernels that no test exercised in round 1 (entropy term, critic
warm-up, rollout_epoch merge, non-finite gradient skip), the fused rollout instances the multi-GPU runs use, the
config-2 shapes end to end (tcgen05 path), optimiser warm-up / LR schedules, and GRPO with auto_reset off."""
import os

import numpy as np
import pytest
import torch

from oracle import rl_oracle as O
from oracle.runner_oracle import RunnerOracle

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def _t(a):
    return torch.from_numpy(np.asarray(a))


def _cpu_batch(b):
    return {k: (_cpu_batch(v) if isinstance(v, dict) else v.detach().cpu().clone()) for k, v in b.items()}


# ---------------------------------------------------------------------------------------------------------------
# a17: entropy term, 1/accum, critic warm-up inside the fused loss kernel
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("warmup", [False, True])
def test_ppo_loss_entropy_bonus_and_critic_warmup(use_mask, warmup):
    """embodied_fsdp_actor_worker.py:678-699: loss -= entropy_bonus * masked_mean(reshape_entropy(entropy)) unless
    critic_warmup; loss /= grad_accum; actor/entropy_loss, actor/total_loss; gradients w.r.t. logprobs/values/entropy."""
    from rlinf_b200 import _lib as L
    from rlinf_b200 import ops

    n, A, accum, bonus = 3000, 8, 4, 0.01
    g = torch.Generator().manual_seed(11)
    old = -1 + 0.3 * torch.randn(n, A, generator=g)
    new = (old + 0.05 * torch.randn(n, A, generator=g)).requires_grad_(True)
    adv, ret, pv = (torch.randn(n, 1, generator=g) for _ in range(3))
    val = (pv + 0.1 * torch.randn(n, 1, generator=g)).requires_grad_(True)
    ent = (1.0 + 0.2 * torch.randn(n, A, generator=g)).requires_grad_(True)
    mask = (torch.rand(n, 1, generator=g) < 0.8) if use_mask else None
    hp = dict(clip_ratio_low=0.2, clip_ratio_high=0.25, value_clip=0.2, huber_delta=10.0)
    loss, metrics, d_lp, d_v, d_e = ops.ppo_loss(
        logprobs=new.detach().cuda(), values=val.detach().cuda(), entropy=ent.detach().cuda(), old_logprobs=old.cuda(),
        advantages=adv.cuda(), returns=ret.cuda(), prev_values=pv.cuda(), loss_mask=None if mask is None else mask.cuda(),
        C_chunks=1, A_dim=A, logprob_type="action_level", critic_warmup=warmup, entropy_bonus=bonus,
        loss_scale=1.0 / accum, **hp)
    oloss, om = O.policy_loss_embodied("actor_critic", new, old, adv, "action_level", A, loss_mask=mask, values=val,
                                       prev_values=pv, returns=ret, critic_warmup=warmup, **hp)
    ent_loss = torch.tensor(0.0)
    if not warmup:
        ent_loss = O.entropy_term(ent, "action_level", A, n, mask)
        oloss = oloss - bonus * ent_loss
    oloss = oloss / accum
    oloss.backward()
    torch.testing.assert_close(loss.cpu().reshape(()), oloss.detach(), rtol=RTOL, atol=1e-7)
    m = metrics.cpu()
    np.testing.assert_allclose(m[16].item(), float(oloss.detach()), rtol=RTOL, atol=1e-7)  # actor/total_loss
    np.testing.assert_allclose(m[15].item(), float(ent_loss.detach()), rtol=RTOL, atol=1e-7)  # actor/entropy_loss
    for slot, key in L.M_KEYS.items():
        if key in om and key != "critic/value_clip_ratio":
            np.testing.assert_allclose(m[slot].item(), om[key], rtol=RTOL, atol=1e-7, err_msg=key)
    zero = torch.zeros(n, A)
    torch.testing.assert_close(d_lp.cpu(), new.grad if new.grad is not None else zero, rtol=RTOL, atol=1e-10)
    torch.testing.assert_close(d_v.cpu(), val.grad, rtol=RTOL, atol=1e-10)
    torch.testing.assert_close(d_e.cpu(), ent.grad if ent.grad is not None else zero, rtol=RTOL, atol=1e-12)
    if warmup:
        assert float(d_lp.abs().max()) == 0.0 and float(d_e.abs().max()) == 0.0


def test_fused_embodied_policy_loss_takes_entropy_kwargs():
    """The plugin-level entry routes entropy / entropy_bonus / loss_scale to the kernel (extension kwargs; without
    them it is the reference's policy_loss)."""
    from rlinf_b200.algorithms import policy_loss

    n, A = 512, 4
    g = torch.Generator().manual_seed(2)
    old = -1 + 0.3 * torch.randn(n, A, generator=g)
    new = (old + 0.05 * torch.randn(n, A, generator=g)).cuda().requires_grad_(True)
    ent = (1.0 + 0.2 * torch.randn(n, A, generator=g)).cuda().requires_grad_(True)
    adv, ret, pv = (torch.randn(n, 1, generator=g) for _ in range(3))
    val = (pv + 0.1 * torch.randn(n, 1, generator=g)).cuda().requires_grad_(True)
    kw = dict(task_type="embodied", loss_type="actor_critic", logprob_type="action_level", reward_type="action_level",
              single_action_dim=A, logprobs=new, values=val, old_logprobs=old, advantages=adv, returns=ret,
              prev_values=pv, clip_ratio_high=0.2, clip_ratio_low=0.2, value_clip=0.2, huber_delta=10.0,
              loss_mask=None, loss_mask_sum=None, max_episode_steps=10, critic_warmup=False)
    loss, md = policy_loss(entropy=ent, entropy_bonus=0.02, entropy_type="action_level", **kw)
    loss.backward()
    n_new, n_val, n_ent = (new.detach().cpu().requires_grad_(True), val.detach().cpu().requires_grad_(True),
                           ent.detach().cpu().requires_grad_(True))
    hp = dict(clip_ratio_low=0.2, clip_ratio_high=0.2, value_clip=0.2, huber_delta=10.0)
    oloss, _ = O.policy_loss_embodied("actor_critic", n_new, old, adv, "action_level", A, values=n_val, prev_values=pv,
                                      returns=ret, **hp)
    e = O.entropy_term(n_ent, "action_level", A, n, None)
    oloss = oloss - 0.02 * e
    oloss.backward()
    torch.testing.assert_close(loss.detach().cpu(), oloss.detach(), rtol=RTOL, atol=1e-7)
    np.testing.assert_allclose(md["actor/entropy_loss"], float(e.detach()), rtol=RTOL)
    torch.testing.assert_close(new.grad.cpu(), n_new.grad, rtol=RTOL, atol=1e-10)
    torch.testing.assert_close(ent.grad.cpu(), n_ent.grad, rtol=RTOL, atol=1e-12)
    torch.testing.assert_close(val.grad.cpu(), n_val.grad, rtol=RTOL, atol=1e-10)


# ---------------------------------------------------------------------------------------------------------------
# a11: rollout_epoch > 1 merge through the actor; chunk_level reward preprocessing
# ---------------------------------------------------------------------------------------------------------------
def test_rollout_epoch_merge_through_actor(golden):
    """process_nested_dict_for_adv (nested_dict_process.py:251-269) as EmbodiedActor.recv_rollout_trajectories applies
    it: [E*nc, B, ...] -> [nc, E*B, ...], against the reference-generated golden and on a full batch."""
    from rlinf_b200.actor import EmbodiedActor
    from rlinf_b200.config import synthetic_ppo_config

    g = golden("indexing")
    E, nc, B, obs, act = 2, 6, 16, 4, 2
    cfg = synthetic_ppo_config(B=B, T=nc, obs_dim=obs, action_dim=act, update_epoch=1, num_minibatches=2,
                               **{"env.train.rollout_epoch": E, "runner.rollout_metrics": False})
    cfg.actor.global_batch_size = E * nc * B // 2
    cfg.actor.micro_batch_size = E * nc * B // 2
    actor = EmbodiedActor(cfg)
    x = _t(g["merge_in"])
    merged = actor._process_received_rollout_batch({"x": x.cuda(), "dones": torch.zeros(E * 4, 4, 1, dtype=torch.bool).cuda()})
    assert torch.equal(merged["x"].cpu().contiguous(), _t(g["merge_out"]))
    # full batch: two rollout epochs stacked on the time axis, as the reference's channel delivers them
    gen = torch.Generator().manual_seed(4)
    batch = {
        "rewards": torch.randn(E * nc, B, 1, generator=gen),
        "dones": torch.rand(E * (nc + 1), B, 1, generator=gen) < 0.1,
        "prev_values": torch.randn(E * (nc + 1), B, 1, generator=gen),
        "prev_logprobs": -1 + 0.3 * torch.randn(E * nc, B, act, generator=gen),
        "forward_inputs": {"states": torch.randn(E * nc, B, obs, generator=gen),
                           "action": torch.randn(E * nc, B, act, generator=gen)},
    }
    for e in range(E):
        batch["dones"][e * (nc + 1)] = False
    batch["terminations"] = batch["dones"].clone()
    batch["truncations"] = torch.zeros_like(batch["dones"])
    orc = RunnerOracle(cfg, params={k: p.detach().cpu().clone() for k, p in actor.model.named_parameters()})
    om = orc.update({k: (dict(v) if isinstance(v, dict) else v.clone()) for k, v in batch.items()})
    actor.recv_rollout_trajectories(batch)
    rb = actor.rollout_batch
    assert rb["rewards"].shape == (nc, E * B, 1) and rb["dones"].shape == (nc + 1, E * B, 1)
    ref_merged = O.merge_rollout_epochs(batch, E)
    for k in ("rewards", "dones", "prev_values", "prev_logprobs"):
        assert torch.equal(rb[k].cpu(), ref_merged[k]), k
    actor.compute_advantages_and_returns()
    m = actor.run_training()
    for name, p in actor.model.named_parameters():
        torch.testing.assert_close(p.cpu(), orc.params[name].detach(), rtol=1e-4, atol=2e-5, msg=name)
    for k in ("actor/policy_loss", "critic/value_loss", "actor/grad_norm", "actor/approx_kl"):
        np.testing.assert_allclose(m[k], om[k], rtol=2e-4, atol=1e-6, err_msg=k)


@pytest.mark.parametrize("with_mask", [False, True])
def test_chunk_level_reward_preprocessing_vs_oracle(with_mask):
    """preprocess_embodied_advantages_inputs, reward_type='chunk_level' (algorithms/utils.py:67-131): rewards summed and
    dones max-ed over the chunk, [nc,B,1] in / out."""
    import rlinf_b200.algorithms as A

    nc, B, C = 10, 24, 4
    g = torch.Generator().manual_seed(8)
    rewards = torch.randn(nc, B, C, generator=g)
    dones = torch.rand(nc + 1, B, C, generator=g) < 0.05
    dones[0] = False
    values = torch.randn(nc + 1, B, 1, generator=g)
    lm, lms = (O.loss_mask_from_dones(dones) if with_mask else (None, None))
    if with_mask:
        lm, lms = lm.any(dim=-1, keepdim=True), lms[..., -1:]
    kw = dict(task_type="embodied", adv_type="gae", rewards=rewards, dones=dones, values=values, gamma=0.99,
              gae_lambda=0.95, group_size=8, reward_type="chunk_level", num_action_chunks=C, loss_mask=lm,
              loss_mask_sum=lms)
    res = A.calculate_adv_and_returns(**kw)
    ref = O.adv_and_returns_embodied("gae", rewards, dones, values, lm, lms, 0.99, 0.95, 8, "chunk_level")
    assert res["returns"].shape == ref["returns"].shape == (nc, B, 1)
    # the chunk sum of the rewards is a device reduction (summation order differs from the CPU's): close, not bit-equal
    torch.testing.assert_close(res["returns"].cpu(), ref["returns"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(res["advantages"].cpu(), ref["advantages"], rtol=RTOL, atol=1e-5)


# ---------------------------------------------------------------------------------------------------------------
# a23: non-finite gradient norm -> the optimiser step is skipped; frozen groups; device-side lr table
# ---------------------------------------------------------------------------------------------------------------
def test_non_finite_grad_norm_skips_the_step():
    """fsdp_model_manager.py:442-447: `if not torch.isfinite(grad_norm): skip`; parameters, moments and the step count
    are untouched and the skipped flag is raised; the next finite step proceeds normally."""
    from rlinf_b200.policy import FlatAdamW, MLPPolicy

    pol = MLPPolicy(obs_dim=8, action_dim=2, seed=3)
    opt = FlatAdamW(pol, lr=1e-3, value_lr=1e-3, clip_grad=0.5)
    pol.flat_grads.normal_(generator=torch.Generator(device="cuda").manual_seed(0))
    opt.step()
    p1, m1, v1 = pol.flat_params.clone(), opt.exp_avg.clone(), opt.exp_avg_sq.clone()
    assert opt.state[0].item() == 1 and opt.state[3].item() == 0
    for bad in (float("nan"), float("inf")):
        pol.flat_grads[17] = bad
        opt.step()
        assert opt.state[3].item() == 1 and opt.state[0].item() == 1
        assert torch.equal(pol.flat_params, p1) and torch.equal(opt.exp_avg, m1) and torch.equal(opt.exp_avg_sq, v1)
    pol.flat_grads.normal_(generator=torch.Generator(device="cuda").manual_seed(1))
    opt.step()
    assert opt.state[3].item() == 0 and opt.state[0].item() == 2 and not torch.equal(pol.flat_params, p1)


def test_frozen_group_is_untouched_and_lr_table_follows_lr_scale():
    from rlinf_b200.policy import FlatAdamW, MLPPolicy

    pol = MLPPolicy(obs_dim=8, action_dim=2, seed=3)
    params = {n: p.detach().cpu().clone().requires_grad_(True) for n, p in pol.named_parameters()}
    opt = FlatAdamW(pol, lr=1e-3, value_lr=2e-3, clip_grad=0.0)
    gen = torch.Generator().manual_seed(0)
    oopt = O.build_adamw(params, 1e-3, 2e-3, enable_critic_warmup=True)
    opt.frozen = {"actor"}
    for step in range(3):
        opt.lr_scale = 0.5 + 0.25 * step
        for gname, gr in pol.named_grads():
            x = torch.randn(gr.shape, generator=gen)
            gr.copy_(x)
            params[gname].grad = x.clone() if "value_head" in gname else None
        for grp in oopt.param_groups:
            grp["lr"] = 2e-3 * opt.lr_scale
        opt.step()
        oopt.step()
    for n, p in pol.named_parameters():
        torch.testing.assert_close(p.cpu(), params[n].detach(), rtol=1e-5, atol=1e-7, msg=n)
    assert opt.lr_list() == [2e-3 * opt.lr_scale]


# ---------------------------------------------------------------------------------------------------------------
# a21: every fused-rollout template instance vs the ORACLE (not vs the per-kernel path)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [600, 1100, 2100, 4096])
def test_fused_rollout_instances_vs_oracle(B):
    """E = ceil(B/148) = 5, 8, 15, 28 environments per CTA: the <=8, <=16 and register-tiled instances the N = 2/4/8
    scaling runs use, with injected noise: flags bit-exact, floats within 1e-4 of the oracle's loop."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    T, obs, act = 12, 16, 3
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=act, **{"rollout.fused_kernel": True,
                                                                          "env.train.p_term": 0.03,
                                                                          "env.train.max_episode_steps": 5,
                                                                          "algorithm.bootstrap_type": "standard"})
    run = EmbodiedRunner(cfg)
    assert run.rollout._fused
    orc = RunnerOracle(cfg, params={n: p.detach().cpu().clone() for n, p in run.actor.model.named_parameters()})
    g = torch.Generator().manual_seed(B)
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
    assert (run.env.elapsed.cpu() == orc.env.elapsed).all()


# ---------------------------------------------------------------------------------------------------------------
# end to end at the config-2 network shapes (obs=128, act=8 -> every hidden GEMM on tcgen05)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(os.environ.get("RB200_SLOW", "1") == "0", reason="RB200_SLOW=0 skips the ~1 min oracle run")
def test_runner_update_vs_oracle_with_tensor_core_towers():
    """B=256, T=64 (16384 samples), obs=128, act=8, 2 epochs x 2 mini-batches x 2 micro-batches: rollout on the device,
    then the same batch through RunnerOracle.update and EmbodiedRunner.update_phase; parameters after 4 optimiser
    steps and every metric within 1e-4 / 2e-4."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    B, T, obs, act = 256, 64, 128, 8
    n = B * T
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=act, update_epoch=2, num_minibatches=2,
                               micro_batch_size=n // 4, **{"algorithm.entropy_bonus": 0.005})
    run = EmbodiedRunner(cfg)
    run.rollout_phase()
    torch.cuda.synchronize()
    batch = _cpu_batch(run.buffer.as_batch())
    orc = RunnerOracle(cfg, params={k: p.detach().cpu().clone() for k, p in run.actor.model.named_parameters()})
    om = orc.update(batch)
    m = run.update_phase()
    worst = 0.0
    for name, p in run.actor.model.named_parameters():
        ref = orc.params[name].detach()
        torch.testing.assert_close(p.cpu(), ref, rtol=1e-4, atol=2e-5, msg=name)
        worst = max(worst, (p.cpu() - ref).abs().max().item())
        frac_tight = ((p.cpu() - ref).abs() <= 1e-4 * ref.abs() + 1e-6).float().mean().item()
        assert frac_tight > 0.99, (name, frac_tight)
    print("config-2 shapes: max |param - oracle| after 4 steps:", worst)
    for k, v in om.items():
        if k in ("critic/value_clip_ratio",):
            continue
        assert k in m, k
        np.testing.assert_allclose(m[k], v, rtol=2e-4, atol=1e-6, err_msg=k)


# ---------------------------------------------------------------------------------------------------------------
# critic warm-up and LR schedule through the runner; GRPO with auto_reset off over several iterations
# ---------------------------------------------------------------------------------------------------------------
def test_critic_warmup_matches_reference_optimizer_semantics():
    """critic_warmup_steps=3 with 4 optimiser steps per run_training: actor frozen (no update, no decay) for 3 steps,
    lr reported 0.0, then a REBUILT optimiser (step count 0; moments primed by warmup_optimizer_state with the last
    warm-up gradient of the value head, zeros for the actor) - fsdp_model_manager.py:451-459, utils/utils.py:594-663;
    the oracle side of this comparison is pinned against the reference worker by golden_r5 "warmup"."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    B, T, obs, act = 64, 16, 4, 2
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=obs, action_dim=act, update_epoch=2, num_minibatches=2,
                               **{"actor.optim.critic_warmup_steps": 3, "actor.optim.value_lr": 5e-4})
    run = EmbodiedRunner(cfg)
    p0 = {k: p.detach().cpu().clone() for k, p in run.actor.model.named_parameters()}
    orc = RunnerOracle(cfg, params={k: v.clone() for k, v in p0.items()})
    for it in range(2):
        run.rollout_phase()
        torch.cuda.synchronize()
        batch = _cpu_batch(run.buffer.as_batch())
        om = orc.update(batch)
        m = run.update_phase()
        for name, p in run.actor.model.named_parameters():
            ref = orc.params[name].detach()
            # Adam is sign-like for |g| ~ eps: a few near-zero-gradient entries move by up to ~1 % of steps * lr
            torch.testing.assert_close(p.cpu(), ref, rtol=1e-4, atol=4e-5, msg=f"{it} {name}")
            assert ((p.cpu() - ref).abs() <= 1e-4 * ref.abs() + 2e-6).float().mean().item() > 0.99, (it, name)
            if it == 0 and "value_head" not in name and name != "actor_logstd":
                # 3 of the 4 steps froze the actor (no update, NO weight decay): it moved by exactly one Adam step
                assert float((p.cpu() - p0[name]).abs().max()) <= 3.0e-4 * 1.01 + 3e-4 * 0.01 * float(p0[name].abs().max())
        for k in ("actor/lr", "critic/lr", "actor/policy_loss", "critic/value_loss", "actor/grad_norm"):
            if k in om:
                np.testing.assert_allclose(m[k], om[k], rtol=2e-4, atol=1e-9, err_msg=f"{it} {k}")
        assert ("critic/lr" in m) == ("critic/lr" in om)
    assert run.actor.critic_warmup_steps == 0 and run.actor.optimizer.state[0].item() == 5


@pytest.mark.parametrize("kind", ["constant", "cosine", "openpi_cosine"])
def test_lr_schedule_through_the_runner(kind):
    """LambdaLR stepped once per run_training (embodied_fsdp_actor_worker.py:571): lr of iteration k = base*lambda(k)."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    over = {"actor.optim.lr_scheduler": kind, "actor.optim.lr_warmup_steps": 2, "actor.optim.total_training_steps": 6,
            "actor.optim.min_lr": 3e-5, "actor.optim.value_lr": 1e-3}
    cfg = synthetic_ppo_config(B=32, T=8, obs_dim=4, action_dim=2, update_epoch=1, num_minibatches=2, **over)
    run = EmbodiedRunner(cfg)
    orc = RunnerOracle(cfg, params={k: p.detach().cpu().clone() for k, p in run.actor.model.named_parameters()})
    for it in range(4):
        run.rollout_phase()
        torch.cuda.synchronize()
        om = orc.update(_cpu_batch(run.buffer.as_batch()))
        m = run.update_phase()
        np.testing.assert_allclose(m["actor/lr"], om["actor/lr"], rtol=1e-12, atol=0, err_msg=f"{it}")
        np.testing.assert_allclose(m["critic/lr"], om["critic/lr"], rtol=1e-12, atol=0, err_msg=f"{it}")
        for name, p in run.actor.model.named_parameters():
            torch.testing.assert_close(p.cpu(), orc.params[name].detach(), rtol=1e-4, atol=2e-5, msg=f"{it} {name}")


def test_grpo_auto_reset_off_resets_envs_every_rollout():
    """bootstrap_step (env_worker.py:908-935): with auto_reset off the envs are reset at every rollout epoch, so
    `elapsed` restarts and the loss mask keeps whole first episodes in EVERY iteration (not one step per env)."""
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    B, T = 64, 12
    cfg = synthetic_ppo_config(B=B, T=T, obs_dim=6, action_dim=2, update_epoch=1, num_minibatches=2, adv_type="grpo",
                               loss_type="actor", group_size=8,
                               **{"env.train.auto_reset": False, "env.train.max_episode_steps": 6,
                                  "env.train.p_term": 0.02, "actor.model.add_value_head": False})
    run = EmbodiedRunner(cfg)
    orc = RunnerOracle(cfg, params={k: p.detach().cpu().clone() for k, p in run.actor.model.named_parameters()})
    kept = []
    for it in range(3):
        run.rollout_phase()
        torch.cuda.synchronize()
        batch = _cpu_batch(run.buffer.as_batch())
        d = batch["dones"][..., 0]
        first_done = torch.where(d.any(0), d.float().argmax(0), torch.full((B,), T + 1))
        assert int(first_done.max()) <= 6 and int(first_done.min()) >= 1  # truncation at 6 at the latest, in EVERY rollout
        assert int(first_done.float().mean()) >= 4, first_done
        om = orc.update(batch)
        m = run.update_phase()
        kept.append(float(run.actor.rollout_batch["loss_mask"].float().mean()))
        for name, p in run.actor.model.named_parameters():
            torch.testing.assert_close(p.cpu(), orc.params[name].detach(), rtol=1e-4, atol=2e-5, msg=f"{it} {name}")
        np.testing.assert_allclose(m["actor/policy_loss"], om["actor/policy_loss"], rtol=2e-4, atol=1e-7)
    assert min(kept) > 0.3, kept  # ~ first-episode length / T each iteration; round 1 collapsed to 1/T from iteration 2


# ---------------------------------------------------------------------------------------------------------------
# 2 ranks over NCCL: per-rank shuffles + averaged gradients == the oracle's data-parallel emulation
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("graph", [False, True])
def test_two_rank_nccl_update_matches_oracle(tmp_path, graph):
    import json
    import socket
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    if graph and os.environ.get("RB200_EXPERIMENTAL", "0") != "1":
        # measured on 2 x B200: with the NCCL all-reduce captured inside the step graph the run never completed (500 s
        # timeout, profiles/r02_two_rank_nccl.txt); multi-rank graphed steps are therefore opt-in
        # (actor.cuda_graph_multi_rank) and this variant only runs with RB200_EXPERIMENTAL=1
        pytest.skip("experimental: multi-rank CUDA-graphed optimiser step (hangs on 2 x B200)")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    outp = tmp_path / "dist.json"
    env = dict(os.environ, RB200_DIST_OUT=str(outp), RB200_DIST_GRAPH="1" if graph else "0")
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "dist_nccl_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), worker], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads(outp.read_text())
    print(res)
    assert res["ok"], res
    assert all(i["replicas_identical"] for i in res["iters"])
