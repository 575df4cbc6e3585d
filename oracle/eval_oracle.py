"""CPU restatement of EmbodiedRunner.evaluate: mean-action episodes on the synthetic env with ManiSkill's episode
bookkeeping, and compute_evaluate_metrics.

TEST INFRASTRUCTURE ONLY (see oracle/rl_oracle.py header).  `EvalRunnerOracle` is `RunnerOracle` with `evaluate`; it is
pinned against executed reference code by tests/test_oracle_eval.py (tests/golden/golden_r7.npz) and is what the GPU
evaluation tests compare the CUDA path with.
"""
from __future__ import annotations

import torch

from . import rl_oracle as O
from .runner_oracle import RunnerOracle, SyntheticEnvCPU


class EvalRunnerOracle(RunnerOracle):
    """RunnerOracle + evaluation (embodied_runner.py:193-206, env_worker.py:1374-1460 / 557-620,
    huggingface_worker.py:803-872)."""

    @torch.no_grad()
    def evaluate(self, env_noise, init_states, num_envs=None):
        """One EmbodiedRunner.evaluate of this rank's eval envs (`cfg["env"]["eval"]`) with the mean action
        (MLPPolicy mode="eval", mlp_policy.py:268-271) and injected env noise [epochs*n_chunk_steps, B, C*(obs+2)+obs] /
        initial states [resets, B, obs] (one per epoch without auto_reset, else one).  Returns (metrics, episodes):
        compute_evaluate_metrics of this rank alone, and the reported per-episode records in the reference's order."""
        ev = self.cfg["env"]["eval"]
        B = num_envs or ev["total_num_envs"]
        Cn = self.num_action_chunks
        n = ev["max_steps_per_rollout_epoch"] // Cn  # n_eval_chunk_steps
        auto_reset, ignore_term = ev["auto_reset"], ev.get("ignore_terminations", False)
        et = self.cfg["env"]["train"]
        env = EpisodeEnvCPU(SyntheticEnvCPU(B, self.obs_dim, self.act_dim // Cn, ev["max_episode_steps"], auto_reset,
                                            ev.get("p_term", et.get("p_term", 0.005)),
                                            ev.get("noise_std", et.get("noise_std", 0.1)),
                                            ev.get("reward_noise_std", et.get("reward_noise_std", 0.01)),
                                            et.get("seed", 1234)), ignore_term)
        episodes = {}
        prev_done = None
        for e in range(ev.get("rollout_epoch", 1)):
            if not auto_reset or e == 0:  # evaluate(): reset at epoch 0, or every epoch without auto_reset
                state = env.reset(init_states[e if not auto_reset else 0])
                prev_done = torch.zeros(B, dtype=torch.bool)  # eval_prev_done
            for k in range(n):
                mean = O.mlp_forward(self.params, state, None, want_entropy=False, want_values=False)["mean"]
                state, done, info = env.chunk_step(mean.reshape(B, Cn, -1), env_noise[e * n + k])
                if auto_reset:
                    newly = done
                else:
                    newly = done & ~prev_done
                    prev_done = prev_done | done
                if bool(newly.any()):
                    for key, v in info.items():
                        episodes.setdefault(key, []).append(v[newly])
        episodes = {k: torch.cat(v) for k, v in episodes.items()}
        return compute_evaluate_metrics([episodes]), episodes


class EpisodeEnvCPU:
    """SyntheticEnvCPU behind ManiskillEnv's episode bookkeeping (maniskill_env.py:232-391): _record_metrics on every
    sub-step (returns += r in fp32, success_once |= success, episode_len = elapsed, reward = return / episode_len),
    ignore_terminations (terminations dropped after recording, success_at_end = success), chunk_step running its
    sub-steps past a done, and one _handle_auto_reset after the chunk (_reset_metrics of the reset envs).  The synthetic
    env's termination draw is its `success` info."""

    def __init__(self, env: SyntheticEnvCPU, ignore_terminations=False):
        self.env, self.ignore_terminations = env, ignore_terminations

    def reset(self, states):
        B = self.env.B
        self.env.elapsed.zero_()
        self.returns = torch.zeros(B, dtype=torch.float32)
        self.success_once = torch.zeros(B, dtype=torch.bool)
        self.state = states.clone()
        return self.state

    def chunk_step(self, chunk_actions, noise):
        """-> (next state, chunk done [B], infos["episode"] of the chunk's last sub-step)."""
        C, obs = chunk_actions.shape[1], self.env.obs_dim
        state, term_any, trunc_any = self.state, None, None
        for c in range(C):
            state, r, term, trunc = self.env.substep_given_noise(state, chunk_actions[:, c],
                                                                 noise[:, c * (obs + 2):(c + 1) * (obs + 2)])
            success = term.clone()
            self.returns = self.returns + r
            self.success_once = self.success_once | success
            info = {"success_once": self.success_once.clone(), "return": self.returns.clone(),
                    "episode_len": self.env.elapsed.clone()}
            info["reward"] = info["return"] / info["episode_len"]
            if self.ignore_terminations:
                term = torch.zeros_like(term)
                info["success_at_end"] = success.clone()
            term_any = term if term_any is None else term_any | term
            trunc_any = trunc if trunc_any is None else trunc_any | trunc
        done = term_any | trunc_any
        if self.env.auto_reset and bool(done.any()):
            state = torch.where(done.unsqueeze(-1), noise[:, C * (obs + 2):], state)
            self.env.elapsed[done] = 0
            self.returns[done] = 0.0
            self.success_once[done] = False
        self.state = state
        return state, done, info


def compute_evaluate_metrics(eval_metrics_list):
    """compute_evaluate_metrics (rlinf/utils/metric_utils.py:372-420) for per-episode dicts: the fp32 mean of each key
    over every rank's episodes, plus num_trajectories."""
    keys = []
    for d in eval_metrics_list:
        keys += [k for k in d if k not in keys]
    out = {}
    for k in keys:
        stacked = torch.cat([d[k].reshape(-1).float() for d in eval_metrics_list if k in d])
        out[k] = float(stacked.mean()) if stacked.numel() > 0 else 0.0
    out["num_trajectories"] = sum(next(iter(d.values())).shape[0] if d else 0 for d in eval_metrics_list)
    return out
