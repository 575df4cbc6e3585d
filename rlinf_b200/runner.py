"""Single-process-per-GPU driver loop - mirror of EmbodiedRunner.run().

Reference: rlinf/runners/embodied_runner.py:478-563 (set_global_step, update_rollout_weights,
env.interact || rollout.generate || actor.recv_rollout_trajectories, compute_advantages_and_returns,
run_training, metrics).  Not a port of the Ray worker stack: one process per GPU owns the env shard,
the rollout policy replica and the learner; experience shards over ranks by environment.
"""
from __future__ import annotations

import time

import torch
import torch.distributed as dist

from . import _lib as L
from .actor import EmbodiedActor
from .config import wrap
from .envs import SyntheticVectorEnv
from .rollout import RolloutBuffer, RolloutWorker


class EmbodiedRunner:
    def __init__(self, cfg, rank=None, world_size=None, process_group=None):
        self.cfg = cfg = wrap(cfg)
        self._dist = dist.is_available() and dist.is_initialized()
        self.rank = rank if rank is not None else (dist.get_rank() if self._dist else 0)
        self.world_size = world_size if world_size is not None else (dist.get_world_size() if self._dist else 1)
        et, m = cfg.env.train, cfg.actor.model
        from .dist_utils import shard_envs
        self.env_start, self.B = shard_envs(et.total_num_envs, self.world_size, self.rank,
                                            cfg.algorithm.get("group_size", 1))  # envs owned by this rank
        self.T = et.max_steps_per_rollout_epoch
        Cn = int(m.get("num_action_chunks", 1))
        if self.T % Cn != 0:
            raise ValueError(f"max_steps_per_rollout_epoch {self.T} is not a multiple of num_action_chunks {Cn}")
        self.n_chunk_steps = self.T // Cn  # env_worker.py: n_chunk_steps = max_steps_per_rollout_epoch // num_action_chunks
        self.actor = EmbodiedActor(cfg, rank=self.rank, world_size=self.world_size, process_group=process_group)
        pol = self.actor.model
        self.env = SyntheticVectorEnv(self.B, m.obs_dim, m.action_dim,  # the env takes ONE action per sub-step
                                      et.max_episode_steps, auto_reset=et.auto_reset, p_term=et.get("p_term", 0.005),
                                      noise_std=et.get("noise_std", 0.1),
                                      reward_noise_std=et.get("reward_noise_std", 0.01),
                                      seed=et.get("seed", 1234) + 1000 * self.rank)
        # dynamics are identical on every rank (same W_s / W_a), only the noise stream differs
        g = torch.Generator().manual_seed(et.get("seed", 1234))
        import math
        self.env.w_s.copy_(torch.randn(m.obs_dim, m.obs_dim, generator=g) / math.sqrt(m.obs_dim))
        self.env.w_a.copy_(torch.randn(m.action_dim, m.obs_dim, generator=g) / math.sqrt(m.action_dim))
        self.buffer = RolloutBuffer(self.n_chunk_steps, self.B, m.obs_dim, pol.act_dim, max(pol.value_dim, 1),
                                    num_action_chunks=Cn)
        self.rollout = RolloutWorker(cfg, pol, self.env, self.buffer)
        self.global_step = 0
        self._process_group = process_group
        self.eval_worker = None  # built on the first evaluate()
        r = cfg.runner
        self.max_steps = int(r.max_epochs)  # set_max_steps (embodied_runner.py:655-660): one step per epoch
        if int(r.get("max_steps", -1)) >= 0:
            self.max_steps = min(self.max_steps, int(r.max_steps))
        if self.world_size > 1:  # same initial weights everywhere (rank 0's)
            dist.broadcast(pol.flat_params, src=0, group=process_group)

    def update_rollout_weights(self):
        self.actor.sync_model_to_rollout(self.rollout.policy.flat_params)

    def rollout_phase(self):
        self.rollout.generate()

    def update_phase(self, batch=None):
        self.actor.recv_rollout_trajectories(batch if batch is not None else self.buffer.as_batch())
        rollout_metrics = self.actor.compute_advantages_and_returns()
        metrics = self.actor.run_training()
        metrics.update({f"rollout/{k}": v for k, v in rollout_metrics.items()})
        return metrics

    def evaluate(self, return_episodes=False, env_noise=None, init_states=None):
        """EmbodiedRunner.evaluate (embodied_runner.py:193-206): mean-action episodes on the eval env (`env.eval.*`),
        aggregated like compute_evaluate_metrics -> {success_once, return, episode_len, reward, [success_at_end],
        num_trajectories} as floats, over all ranks.  return_episodes: also this rank's per-episode records (eval step
        major, env index minor).  env_noise / init_states: pre-drawn env noise and initial states (parity tests).
        Reads the weights the rollout policy holds; call update_rollout_weights() first after an update."""
        if self.eval_worker is None:
            from .evaluation import EvalWorker

            self.eval_worker = EvalWorker(self.cfg, self.rollout.policy, self.env, self.rank, self.world_size,
                                          self._process_group)
        return self.eval_worker.evaluate(return_episodes, env_noise, init_states)

    def _maybe_eval(self):
        """_maybe_eval_and_checkpoint (embodied_runner.py:308-329) without checkpointing: evaluate every
        runner.val_check_interval steps and at the last step, after a weight sync."""
        r = self.cfg.runner
        vci = r.get("val_check_interval")
        if vci is None or vci <= 0:
            return {}
        from .evaluation import check_progress

        run_val, _, _ = check_progress(self.global_step, self.max_steps, vci, r.get("save_interval", -1), 1.0)
        if not run_val:
            return {}
        self.update_rollout_weights()
        return {f"eval/{k}": v for k, v in self.evaluate().items()}

    def run_iteration(self):
        self.actor.version = self.global_step
        if self.global_step % self.cfg.runner.get("weight_sync_interval", 1) == 0:
            self.update_rollout_weights()
        self.rollout_phase()
        metrics = self.update_phase()
        self.global_step += 1
        metrics.update(self._maybe_eval())
        return metrics

    def run(self, max_epochs=None):
        out = []
        for _ in range(max_epochs or self.cfg.runner.max_epochs):
            out.append(self.run_iteration())
        return out
