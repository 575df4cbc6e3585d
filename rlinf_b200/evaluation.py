"""Policy evaluation with per-episode environment metrics: the eval half of EmbodiedRunner.

Reference: EmbodiedRunner._maybe_eval_and_checkpoint / evaluate (rlinf/runners/embodied_runner.py:193-206, 308-329),
check_progress (rlinf/utils/runner_utils.py:31-60), EnvWorker.evaluate / env_evaluate_step
(rlinf/workers/env/env_worker.py:1374-1460, 557-620), MultiStepRolloutWorker.evaluate
(rlinf/workers/rollout/hf/huggingface_worker.py:803-872) with MLPPolicy mode="eval" (the action is the mean,
mlp_policy.py:268-271), the episode bookkeeping of ManiskillEnv (rlinf/envs/maniskill/maniskill_env.py:232-391) and
compute_evaluate_metrics (rlinf/utils/metric_utils.py:372-420).

Per chunk step: one mean-action inference (`rb200_mlp_mean`) and one eval env step (`rb200_synth_env_eval_step`), which
writes one row of per-episode records `[epochs * n_chunk_steps, B]` (reported flag | success_once | success_at_end,
return, episode_len).  After the loop `rb200_eval_metrics` reduces the records to six fp64 sums; that vector (all-reduced
over ranks) is the only thing read back on the host.  The loop is captured as a CUDA graph after the first call,
weight-split refresh included, so a replay after an optimiser step reads the current weights.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist

from . import _lib as L
from .config import wrap
from .envs import SyntheticVectorEnv

# order of the sums rb200_eval_metrics returns (the count is the 6th)
SUM_KEYS = ("return", "episode_len", "reward", "success_once", "success_at_end")
EVAL_MAX_PARTS = 512  # RB200_EVAL_MAX_PARTS


def check_progress(step, max_steps, val_check_interval, save_interval, limit_val_batches, run_time_exceeded=False):
    """check_progress (rlinf/utils/runner_utils.py:31-60): (run_val, save_model, is_train_end)."""
    is_validation_enabled = limit_val_batches != 0 and val_check_interval > 0
    is_save_enabled = save_interval > 0
    is_train_end = step == max_steps
    if is_validation_enabled and not (save_interval < 0 or save_interval % val_check_interval == 0):
        raise ValueError(f"save_interval={save_interval} must be divisible by val_check_interval={val_check_interval}")

    def divisible(a, b):
        return a != 0 and b != 0 and a % b == 0

    run_val = (divisible(step, val_check_interval) or is_train_end or run_time_exceeded) and is_validation_enabled
    save_model = (divisible(step, save_interval) or is_train_end or run_time_exceeded) and is_save_enabled
    return run_val, save_model, is_train_end


def metrics_from_sums(sums, ignore_terminations):
    """compute_evaluate_metrics over all reported episodes: the mean of each key plus num_trajectories.  `sums` = the
    (all-reduced) rb200_eval_metrics vector.  success_at_end exists only with ignore_terminations (maniskill_env.py:
    306-312); no reported episode -> only num_trajectories, as in the reference."""
    count = float(sums[5])
    out = {}
    if count > 0:
        for i, k in enumerate(SUM_KEYS):
            if k != "success_at_end" or ignore_terminations:
                out[k] = float(sums[i]) / count
    out["num_trajectories"] = count
    return out


class EvalWorker:
    """One rank's eval env and the device-resident evaluation loop."""

    def __init__(self, cfg, policy, train_env, rank=0, world_size=1, process_group=None):
        self.cfg, self.policy = cfg, policy
        ev, et = wrap(cfg.env["eval"]), cfg.env.train
        self.rank, self.world_size, self.pg = rank, world_size, process_group
        total = int(ev.total_num_envs)
        if total % world_size != 0:
            raise ValueError(f"env.eval.total_num_envs={total} is not divisible by world_size={world_size}")
        self.B = total // world_size
        self.C = int(cfg.actor.model.get("num_action_chunks", 1))
        T = int(ev.max_steps_per_rollout_epoch)
        if T % self.C != 0:
            raise ValueError(f"env.eval.max_steps_per_rollout_epoch {T} is not a multiple of num_action_chunks {self.C}")
        self.n_chunk_steps = T // self.C  # n_eval_chunk_steps
        self.epochs = int(ev.get("rollout_epoch", 1))
        self.auto_reset = bool(ev.auto_reset)
        self.ignore_terminations = bool(ev.get("ignore_terminations", False))
        seed = int(ev.get("seed", et.get("seed", 1234))) + 1000 * rank
        self.env = SyntheticVectorEnv(self.B, train_env.obs_dim, train_env.action_dim, int(ev.max_episode_steps),
                                      auto_reset=self.auto_reset, p_term=ev.get("p_term", et.get("p_term", 0.005)),
                                      noise_std=ev.get("noise_std", et.get("noise_std", 0.1)),
                                      reward_noise_std=ev.get("reward_noise_std", et.get("reward_noise_std", 0.01)),
                                      seed=seed, device=policy.device)
        self.env.w_s.copy_(train_env.w_s)  # same dynamics as the training env
        self.env.w_a.copy_(train_env.w_a)
        dev, B, obs = policy.device, self.B, train_env.obs_dim
        R = self.epochs * self.n_chunk_steps
        self.n_resets = self.epochs if not self.auto_reset else 1  # evaluate(): reset at epoch 0 / every epoch
        self.init_states = torch.zeros(self.n_resets, B, obs, device=dev)
        self.ep_return = torch.zeros(B, dtype=torch.float32, device=dev)
        self.ep_flags = torch.zeros(B, dtype=torch.uint8, device=dev)
        self.rec_flags = torch.zeros(R, B, dtype=torch.uint8, device=dev)
        self.rec_return = torch.zeros(R, B, dtype=torch.float32, device=dev)
        self.rec_len = torch.zeros(R, B, dtype=torch.int32, device=dev)
        self.mean = torch.zeros(B, policy.act_dim, dtype=torch.float32, device=dev)
        self.noise = None  # [R, B, C*(obs+2)+obs] when the caller injects the env noise (parity tests)
        self._scratch = torch.empty(3, B, obs, device=dev)
        self._work = torch.empty(int(L.load().rb200_mlp_fwd_scratch_floats(C.byref(policy.layout), B)), device=dev)
        self._part = torch.zeros(EVAL_MAX_PARTS, 6, dtype=torch.float64, device=dev)
        self.sums = torch.zeros(6, dtype=torch.float64, device=dev)
        self._graphs = {}
        self._calls = set()
        self.graph_kernel_count = 0  # kernels replayed per evaluate once the CUDA graph exists
        self._use_graph = bool(cfg.rollout.get("enable_cuda_graph", True))

    def _rewind(self):
        """Initial states of every reset of one evaluate(): the reset generator is rewound first, so they (and the
        Philox env noise, whose chunk counter restarts at 0) are the same on every call."""
        self.env._reset_gen.manual_seed(self.env.seed + 1)
        for k in range(self.n_resets):
            obs, _ = self.env.reset()
            self.init_states[k].copy_(obs["states"])

    def _loop(self, noise):
        """The whole evaluation on the current stream: resets, chunk steps, metric reduction (captured as a graph)."""
        lib = L.load()
        pol, env, st = self.policy, self.env, L.stream_ptr()
        pol.mark_params_changed()  # the weight-split refresh is part of the (captured) loop
        lay = C.byref(pol.layout)
        n = self.n_chunk_steps
        obs, act = env.obs_dim, env.action_dim
        for e in range(self.epochs):
            if e == 0 or not self.auto_reset:
                env.state.copy_(self.init_states[e if not self.auto_reset else 0])
                env.elapsed.zero_()
                self.ep_return.zero_()
                self.ep_flags.zero_()
            for k in range(n):
                row = e * n + k
                L.check(lib.rb200_mlp_mean(lay, L.ptr(pol.flat_params), pol._ws(), L.ptr(env.state), self.B,
                                           L.ptr(self.mean), L.ptr(self._work), st), "mlp_mean")
                L.check(lib.rb200_synth_env_eval_step(
                    L.ptr(env.w_s), L.ptr(env.w_a), L.ptr(env.state), L.ptr(self.mean),
                    None if noise is None else L.ptr(noise[row]), L.ptr(env.elapsed), L.ptr(self.ep_return),
                    L.ptr(self.ep_flags), L.ptr(self.rec_flags[row]), L.ptr(self.rec_return[row]),
                    L.ptr(self.rec_len[row]), L.ptr(self._scratch), self.B, obs, act, self.C, env.max_episode_steps,
                    int(self.auto_reset), int(self.ignore_terminations), env.p_term, env.noise_std,
                    env.reward_noise_std, env.seed, row, st), "synth_env_eval_step")
        L.check(lib.rb200_eval_metrics(L.ptr(self.rec_flags), L.ptr(self.rec_return), L.ptr(self.rec_len),
                                       self.rec_flags.numel(), L.ptr(self._part), L.ptr(self.sums), st), "eval_metrics")

    def run(self, env_noise=None, init_states=None):
        """One evaluation; returns the device sum vector (not yet all-reduced).  env_noise [R, B, C*(obs+2)+obs] /
        init_states [n_resets, B, obs]: pre-drawn noise and initial states (parity tests); None -> Philox / the
        rewound reset generator."""
        if init_states is not None:
            self.init_states.copy_(init_states)
        else:
            self._rewind()
        noise = None
        if env_noise is not None:
            if self.noise is None:
                self.noise = torch.empty(env_noise.shape, dtype=torch.float32, device=self.policy.device)
            self.noise.copy_(env_noise)
            noise = self.noise
        key = noise is not None
        if not self._use_graph or key not in self._calls:
            self._calls.add(key)
            self._loop(noise)  # the first call of each kind runs eagerly
            return self.sums
        g = self._graphs.get(key)
        if g is None:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            n0 = L.load().rb200_launch_count()
            with torch.cuda.graph(g):
                self._loop(noise)
            self.graph_kernel_count = int(L.load().rb200_launch_count() - n0)
            self._graphs[key] = g
        g.replay()
        return self.sums

    def episodes(self):
        """Per-episode records of the last evaluation, compacted in the reference's order (eval step major, env
        index minor): dict of 1-D CPU tensors keyed like final_info["episode"]."""
        f = self.rec_flags.reshape(-1)
        sel = (f & 1).nonzero().squeeze(1)
        ret = self.rec_return.reshape(-1)[sel].cpu()
        ln = self.rec_len.reshape(-1)[sel].cpu()
        fs = f[sel].cpu()
        out = {"success_once": (fs & 2) != 0, "return": ret, "episode_len": ln, "reward": ret / ln}
        if self.ignore_terminations:
            out["success_at_end"] = (fs & 4) != 0
        return out

    def evaluate(self, return_episodes=False, env_noise=None, init_states=None):
        sums = self.run(env_noise, init_states)
        if self.world_size > 1:
            sums = sums.clone()
            dist.all_reduce(sums, group=self.pg)
        metrics = metrics_from_sums(sums.cpu().tolist(), self.ignore_terminations)  # the one host sync
        if return_episodes:
            return metrics, self.episodes()
        return metrics
