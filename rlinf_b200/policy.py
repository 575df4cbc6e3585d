"""MLP policy on one flat fp32 parameter buffer (+ matching flat gradient buffer).

Host-side mirror of rlinf/models/embodiment/mlp_policy/mlp_policy.py (`MLPPolicy`: 3x256 tanh
backbone, `actor_mean`, state-independent `actor_logstd`, `ValueHead` 3x256) for the
`add_value_head=True, add_q_head=False` configuration used by PPO/GRPO
(examples/embodiment/config/model/mlp_policy.yaml).  Parameter names, shapes and ordering are the
reference's `named_parameters()`, so a reference state_dict loads unchanged; storage is one flat
buffer so the gradient all-reduce, the clip and AdamW are single launches on contiguous memory.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import torch

from . import _lib as L

HIDDEN = 256


class MLPPolicy:
    def __init__(self, obs_dim: int, action_dim: int, num_action_chunks: int = 1, add_value_head: bool = True,
                 value_granularity: str = "action_level", device=None, seed: Optional[int] = None):
        self.obs_dim, self.action_dim, self.num_action_chunks = int(obs_dim), int(action_dim), int(num_action_chunks)
        self.act_dim = self.action_dim * self.num_action_chunks
        self.value_dim = 0 if not add_value_head else (1 if value_granularity == "chunk_level" else self.num_action_chunks)
        self.device = device or L.default_device()
        lib = L.load()
        self.layout = L.MlpLayout()
        L.check(lib.rb200_mlp_layout_init(C.byref(self.layout), self.obs_dim, self.act_dim, self.value_dim, HIDDEN),
                "mlp_layout_init")
        n = self.layout.total
        # 4 spare floats behind the parameters: slot n carries the weight VERSION in the parameter broadcast
        # (rlinf_b200/weight_sync.py: one NCCL broadcast of [params | version])
        self._param_store = torch.zeros(n + 4, dtype=torch.float32, device=self.device)
        self.flat_params = self._param_store[:n]
        self.flat_grads = torch.zeros(n, dtype=torch.float32, device=self.device)
        self._spec = self._build_spec()
        self._scratch: dict[tuple, torch.Tensor] = {}
        # tensor-core operand cache (packed fp16 hi/lo tiles of the hidden-layer weights)
        self.wsplit = torch.zeros(int(lib.rb200_mlp_wsplit_floats(C.byref(self.layout))), dtype=torch.float32,
                                  device=self.device)
        self._wsplit_fresh = False
        self.reset_parameters(seed)

    # ---- parameter bookkeeping --------------------------------------------------------------
    def _build_spec(self):
        Lo, H, O, A, V = self.layout, HIDDEN, self.obs_dim, self.act_dim, self.value_dim
        spec = [("actor_logstd", Lo.logstd, (1, A)),
                ("value_head.mlp.0.weight", Lo.vw0, (H, O)), ("value_head.mlp.0.bias", Lo.vb0, (H,)),
                ("value_head.mlp.2.weight", Lo.vw1, (H, H)), ("value_head.mlp.2.bias", Lo.vb1, (H,)),
                ("value_head.mlp.4.weight", Lo.vw2, (H, H)), ("value_head.mlp.4.bias", Lo.vb2, (H,)),
                ("value_head.mlp.6.weight", Lo.vw3, (V, H)),
                ("backbone.0.weight", Lo.bw0, (H, O)), ("backbone.0.bias", Lo.bb0, (H,)),
                ("backbone.2.weight", Lo.bw1, (H, H)), ("backbone.2.bias", Lo.bb1, (H,)),
                ("backbone.4.weight", Lo.bw2, (H, H)), ("backbone.4.bias", Lo.bb2, (H,)),
                ("actor_mean.weight", Lo.mw, (A, H)), ("actor_mean.bias", Lo.mb, (A,))]
        if V == 0:
            spec = [s for s in spec if not s[0].startswith("value_head")]
        return spec

    def named_parameters(self):
        for name, off, shape in self._spec:
            yield name, self.flat_params[off: off + math.prod(shape)].view(shape)

    def named_grads(self):
        for name, off, shape in self._spec:
            yield name, self.flat_grads[off: off + math.prod(shape)].view(shape)

    def state_dict(self):
        return {k: v.clone() for k, v in self.named_parameters()}

    def sync_buffer(self) -> torch.Tensor:
        """[flat parameters | version slot]: the tensor weight_sync.broadcast_flat sends."""
        return self._param_store[: self.flat_params.numel() + 1]

    def mark_params_changed(self):
        """Call after flat_params was modified (optimiser step, load, broadcast)."""
        self._wsplit_fresh = False

    def _ws(self):
        """Pointer to an up-to-date weight split (refreshed lazily, one launch)."""
        if not self._wsplit_fresh:
            L.check(L.load().rb200_mlp_prepare_weights(C.byref(self.layout), L.ptr(self.flat_params),
                                                       L.ptr(self.wsplit), L.stream_ptr()), "mlp_prepare_weights")
            self._wsplit_fresh = True
        return L.ptr(self.wsplit)

    def load_state_dict(self, sd: dict):
        views = dict(self.named_parameters())
        missing = [k for k in views if k not in sd]
        if missing:
            raise KeyError(f"missing parameters: {missing}")
        for k, v in views.items():
            v.copy_(sd[k].to(self.device, torch.float32).reshape(v.shape))
        self.mark_params_changed()

    def lr_group_ends(self):
        """Flat-buffer segments by lr group, in buffer order: names containing `value_head` use
        `optim.value_lr`, the rest `optim.lr` (fsdp_model_manager.py:534-559)."""
        segs = []
        for name, off, shape in self._spec:
            kind = "critic" if "value_head" in name else "actor"
            end = off + math.prod(shape)
            if segs and segs[-1][0] == kind:
                segs[-1][1] = end
            else:
                segs.append([kind, end])
        segs[-1][1] = int(self.layout.total)  # trailing alignment pad belongs to the last group
        return segs

    def reset_parameters(self, seed: Optional[int] = None):
        """Random init with the reference's distributions (layer_init orthogonal(sqrt 2), zero bias,
        actor_mean orthogonal(0.01*sqrt 2), logstd -0.5; value head kaiming_normal(fan_out, tanh) /
        N(0, 0.02)) - mlp_policy.py:91-105, modules/value_head.py:50-63.  Init runs on the host (torch
        CPU RNG) once; it is not on the hot path."""
        g = torch.Generator().manual_seed(0 if seed is None else int(seed))
        for name, p in self.named_parameters():
            if name == "actor_logstd":
                p.fill_(-0.5)
            elif name.endswith("bias"):
                p.zero_()
            elif name == "value_head.mlp.6.weight":
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif name.startswith("value_head"):
                p.copy_(torch.randn(p.shape, generator=g) * ((5.0 / 3.0) / math.sqrt(p.shape[0])))
            else:
                w = torch.empty(p.shape)
                gain = 0.01 * math.sqrt(2) if name.startswith("actor_mean") else math.sqrt(2)
                torch.nn.init.orthogonal_(w, gain=gain, generator=g)
                p.copy_(w)
        self.mark_params_changed()

    # ---- compute -------------------------------------------------------------------------------
    def _buf(self, key, numel):
        t = self._scratch.get(key)
        if t is None or t.numel() < numel:
            t = torch.empty(numel, dtype=torch.float32, device=self.device)
            self._scratch[key] = t
        return t

    def forward_train(self, states, action, idx=None, n=None, compute_entropy=True, compute_values=True):
        """default_forward (mlp_policy.py:202-236). states/action may be the whole rollout buffer with
        `idx` (int64) selecting this micro-batch's rows.  Keeps activations for `backward`."""
        lib = L.load()
        n = int(n if n is not None else (idx.numel() if idx is not None else states.shape[0]))
        nscr = lib.rb200_mlp_fwd_scratch_floats(C.byref(self.layout), n)
        acts = self._buf("acts", nscr)
        work = self._buf("work", nscr)
        logp = torch.empty((n, self.act_dim), dtype=torch.float32, device=self.device)
        ent = torch.empty_like(logp) if compute_entropy else None
        vals = torch.empty((n, self.value_dim), dtype=torch.float32, device=self.device) if (
            compute_values and self.value_dim > 0) else None
        L.check(lib.rb200_mlp_forward(C.byref(self.layout), L.ptr(self.flat_params), self._ws(), L.ptr(states),
                                      L.ptr(action), L.ptr(idx), n, L.ptr(logp), L.ptr(ent), L.ptr(vals), L.ptr(acts),
                                      L.ptr(work), L.stream_ptr()), "mlp_forward")
        self._last = (states, action, idx, n, acts)
        out = {"logprobs": logp}
        if ent is not None:
            out["entropy"] = ent
        if vals is not None:
            out["values"] = vals
        return out

    def backward(self, d_logprobs, d_values=None, d_entropy=None):
        """Accumulate (+=) parameter gradients of the last forward_train into `flat_grads`."""
        lib = L.load()
        states, action, idx, n, acts = self._last
        work = self._buf("work", acts.numel())
        L.check(lib.rb200_mlp_backward(C.byref(self.layout), L.ptr(self.flat_params), self._ws(), L.ptr(states),
                                       L.ptr(action), L.ptr(idx), n, L.ptr(d_logprobs), L.ptr(d_entropy), L.ptr(d_values),
                                       L.ptr(acts), L.ptr(work), L.ptr(self.flat_grads), L.stream_ptr()),
                "mlp_backward")

    def sample(self, states, noise=None, seed=0, offset=0, calculate_values=True, counter=None, out=None):
        """_generate_actions(mode="train") (mlp_policy.py:256-293): action ~ N(mean, exp(logstd)),
        log_prob, value. `noise` ([n,act] N(0,1) draws) makes the step reproducible for parity tests;
        otherwise Philox(seed, offset) on the device."""
        lib = L.load()
        n = states.shape[0]
        work = self._buf("sample", lib.rb200_mlp_fwd_scratch_floats(C.byref(self.layout), n))
        if out is not None:  # write straight into rollout-buffer rows
            action, logp, vals = out
        else:
            action = torch.empty((n, self.act_dim), dtype=torch.float32, device=self.device)
            logp = torch.empty_like(action)
            vals = torch.empty((n, self.value_dim), dtype=torch.float32, device=self.device) if (
                calculate_values and self.value_dim > 0) else None
        L.check(lib.rb200_mlp_sample(C.byref(self.layout), L.ptr(self.flat_params), self._ws(), L.ptr(states), L.ptr(noise),
                                     int(seed), int(offset), L.ptr(counter), n, L.ptr(action), L.ptr(logp),
                                     L.ptr(vals), L.ptr(work), L.stream_ptr()), "mlp_sample")
        return action, logp, vals

    def value(self, states, out=None):
        """ValueHead(states) only - bootstrap values of final observations."""
        lib = L.load()
        n = states.shape[0]
        work = self._buf("value", lib.rb200_mlp_fwd_scratch_floats(C.byref(self.layout), n))
        vals = out if out is not None else torch.empty((n, self.value_dim), dtype=torch.float32, device=self.device)
        L.check(lib.rb200_mlp_value(C.byref(self.layout), L.ptr(self.flat_params), self._ws(), L.ptr(states), n, L.ptr(vals),
                                    L.ptr(work), L.stream_ptr()), "mlp_value")
        return vals

    def predict_action_batch(self, env_obs, calculate_values=True, noise=None, seed=0, offset=0, **kwargs):
        """predict_action_batch (mlp_policy.py:296-321): returns (chunk_actions [B,C,A], result dict)."""
        states = env_obs["states"]
        action, logp, vals = self.sample(states, noise=noise, seed=seed, offset=offset,
                                         calculate_values=calculate_values)
        if vals is None:
            vals = torch.zeros((states.shape[0], 1), dtype=torch.float32, device=self.device)
        result = {"prev_logprobs": logp, "prev_values": vals,
                  "forward_inputs": {"action": action, "model_action": action, "states": states}}
        return action.reshape(-1, self.num_action_chunks, self.action_dim), result


class FlatAdamW:
    """clip_grad_norm_ + AdamW over the policy's flat buffers, decisions taken on the device.

    Semantics of FSDPModelManager.optimizer_step (fsdp_model_manager.py:429-463) on the no_shard path:
    coef = min(1, clip_grad/(norm+1e-6)); non-finite norm => the step is skipped; two lr groups.
    `grad_scale` folds the 1/world_size of the data-parallel gradient average into the same pass.
    """

    def __init__(self, policy: MLPPolicy, lr=3e-4, value_lr=3e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2,
                 clip_grad=0.5):
        self.policy = policy
        self.lr, self.value_lr, self.betas, self.eps, self.weight_decay = lr, value_lr, betas, eps, weight_decay
        self.clip_grad = float(clip_grad)
        n = policy.flat_params.numel()
        dev = policy.device
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        self.grad_sq = torch.zeros(1, dtype=torch.float64, device=dev)
        self.state = torch.zeros(4, dtype=torch.float64, device=dev)  # step, last norm, last coef, skipped
        segs = policy.lr_group_ends()
        self._ends = (C.c_int64 * len(segs))(*[e for _, e in segs])
        self._kinds = [k for k, _ in segs]
        self.lr_scale = 1.0          # LambdaLR multiplier (rlinf_b200/lr_scheduler.py), set once per run_training
        self.frozen: set = set()     # group kinds ("actor" / "critic") the next steps leave untouched
        # per-segment learning rates in device memory: a captured optimiser step follows LR schedules / warm-up
        self._lr_dev = torch.zeros(8, dtype=torch.float64, device=dev)
        self._lr_key = None

    def zero_grad(self):
        self.policy.flat_grads.zero_()

    def _segment_lrs(self):
        return [-1.0 if k in self.frozen else (self.value_lr if k == "critic" else self.lr) * self.lr_scale
                for k in self._kinds]

    def sync_lr_table(self):
        """Upload the per-segment lr table if it changed (call OUTSIDE graph capture; replays read the device copy)."""
        lrs = self._segment_lrs()
        key = tuple(lrs)
        if key != self._lr_key:
            host = torch.zeros(8, dtype=torch.float64)
            host[: len(lrs)] = torch.tensor(lrs, dtype=torch.float64)
            self._lr_dev.copy_(host)  # stream-ordered H2D of 64 bytes, only when the table changes
            self._lr_key = key

    def step(self, grad_scale: float = 1.0):
        lib = L.load()
        p = self.policy
        n = p.flat_params.numel()
        st = L.stream_ptr()
        if not torch.cuda.is_current_stream_capturing():
            self.sync_lr_table()
        L.check(lib.rb200_grad_sqnorm(L.ptr(p.flat_grads), n, L.ptr(self.grad_sq), st), "grad_sqnorm")
        L.check(lib.rb200_adamw_step_dev(L.ptr(p.flat_params), L.ptr(p.flat_grads), L.ptr(self.exp_avg),
                                         L.ptr(self.exp_avg_sq), n, self._ends, L.ptr(self._lr_dev), len(self._kinds),
                                         self.betas[0], self.betas[1], self.eps, self.weight_decay, self.clip_grad,
                                         float(grad_scale), L.ptr(self.grad_sq), L.ptr(self.state), st), "adamw_step")
        self._last_grad_scale = float(grad_scale)
        p.mark_params_changed()

    def reset_state(self, carry_grads: bool = False):
        """Fresh moments and step count: the reference REBUILDS its optimiser when critic warm-up ends
        (fsdp_model_manager.py:452-459).

        `carry_grads`: build_optimizer finishes with warmup_optimizer_state (rlinf/utils/utils.py:594-663) - one lr = 0
        step over the CURRENT `.grad` tensors (zeros only where `.grad` is None) followed by a step-count reset.  At
        the end of critic warm-up the value-head parameters still hold the clipped gradient g of the last warm-up step
        (zero_grad only runs at the start of the next global batch), so the rebuilt optimiser starts from
        exp_avg = (1-b1) g, exp_avg_sq = (1-b2) g^2 there and from zeros for the actor (grad None while frozen; the
        flat buffer holds exact zeros for it).  Pinned by tests/golden/golden_r5.npz case "warmup"."""
        self.state[0].zero_()
        if not carry_grads:
            self.exp_avg.zero_()
            self.exp_avg_sq.zero_()
            return
        # what clip_grad_norm_ left in .grad: (1/world_size average) x clip coefficient, rounded like the step kernel
        gmul = self.state[2].to(torch.float32) * getattr(self, "_last_grad_scale", 1.0)
        g = self.policy.flat_grads * gmul
        g = torch.where(self.state[3] != 0, torch.zeros_like(g), g)  # skipped (non-finite) step: plain zeros
        torch.mul(g, 1.0 - self.betas[0], out=self.exp_avg)
        torch.mul(g * g, 1.0 - self.betas[1], out=self.exp_avg_sq)

    def last_grad_norm(self) -> torch.Tensor:
        """0-dim device tensor (read it on the host once per run_training, not per step)."""
        return self.state[1]

    def lr_list(self):
        """[group["lr"] for group in optimizer.param_groups]: actor group first, then the value-head group; frozen
        groups are not part of the reference's (warm-up) optimiser."""
        lrs = []
        if "actor" not in self.frozen:
            lrs.append(self.lr * self.lr_scale)
        if "critic" in self._kinds and "critic" not in self.frozen:
            lrs.append(self.value_lr * self.lr_scale)
        return lrs
