"""ctypes binding of librlinf_b200.so (the C ABI declared in include/rlinf_b200.h).

There is NO fallback: if the shared library is missing or a call fails, the caller gets an
exception.  PyTorch is used only for device memory, streams and torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "librlinf_b200.so")

c_void_p, c_int, c_int64, c_float, c_double, c_uint64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_uint64

NUM_METRICS = 24
LOGPROB_TYPES = {"token_level": 0, "action_level": 1, "chunk_level": 2}

# metric slots (mirror of the RB200_M_* enum)
M_KEYS = {
    0: "actor/policy_loss", 1: "actor/policy_loss_abs", 2: "actor/ratio", 3: "actor/ratio_abs",
    4: "actor/clipped_ratio", 5: "actor/dual_cliped_ratio", 6: "actor/approx_kl", 7: "actor/clip_fraction",
    8: "critic/value_loss", 9: "critic/value_clip_ratio",
    10: "__sum__/_critic_explained_variance/count",
    11: "__sum__/_critic_explained_variance/returns_sum",
    12: "__sum__/_critic_explained_variance/returns_sq_sum",
    13: "__sum__/_critic_explained_variance/errors_sum",
    14: "__sum__/_critic_explained_variance/errors_sq_sum",
    15: "actor/entropy_loss", 16: "actor/total_loss", 17: "actor/token_num",
}
ACTOR_SLOTS = (0, 1, 2, 3, 4, 5, 6, 7)
CRITIC_SLOTS = (8, 9, 10, 11, 12, 13, 14)


class PpoArgs(C.Structure):
    _fields_ = [
        ("bsz", c_int64), ("C", C.c_int32), ("A", C.c_int32), ("logprob_type", C.c_int32), ("with_critic", C.c_int32),
        ("logprobs", c_void_p), ("values", c_void_p), ("entropy", c_void_p),
        ("idx", c_void_p), ("old_logprobs", c_void_p), ("advantages", c_void_p), ("returns", c_void_p),
        ("prev_values", c_void_p), ("loss_mask", c_void_p), ("loss_mask_sum", c_void_p),
        ("mask_sum_row_mod", c_int64),
        ("adv_stats", c_void_p), ("adv_norm_eps", c_float),
        ("clip_ratio_low", c_double), ("clip_ratio_high", c_double), ("clip_ratio_c", c_double),
        ("has_clip_log_ratio_min", C.c_int32), ("has_clip_log_ratio_max", C.c_int32),
        ("clip_log_ratio_min", c_double), ("clip_log_ratio_max", c_double),
        ("value_clip", c_double), ("huber_delta", c_double),
        ("max_episode_steps", C.c_int32), ("critic_warmup", C.c_int32),
        ("entropy_bonus", c_double), ("loss_scale", c_double),
        ("workspace", c_void_p),
        ("loss", c_void_p), ("metrics", c_void_p), ("d_logprobs", c_void_p), ("d_values", c_void_p),
        ("d_entropy", c_void_p),
    ]


class DppoArgs(C.Structure):
    _fields_ = [("base", PpoArgs), ("proximal_logprobs", c_void_p), ("versions", c_void_p),
                ("has_current_version", C.c_int32), ("current_version", c_double),
                ("has_behave_weight_threshold", C.c_int32), ("behave_weight_threshold", c_double)]


DM_KEYS = {
    0: "actor/policy_loss", 1: "actor/proximal_ratio", 2: "actor/clipped_proximal_ratio", 3: "actor/clip_fraction",
    4: "actor/dual_clip_fraction", 5: "actor/behav_clip_fraction", 6: "actor/proximal_approx_kl",
    7: "actor/behav_approx_kl", 8: "critic/value_loss", 9: "critic/value_clip_ratio",
    10: "__sum__/_critic_explained_variance/count", 11: "__sum__/_critic_explained_variance/returns_sum",
    12: "__sum__/_critic_explained_variance/returns_sq_sum", 13: "__sum__/_critic_explained_variance/errors_sum",
    14: "__sum__/_critic_explained_variance/errors_sq_sum",
}


class MlpLayout(C.Structure):
    _fields_ = [
        ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("value_dim", C.c_int32), ("hidden", C.c_int32),
        ("logstd", c_int64),
        ("vw0", c_int64), ("vb0", c_int64), ("vw1", c_int64), ("vb1", c_int64), ("vw2", c_int64), ("vb2", c_int64),
        ("vw3", c_int64),
        ("bw0", c_int64), ("bb0", c_int64), ("bw1", c_int64), ("bb1", c_int64), ("bw2", c_int64), ("bb2", c_int64),
        ("mw", c_int64), ("mb", c_int64), ("total", c_int64),
    ]


# name -> (restype, argtypes); every symbol include/rlinf_b200.h declares must appear here
SIGNATURES = {
    "rb200_abi_version": (c_int, []),
    "rb200_strerror": (C.c_char_p, [c_int]),
    "rb200_device_info": (c_int, [C.POINTER(c_int)] * 3),
    "rb200_launch_count": (c_uint64, []),
    "rb200_loss_mask": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "rb200_gae": (c_int, [c_void_p] * 7 + [c_int, c_int, c_double, c_double, c_void_p]),
    "rb200_normalize": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_void_p]),
    "rb200_grpo_scores": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "rb200_grpo_advantages": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p]),
    "rb200_gather_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "rb200_ppo_loss": (c_int, [C.POINTER(PpoArgs), c_void_p]),
    "rb200_decoupled_ppo_loss": (c_int, [C.POINTER(DppoArgs), c_void_p]),
    "rb200_opd_loss": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int, c_double] + [c_void_p] * 5),
    "rb200_scale": (c_int, [c_void_p, c_int64, c_float, c_void_p]),
    "rb200_scale_by": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "rb200_grad_sqnorm": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "rb200_adamw_step": (c_int, [c_void_p] * 4 + [c_int64, C.POINTER(c_int64), C.POINTER(c_double), c_int,
                                                  c_double, c_double, c_double, c_double, c_float, c_float,
                                                  c_void_p, c_void_p, c_void_p]),
    "rb200_adamw_step_dev": (c_int, [c_void_p] * 4 + [c_int64, C.POINTER(c_int64), c_void_p, c_int,
                                                      c_double, c_double, c_double, c_double, c_float, c_float,
                                                      c_void_p, c_void_p, c_void_p]),
    "rb200_mlp_layout_init": (c_int, [C.POINTER(MlpLayout), c_int, c_int, c_int, c_int]),
    "rb200_mlp_fwd_scratch_floats": (c_int64, [C.POINTER(MlpLayout), c_int64]),
    "rb200_mlp_wsplit_floats": (c_int64, [C.POINTER(MlpLayout)]),
    "rb200_mlp_prepare_weights": (c_int, [C.POINTER(MlpLayout), c_void_p, c_void_p, c_void_p]),
    "rb200_mlp_forward": (c_int, [C.POINTER(MlpLayout)] + [c_void_p] * 5 + [c_int64] + [c_void_p] * 6),
    "rb200_mlp_backward": (c_int, [C.POINTER(MlpLayout)] + [c_void_p] * 5 + [c_int64] + [c_void_p] * 7),
    "rb200_mlp_sample": (c_int, [C.POINTER(MlpLayout)] + [c_void_p] * 4 + [c_uint64, c_uint64, c_void_p, c_int64] + [c_void_p] * 5),
    "rb200_tc_gemm_h": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "rb200_tc_wgrad_h": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "rb200_tc_h_debug": (c_int, [c_void_p]),
    "rb200_rollout_fused_wt_floats": (c_int64, [C.POINTER(MlpLayout)]),
    "rb200_rollout_fused_supported": (c_int, [C.POINTER(MlpLayout), c_int]),
    "rb200_rollout_fused_prepare": (c_int, [C.POINTER(MlpLayout), c_void_p, c_void_p, c_void_p]),
    "rb200_rollout_fused": (c_int, [C.POINTER(MlpLayout)] + [c_void_p] * 19 + [c_uint64] * 3 + [c_int] * 5 +
                            [c_double] * 4 + [c_void_p]),
    "rb200_rollout_tc_supported": (c_int, [C.POINTER(MlpLayout), c_int]),
    "rb200_rollout_tc_debug": (c_int, [c_int, c_void_p]),
    "rb200_rollout_tc_pack_bytes": (c_int64, [C.POINTER(MlpLayout)]),
    "rb200_rollout_tc_prepare": (c_int, [C.POINTER(MlpLayout), c_void_p, c_void_p, c_void_p, c_void_p]),
    "rb200_rollout_tc": (c_int, [C.POINTER(MlpLayout)] + [c_void_p] * 18 + [c_uint64] * 3 + [c_int] * 5 +
                         [c_double] * 4 + [c_void_p]),
    "rb200_logits_logprob_entropy_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int,
                                                 c_int, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "rb200_logits_logprob_entropy_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int,
                                                 c_int, c_int, c_double] + [c_void_p] * 5 + [c_int64, c_int64, c_void_p]),
    "rb200_mlp_value": (c_int, [C.POINTER(MlpLayout), c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "rb200_synth_env_step": (c_int, [c_void_p] * 13 + [c_int] * 5 + [c_float] * 3 + [c_uint64, c_void_p, c_void_p]),
    "rb200_synth_env_chunk_step": (c_int, [c_void_p] * 13 + [c_int] * 6 + [c_float] * 3 + [c_uint64, c_void_p, c_void_p]),
    "rb200_bootstrap_rewards_ld": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_double, c_void_p]),
    "rb200_bootstrap_rewards": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_void_p]),
    "rb200_reward_filter": (c_int, [c_void_p] * 4 + [c_int] * 4 + [c_float, c_float, c_void_p]),
    "rb200_kl_penalty": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_void_p]),
    "rb200_masked_stats": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "rb200_counter_add": (c_int, [c_void_p, c_uint64, c_void_p]),
    "rb200_mlp_mean": (c_int, [C.POINTER(MlpLayout), c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                               c_void_p]),
    "rb200_synth_env_eval_step": (c_int, [c_void_p] * 12 + [c_int] * 7 + [c_float] * 3 + [c_uint64, c_uint64, c_void_p]),
    "rb200_eval_metrics": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "rb200_masked_moments": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "rb200_masked_normalize": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_double, c_int, c_void_p]),
    "rb200_raw_advantages": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "rb200_reinpp_returns": (c_int, [c_void_p] * 5 + [c_int, c_int, c_double, c_int, c_void_p, c_void_p]),
    "rb200_grpo_video_advantages": (c_int, [c_void_p] * 4 + [c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "rb200_grpo_dynamic_turn_advantages": (c_int, [c_void_p] * 3 + [c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "rb200_sub": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
}

_LIB: Optional[C.CDLL] = None


class Rb200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once). Raises if it has not been built: there is no CPU path."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise Rb200Error(
            f"{LIB_PATH} not found: build it with `python -m rlinf_b200.build` "
            "(nvcc, sm_100a). rlinf_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing -> loud
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


def check(code: int, what: str = "") -> None:
    if code == 0:
        return
    msg = load().rb200_strerror(code).decode()
    if code < 0:
        raise ValueError(f"rlinf_b200 {what}: {msg} (code {code})")
    raise Rb200Error(f"rlinf_b200 {what}: CUDA error {code}: {msg}")


def ptr(t: Optional[torch.Tensor]):
    """Device pointer of a CUDA tensor (None -> NULL). The tensor must be contiguous."""
    if t is None:
        return None
    if not t.is_cuda:
        raise Rb200Error("rlinf_b200 kernels take CUDA tensors; move inputs with to_device() first")
    if not t.is_contiguous():
        raise Rb200Error("rlinf_b200 kernels take contiguous tensors")
    return c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def default_device() -> torch.device:
    if not torch.cuda.is_available():
        raise Rb200Error("rlinf_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def to_device(t: Optional[torch.Tensor], device=None, dtype=None) -> Optional[torch.Tensor]:
    """H2D copy of a (possibly CPU) tensor: the reference's embodied rollout batch lives on the host
    (rlinf/data/schema/embodied_types.py:297-311); compute never happens on the host here."""
    if t is None:
        return None
    device = device or default_device()
    if t.device != device:
        t = t.to(device, non_blocking=True)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def as_u8(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    """bool -> uint8 view (no copy)."""
    if t is None:
        return None
    if t.dtype == torch.bool:
        return t.view(torch.uint8)
    if t.dtype != torch.uint8:
        return (t != 0).view(torch.uint8)
    return t
