#!/usr/bin/env python
"""Benchmark of the hot path: env-steps/sec (rollout + PPO update) on the synthetic workload.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (default N=1)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle port)

One "step" = one runner iteration: T-step rollout of B envs on the device + advantages + the full PPO
update (update_epoch x mini-batches, fused loss, backward, clip+AdamW) = B*T env-steps.
Workload = BASELINE.json configs[1]: synthetic vector env obs_dim=128 act_dim=8, MLP policy, PPO,
B=4096 T=512; hyper-parameters of examples/embodiment/config/maniskill_ppo_mlp.yaml.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (rollout+update)"
UNIT = "env-steps/s"


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--T", type=int, default=512)
    ap.add_argument("--obs", type=int, default=128)
    ap.add_argument("--act", type=int, default=8)
    ap.add_argument("--update-epoch", type=int, default=8)
    ap.add_argument("--minibatches", type=int, default=8)
    ap.add_argument("--cpu-envs", type=int, default=0,
                    help="envs in the bounded CPU sample (0 = 512 for cpu_baseline, 256 for --impl reference)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-bench", action="store_true")
    ap.add_argument("--debug-flags", type=int, default=0,
                    help="rb200_debug_set_flags value (experimental kernel variants; 0 = shipped kernels)")
    ap.add_argument("--graph-update", action="store_true",
                    help="experimental: replay one CUDA graph per optimiser step (actor.cuda_graph_update)")
    ap.add_argument("--rollout", default="auto", choices=["auto", "tc", "fused", "graph"],
                    help="rollout implementation: persistent fused kernel, per-kernel CUDA graph, or the library default")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return a


def workload_name(a):
    return (f"synthetic vector env obs_dim={a.obs} act_dim={a.act}, MLP policy, PPO, B={a.B} T={a.T} "
            f"(BASELINE configs[1]), update_epoch={a.update_epoch}, {a.minibatches} mini-batches/epoch")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self._halt = gpu_index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu_index)], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 8:
                    self.rows.append(f)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[1]) for r in self.rows)
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][2]), "reasons": sorted(reasons),
                "samples": len(self.rows), "power_w_max": max(float(r[3]) for r in self.rows)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's CPU path, on the host cores
# ------------------------------------------------------------------------------------------------
def effective_cores() -> int:
    """Host cores this process may actually use: min(visible CPUs, affinity mask, cgroup CPU quota).
    (The GPU boxes show 128 CPUs but cap the container at 16 via cpu.max; 128 threads on 16 cores is
    ~50x slower than 16 threads.)"""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return max(1, n)


_BEST_THREADS = None


def best_thread_count(a) -> int:
    """The oracle's eager-PyTorch ops on [4096]-element rows do not scale with threads (round 1: 20.2 k env-steps/s with
    16 threads on a 16-core box, 12.3 k with 96 threads on a 96-core box): time one small iteration per candidate thread
    count and keep the fastest, so the baseline is the best the host can do."""
    global _BEST_THREADS
    if _BEST_THREADS is not None:
        return _BEST_THREADS
    import torch

    from oracle.runner_oracle import RunnerOracle
    from rlinf_b200.config import synthetic_ppo_config

    cores = effective_cores()
    cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores})
    best, best_t = cores, float("inf")
    for c in cands:
        torch.set_num_threads(c)
        cfg = synthetic_ppo_config(B=512, T=64, obs_dim=a.obs, action_dim=a.act, update_epoch=1, num_minibatches=2)
        r = RunnerOracle(cfg)
        r.run_iteration()
        t0 = time.perf_counter()
        r.run_iteration()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    log(f"cpu thread calibration: {cands} -> {best} threads")
    _BEST_THREADS = best
    return best


def cpu_iteration_rate(a, n_envs, steps, warmup):
    import torch

    from oracle.runner_oracle import RunnerOracle
    from rlinf_b200.config import synthetic_ppo_config

    cores = best_thread_count(a)
    torch.set_num_threads(cores)
    cfg = synthetic_ppo_config(B=n_envs, T=a.T, obs_dim=a.obs, action_dim=a.act, update_epoch=a.update_epoch,
                               num_minibatches=a.minibatches)
    r = RunnerOracle(cfg)
    times, timers = [], []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        r.run_iteration()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
            timers.append(dict(r.timers))
    mean = sum(times) / len(times)
    phases = {k: sum(t[k] for t in timers) / len(timers) for k in timers[0]}
    return n_envs * a.T / mean, mean, cores, phases


def reference_functions_check(a):
    """When /root/reference exists (build container only - never on the GPU box): time the reference's OWN
    calculate_adv_and_returns (GAE) and policy_loss (actor_critic, forward + backward) through tests/golden/ref_loader.py
    beside the oracle port on the same inputs, to show port ~= reference. Returns None when the reference is absent."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        import ref_loader

        if not ref_loader.reference_available():
            return None
        ref = ref_loader.load_reference()
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)}
    import torch

    from oracle import rl_oracle as O

    T, B, A = a.T, min(a.B, 512), a.act
    g = torch.Generator().manual_seed(0)
    rewards, values = torch.randn(T, B, 1, generator=g), torch.randn(T + 1, B, 1, generator=g)
    dones = torch.rand(T + 1, B, 1, generator=g) < 0.01
    dones[0] = False
    n = T * B
    old = -1 + 0.3 * torch.randn(n, A, generator=g)
    adv, ret, pv = (torch.randn(n, 1, generator=g) for _ in range(3))

    def timed(fn, reps=3):
        fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t0) / reps

    def ref_adv():
        return ref.registry.calculate_adv_and_returns(task_type="embodied", adv_type="gae", rewards=rewards, dones=dones,
                                                      values=values, gamma=0.99, gae_lambda=0.95, group_size=8,
                                                      reward_type="action_level", num_action_chunks=1, loss_mask=None,
                                                      loss_mask_sum=None)

    def port_adv():
        return O.adv_and_returns_embodied("gae", rewards, dones, values, gamma=0.99, gae_lambda=0.95)

    def loss_inputs():
        new = (old + 0.05 * torch.randn(n, A, generator=g)).requires_grad_(True)
        val = (pv + 0.1 * torch.randn(n, 1, generator=g)).requires_grad_(True)
        return new, val

    def ref_loss():
        new, val = loss_inputs()
        loss, _ = ref.registry.policy_loss(task_type="embodied", loss_type="actor_critic", logprob_type="action_level",
                                           reward_type="action_level", single_action_dim=A, logprobs=new, values=val,
                                           old_logprobs=old, advantages=adv, returns=ret, prev_values=pv,
                                           clip_ratio_high=0.2, clip_ratio_low=0.2, value_clip=0.2, huber_delta=10.0,
                                           loss_mask=None, loss_mask_sum=None, max_episode_steps=128, critic_warmup=False)
        loss.backward()

    def port_loss():
        new, val = loss_inputs()
        loss, _ = O.policy_loss_embodied("actor_critic", new, old, adv, "action_level", A, values=val, prev_values=pv,
                                         returns=ret, clip_ratio_low=0.2, clip_ratio_high=0.2, value_clip=0.2,
                                         huber_delta=10.0)
        loss.backward()

    return {"shape": f"T={T} B={B} A={A}", "gae_s": {"reference": timed(ref_adv), "port": timed(port_adv)},
            "loss_fwd_bwd_s": {"reference": timed(ref_loss), "port": timed(port_loss)}}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # 1. a small sample (warm caches, estimate the rate), 2. as many FULL-size iterations as fit the time budget
    #    (4096 envs x 512 steps is ~2 min per iteration on 16 cores): `same config` as the GPU arm whenever >= 1 fits
    small = min(a.cpu_envs or 256, a.B)
    v_small, mean_small, cores, phases = cpu_iteration_rate(a, small, 1, max(1, min(a.warmup, 1)))
    budget_s = float(os.environ.get("RB200_REF_BUDGET_S", "240"))
    est_full = a.B * a.T / v_small
    n_full = int(min(a.steps, budget_s // est_full)) if not a.cpu_envs else 0
    if n_full >= 1:
        value, mean_s, cores, phases = cpu_iteration_rate(a, a.B, n_full, 0)
        sample = (f"FULL workload: {n_full} iteration(s) of {a.B} envs x T={a.T} (of --steps {a.steps}: bounded by a "
                  f"{budget_s:.0f} s budget), after a {small}-env warm-up iteration; oracle port of the reference CPU path, "
                  f"torch {cores} threads (fastest of a calibration over thread counts; usable host cores: "
                  f"{effective_cores()}); the reference's own Ray runner cannot be launched offline")
        n_envs = a.B
    else:
        n_envs = small
        value, mean_s, cores, phases = cpu_iteration_rate(a, n_envs, a.steps, a.warmup)
        sample = (f"{n_envs} of {a.B} envs x T={a.T} per step (same update_epoch/mini-batch structure); "
                  f"oracle port of the reference CPU path (torch {cores} threads, fastest of a calibration; usable host "
                  f"cores: {effective_cores()}); the reference's own Ray runner cannot be launched offline")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": mean_s * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "B": a.B, "T": a.T, "obs_dim": a.obs, "act_dim": a.act},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "phases_s": phases, "envs_timed": n_envs},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    chk = reference_functions_check(a)
    if chk is not None:
        line["cpu_baseline"]["port_vs_reference_functions"] = chk
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures
# (profiles/r01_ncu_mlp_step_v3_table.txt, profiles/r01_ncu_gae_v4_summary.txt); only valid at the captured shape.
NCU_TRAFFIC = {
    # profiles/r02_ncu_final_table.txt (ncu --set full, per launch; GEMMs: grouped two-tower launches at 262144 rows, per tower = half)
    ("tc_gemm_fwd", 262144): (537.4e6 + 484.0e6) / 2,   # 268.7 MB read + 242.0 MB written back before the kernel ends
    ("tc_wgrad", 262144): (1074.6e6 + 4.5e6) / 2,
    ("gae_scan", 512, 4096): 18.9e6,    # reads only: the 16.8 MB of results are still in L2 when the kernel ends
    ("ppo", 262144): 64.4e6 + 3.0e6,    # 2x the algorithmic 32.5 MB: every gathered 4-byte scalar pulls a 32-byte sector
    ("logits_fwd", 4096, 32000): 524.6e6 + 3.7e6,
    ("logits_bwd", 4096, 32000): 524.5e6 + 478.7e6,
}


def kernel_rooflines(a, peaks, torch):
    """Live CUDA-event timing of the HBM-bound kernels at the workload's shapes. Each kernel is launched
    from a captured CUDA graph over ROT independent input sets whose total size exceeds L2 (126 MB), so
    every launch streams from HBM; per-launch time = graph time / launches (includes inter-kernel gaps)."""
    from rlinf_b200 import ops

    dev = torch.device("cuda")
    T, B, A = a.T, a.B // max(a.gpus, 1), a.act
    out = {}

    def time_graph(fn, n_launch, reps=5):
        fn()  # warm (allocations, descriptor encode)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = []
        for _ in range(reps):
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            best.append(e0.elapsed_time(e1) * 1e-3 / n_launch)
        best.sort()
        return best[len(best) // 2]

    # ---- GAE scan: 17 B/step + bootstrap row ----
    bytes_gae = 17 * T * B + 5 * B
    rot = max(2, int(300e6 // bytes_gae) + 1)
    sets = []
    for i in range(rot):
        r = torch.randn(T, B, device=dev)
        v = torch.randn(T + 1, B, device=dev)
        d = (torch.rand(T + 1, B, device=dev) < 0.01).view(torch.uint8)
        sets.append((r, v, d, torch.empty(T, B, device=dev), torch.empty(T, B, device=dev),
                     torch.empty(6, dtype=torch.float64, device=dev)))
    from rlinf_b200 import _lib as L
    lib = L.load()

    def gae_all():
        for (r, v, d, ad, rt, stt) in sets:
            L.check(lib.rb200_gae(L.ptr(r), L.ptr(v), L.ptr(d), None, L.ptr(ad), L.ptr(rt), L.ptr(stt), T, B, 0.99,
                                  0.95, L.stream_ptr()), "gae")

    t = time_graph(gae_all, rot)
    out["gae_scan"] = {"bound": "hbm", "achieved": bytes_gae / t / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                       "frac": bytes_gae / t / 1e9 / peaks["hbm_gbs"], "traffic": NCU_TRAFFIC.get(("gae_scan", T, B)),
                       "us_per_launch": t * 1e6,
                       "algorithmic_bytes": bytes_gae, "launch_note": "includes the 48-byte stats memset node"}
    del sets

    # ---- fused gather + PPO loss fwd+bwd on one mini-batch: 124 B/sample ----
    n_all = T * B
    mb = n_all // a.minibatches
    bytes_ppo = (8 + 4 * A + 4 * A + 16 + 4 * A + 4) * mb
    old = torch.randn(n_all, A, device=dev) * 0.3 - 1
    adv, ret, pv = (torch.randn(n_all, 1, device=dev) for _ in range(3))
    perm = torch.randperm(n_all, device=dev)
    rot = max(2, int(300e6 // bytes_ppo) + 1)
    cur = [(torch.randn(mb, A, device=dev) * 0.3 - 1, torch.randn(mb, 1, device=dev)) for _ in range(rot)]
    idxs = [perm[(i * mb) % n_all:][:mb].contiguous() for i in range(rot)]

    def ppo_all():
        for (lp, vv), ix in zip(cur, idxs):
            ops.ppo_loss(logprobs=lp, values=vv, old_logprobs=old, advantages=adv, returns=ret, prev_values=pv,
                         idx=ix, C_chunks=1, A_dim=A, logprob_type="action_level", value_clip=1.0, huber_delta=10.0)

    t = time_graph(ppo_all, rot)
    out["gather_ppo_loss_fwd_bwd"] = {"bound": "hbm", "achieved": bytes_ppo / t / 1e9, "peak": peaks["hbm_gbs"],
                                      "unit": "GB/s", "frac": bytes_ppo / t / 1e9 / peaks["hbm_gbs"],
                                      "traffic": NCU_TRAFFIC.get(("ppo", mb)),
                                      "us_per_launch": t * 1e6, "algorithmic_bytes": bytes_ppo,
                                      "launch_note": "ONE kernel (the last CTA finalises and clears the workspace); rollout rows gathered "
                                                     "through idx: each gathered 4-byte scalar pulls a 32-byte sector"}
    del cur, idxs, old, adv, ret, pv, perm

    # ---- logits -> logprob / entropy (SURVEY 8(f)3), vocabulary-sized rows: N*V*4 bytes forward, 2x backward ----
    Nl, V = 4096, 32000  # 524 MB of fp32 logits: every launch streams from HBM
    lg = torch.randn(Nl, V, device=dev)
    dlg = torch.empty_like(lg)
    tg = torch.randint(0, V, (Nl,), device=dev)
    lpo, eno, lso = (torch.empty(Nl, device=dev) for _ in range(3))
    g1, g2 = torch.randn(Nl, device=dev), torch.randn(Nl, device=dev)

    def lg_fwd():
        L.check(lib.rb200_logits_logprob_entropy_fwd(L.ptr(lg), 0, L.ptr(tg), Nl, Nl, 0, V, V, 0, V, 1.25, L.ptr(lpo),
                                                     L.ptr(eno), L.ptr(lso), L.stream_ptr()), "logits_fwd")

    def lg_bwd():
        L.check(lib.rb200_logits_logprob_entropy_bwd(L.ptr(lg), 0, L.ptr(tg), Nl, Nl, 0, V, V, 0, V, 1.25, L.ptr(lso),
                                                     L.ptr(eno), L.ptr(g1), L.ptr(g2), L.ptr(dlg), 0, V,
                                                     L.stream_ptr()), "logits_bwd")

    lg_fwd()
    for key, fn, nbytes in (("logits_logprob_entropy_fwd", lg_fwd, Nl * V * 4), ("logits_logprob_entropy_bwd", lg_bwd, 2 * Nl * V * 4)):
        t = time_graph(fn, 1)
        out[key] = {"bound": "hbm", "achieved": nbytes / t / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": nbytes / t / 1e9 / peaks["hbm_gbs"],
                    "traffic": NCU_TRAFFIC.get(("logits_fwd" if key.endswith("fwd") else "logits_bwd", Nl, V)),
                    "us_per_launch": t * 1e6,
                    "algorithmic_bytes": nbytes, "rows": Nl, "vocab": V}
    del lg, dlg

    # ---- tcgen05 fp16-split GEMMs of the MLP towers at the mini-batch shape (the shipped kernels, csrc/tc_gemm_h.cu) ----
    n = mb
    K = 256
    Amat = torch.randn(n, K, device=dev)
    Wmat = torch.randn(256, K, device=dev) / 16
    Cmat = torch.empty(n, 256, device=dev)
    wk = torch.empty(512 * K, device=dev)
    Z = torch.randn(n, 256, device=dev) / 64
    dW = torch.zeros(256, K, device=dev)
    reps_k = 4  # n*K*4 = 268 MB per operand at the headline shape: every launch streams from HBM

    def gemm_all():
        for _ in range(reps_k):
            L.check(lib.rb200_tc_gemm_h(L.ptr(Amat), L.ptr(Wmat), L.ptr(Cmat), n, K, 0, None, L.ptr(wk), L.stream_ptr()),
                    "tc_gemm_h")

    def wgrad_all():
        for _ in range(reps_k):
            L.check(lib.rb200_tc_wgrad_h(L.ptr(Z), L.ptr(Amat), L.ptr(dW), n, K, None, L.stream_ptr()), "tc_wgrad_h")

    flops = 2.0 * n * 256 * K
    ceiling = peaks["bf16_tflops"] / 3.0
    bytes_gemm = n * K * 4 + n * 256 * 4
    for key, fn, note in (("tc_gemm_fwd", gemm_all, "C[n,256] = A[n,256] . W^T, plain fp32 in/out; launch includes the 3 us "
                                                    "weight-split kernel of the unit-test entry"),
                          ("tc_wgrad", wgrad_all, "dW[256,256] += Z[n,256]^T . H[n,256], per-chunk partials added to dW in a fixed order")):
        t = time_graph(fn, reps_k)
        out[key] = {"bound": "hbm", "achieved": bytes_gemm / t / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": bytes_gemm / t / 1e9 / peaks["hbm_gbs"],
                    "tensor_tflops": flops / t / 1e12, "frac_of_fp16_split_ceiling": flops / t / 1e12 / ceiling,
                    "traffic": NCU_TRAFFIC.get((key, n)), "us_per_launch": t * 1e6, "algorithmic_flops": flops,
                    "algorithmic_bytes": bytes_gemm, "rows": n, "note": note}
    return out


def _update_phase_bytes(n, obs, act, H):
    """Algorithmic HBM bytes of ONE pass of the update over n samples (fp32; U = n*H*4 bytes = one [n,256] tensor):
    forward: per tower read X (obs) + write H1 | read H1 write H2 | read H2 write H3; heads read H3, G3;
    backward: heads read H3,G3 write dZ3 (both towers); per tower wgrad2 (dZ3,H2), dgrad2 (dZ3,H2 -> dZ2), wgrad1 (dZ2,H1),
    dgrad1 (dZ2,H1 -> dZ1), wgrad0 (dZ1,X); loss / optimiser / small [n,act] tensors are < 1 %."""
    U = n * H * 4
    X = n * obs * 4
    fwd = 2 * (X + U + 2 * U + 2 * U) + 2 * U
    bwd = 4 * U + 2 * (2 * U + 3 * U + 2 * U + 3 * U + (U + X))
    return fwd + bwd


DUMP_BYTES = 64 << 20
DUMP_METRIC_BYTES = 4096  # room kept for the float64 metrics, whose number is known only after the first update


def dump_plan(out_dir, run):
    """The fixed, seeded sample --dump-outputs writes (see dump_outputs), checked against DUMP_BYTES before the benchmark
    runs: env columns of the [T(+1), B, ...] rollout batch and rows of the [T*B, 1] training batch."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    rollout = dict(run.buffer.as_batch())
    rollout.update(rollout.pop("forward_inputs"))
    B, T = run.buffer.B, run.buffer.T
    col_bytes = sum(v[:, 0].numel() * 4 for v in rollout.values())
    n_cols = max(1, min(B, (DUMP_BYTES // 2) // col_bytes))
    n_rows = min(T * B, n_cols * T)
    nbytes = n_cols * col_bytes + 2 * n_rows * 4 + run.actor.model.flat_params.numel() * 4
    if nbytes + DUMP_METRIC_BYTES > DUMP_BYTES:
        raise ValueError(f"--dump-outputs: {nbytes} bytes exceed the {DUMP_BYTES}-byte limit at this shape")
    g = torch.Generator().manual_seed(0)
    dev = run.buffer.rewards.device
    cols = torch.randperm(B, generator=g)[:n_cols].sort().values.to(dev)
    rows = torch.randperm(T * B, generator=g)[:n_rows].sort().values.to(dev)
    return cols, rows


def dump_outputs(out_dir, run, metrics, plan):
    """Write what the last timed step computed to out_dir/<name>.npy, so that two builds run with the same arguments
    (hence the same seeded inputs) can be compared output for output:
      rollout.<key>   the rollout batch the actor consumed ([T(+1), B, ...]), on a fixed, seeded sample of environments
      train.<key>     advantages / returns of the shuffled training batch ([T*B, 1]), on a fixed, seeded sample of rows
      param.<name>    every policy parameter after the update
      metric.<key>    the training metrics the step returned ('/' in a key becomes '.')
    Float tensors are written as float32, flags as float32 0/1, metrics as float64; at most DUMP_BYTES in all."""
    import numpy as np
    import torch

    cols, rows = plan
    rollout = dict(run.buffer.as_batch())
    rollout.update(rollout.pop("forward_inputs"))
    out = {f"rollout.{k}": v.index_select(1, cols) for k, v in rollout.items()}
    out.update({f"train.{k}": run.actor.rollout_batch[k].index_select(0, rows) for k in ("advantages", "returns")})
    out.update({f"param.{n}": p for n, p in run.actor.model.named_parameters()})
    arrays = {k: v.detach().to(torch.float32).cpu().numpy() for k, v in out.items()}
    arrays.update({f"metric.{k.replace('/', '.')}": np.asarray(v, dtype=np.float64) for k, v in metrics.items()})
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte limit at this shape")
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    log(f"dumped {len(arrays)} arrays ({total / 1e6:.1f} MB) to {out_dir}")


def run_ours(a):
    # ONE JSON line on stdout: anything a library prints at the C level (NCCL's "NCCL version ..." line) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == a.gpus or world == 1, f"--gpus {a.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from rlinf_b200 import _lib as L
    from rlinf_b200.config import synthetic_ppo_config
    from rlinf_b200.runner import EmbodiedRunner

    lib = L.load()
    if a.debug_flags:
        lib.rb200_debug_set_flags(int(a.debug_flags))
    peaks = measured_peaks()
    over = {} if a.rollout == "auto" else {"rollout.fused_kernel": {"tc": "tc", "fused": True, "graph": False}[a.rollout]}
    if a.graph_update:
        over["actor.cuda_graph_update"] = True
    cfg = synthetic_ppo_config(B=a.B, T=a.T, obs_dim=a.obs, action_dim=a.act, update_epoch=a.update_epoch,
                               num_minibatches=a.minibatches, world_size=world, **over)
    run = EmbodiedRunner(cfg)
    plan = dump_plan(a.dump_outputs, run) if a.dump_outputs and rank == 0 else None
    n_env_steps = a.B * a.T

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # graph capture of the rollout happens on the 2nd call: make sure warm-up covers it
    warm = max(a.warmup, 3)
    for i in range(warm):
        t0 = time.perf_counter()
        run.run_iteration()
        torch.cuda.synchronize()
        log(f"warm-up iteration {i}: {time.perf_counter() - t0:.3f}s")
    barrier()

    # ---- device-resident timing (value) ----
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * a.steps + 1)]
    launches0 = lib.rb200_launch_count()
    graph_nodes = run.rollout.graph_kernel_count
    barrier()
    torch.cuda.cudart().cudaProfilerStart()  # `ncu --profile-from-start off` captures the timed region only
    t_wall0 = time.perf_counter()
    ev[0].record()
    metrics = None
    for i in range(a.steps):
        run.update_rollout_weights()
        run.rollout_phase()
        ev[3 * i + 1].record()
        metrics = run.update_phase()
        ev[3 * i + 3].record()
    barrier()
    torch.cuda.cudart().cudaProfilerStop()
    t_wall = time.perf_counter() - t_wall0
    total_ms = ev[0].elapsed_time(ev[3 * a.steps])
    log(f"timed {a.steps} steps: {total_ms:.1f} ms")
    rollout_ms = sum((ev[3 * i].elapsed_time(ev[3 * i + 1])) for i in range(a.steps)) / a.steps
    launches = lib.rb200_launch_count() - launches0 + graph_nodes * a.steps
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / a.steps
    value = n_env_steps / (ms_per_step * 1e-3)
    if a.dump_outputs and rank == 0:  # before the end-to-end steps below move the state on
        dump_outputs(a.dump_outputs, run, metrics, plan)

    # ---- end to end through the public API with HOST buffers (the reference hands the actor CPU tensors) ----
    def pin(d):
        return {k: (pin(v) if isinstance(v, dict) else torch.empty(v.shape, dtype=v.dtype).pin_memory())
                for k, v in d.items()}

    host = pin(run.buffer.as_batch())

    def nbytes(d):
        return sum(nbytes(v) if isinstance(v, dict) else v.numel() * v.element_size() for v in d.values())

    def d2h(src, dst):
        for k, v in src.items():
            if isinstance(v, dict):
                d2h(v, dst[k])
            else:
                dst[k].copy_(v, non_blocking=True)

    bytes_batch = nbytes(host)
    for _ in range(1):
        run.rollout_phase()
        d2h(run.buffer.as_batch(), host)
        torch.cuda.synchronize()
        run.update_phase(batch=host)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    e2e_steps = max(1, min(a.steps, 3))
    for _ in range(e2e_steps):
        run.update_rollout_weights()
        run.rollout_phase()
        d2h(run.buffer.as_batch(), host)           # rollout side -> host (what the reference's workers exchange)
        torch.cuda.synchronize()
        m = run.update_phase(batch=host)            # actor: H2D of the batch, advantages, update, metrics D2H
    e1.record()
    barrier()
    e2e_s = max(time.perf_counter() - t0, e0.elapsed_time(e1) * 1e-3)
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = n_env_steps * e2e_steps / float(t.item())
    log(f"e2e {e2e_steps} steps: {float(t.item()):.3f}s")
    metrics_bytes = 8 * 32

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": warm,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "B": a.B, "T": a.T, "obs_dim": a.obs, "act_dim": a.act,
                   "global_batch_size": cfg.actor.global_batch_size, "micro_batch_size": cfg.actor.micro_batch_size,
                   "parallelism": f"dp{a.gpus} over envs, 1 NCCL all-reduce of the flat grad buffer / optimiser step",
                   "l2": "per-step inputs (1.2 GB rollout batch / rank share) exceed the 126 MB L2; kernel "
                         "micro-timings rotate >300 MB of inputs"},
        "phases_ms": {"rollout": rollout_ms, "update": ms_per_step - rollout_ms},
        "wall_ms_per_step": t_wall / a.steps * 1e3,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": bytes_batch,
                "d2h_bytes_per_step": bytes_batch + metrics_bytes,
                "note": "rollout batch staged through pinned host memory both ways, as between the reference's "
                        "rollout/env workers and its actor"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "train_metrics": {k: v for k, v in (metrics or {}).items()},
    }
    if rank == 0:
        # dominant kernel by time: the fp32 MLP GEMMs (forward, dgrad, wgrad) - flops known analytically
        n = a.B * a.T // world
        H, O, A = 256, a.obs, a.act
        fwd = 2 * (O * H + 2 * H * H) * 2          # two towers
        bwd = 2 * (O * H + 2 * H * H) * 2 + 2 * (2 * H * H) * 2  # wgrad (3 layers) + dgrad (2 layers), two towers
        flops_update = (fwd + bwd) * n * a.update_epoch
        upd_s = (ms_per_step - rollout_ms) * 1e-3
        ceiling = peaks["bf16_tflops_sustained"] / 3.0  # fp32-accurate product = 3 kind::f16 MMAs
        bytes_update = _update_phase_bytes(n, O, A, H) * a.update_epoch
        line["roofline"] = {
            "kernel": "whole update phase (tc_h_gemm_kernel / tc_h_wgrad_kernel fp16-split tcgen05 GEMMs + heads + loss + AdamW)",
            "bound": "hbm", "achieved": bytes_update / upd_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": bytes_update / upd_s / 1e9 / peaks["hbm_gbs"], "traffic": None,
            "algorithmic_bytes": bytes_update, "tensor_tflops": flops_update / upd_s / 1e12,
            "frac_of_fp16_split_ceiling": flops_update / upd_s / 1e12 / ceiling,
            "note": "algorithmic HBM bytes of the update phase (fp32 activations / gradients read and written once per GEMM, "
                    "DESIGN.md section 4) / update time; the fp32 [n,256] activation traffic, not the tensor pipe, bounds it"}
        if not a.no_kernel_bench:
            log("kernel rooflines ...")
            try:
                kr = kernel_rooflines(a, peaks, torch)
                g = kr.pop("tc_gemm_fwd")
                w = kr.pop("tc_wgrad")
                line["roofline_update_phase"] = line["roofline"]
                # dominant kernel of the step, timed alone with CUDA events
                line["roofline"] = {
                    "kernel": "rb::tch::tc_h_gemm_kernel (tcgen05 kind::f16, 2-way fp16 split = fp32-accurate GEMM of the MLP "
                              "towers; forward/dgrad), mini-batch shape, one tower",
                    "bound": "hbm", "achieved": g["achieved"], "peak": g["peak"], "unit": "GB/s", "frac": g["frac"],
                    "traffic": g["traffic"], "algorithmic_bytes": g["algorithmic_bytes"],
                    "tensor_tflops": g["tensor_tflops"], "frac_of_fp16_split_ceiling": g["frac_of_fp16_split_ceiling"],
                    "us_per_launch": g["us_per_launch"], "algorithmic_flops": g["algorithmic_flops"],
                    "note": "achieved = algorithmic bytes (A [n,256] fp32 read + C [n,256] fp32 written) / live CUDA-event time "
                            "per launch; peak = measured HBM copy bandwidth.  2*n*256*256 flops over 2 KB per row = 64 "
                            "flop/B: at 3 kind::f16 MMAs per product the tensor time (peak/3) is below the HBM time of the "
                            "fp32 operands, so HBM bounds the kernel (DESIGN.md section 4). " + g["note"]}
                line["roofline_tc_wgrad"] = w
                line["roofline_hbm_kernels"] = kr
            except Exception as e:  # pragma: no cover
                line["roofline_hbm_kernels"] = {"error": repr(e)}
        if not a.no_cpu_baseline and world == 1:
            n_envs = min(a.cpu_envs or 512, a.B)
            log("cpu baseline ...")
            v, mean_s, cores, phases = cpu_iteration_rate(a, n_envs, 1, 1)
            log(f"cpu baseline iteration {mean_s:.2f}s {phases}")
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"1 iteration of {n_envs} of {a.B} envs x T={a.T}, same update structure; "
                                              f"oracle port of the reference CPU path, torch {cores} threads",
                                    "seconds": mean_s, "phases_s": phases}
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
