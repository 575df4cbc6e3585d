// Persistent fused rollout: the whole T-step actor/critic inference + synthetic-env loop of one rank in ONE kernel.
//
// Reference loop replaced: EnvWorker.interact / MultiStepRolloutWorker.generate (rlinf/workers/env/env_worker.py:
// 1059-1349, rlinf/workers/rollout/hf/huggingface_worker.py:678-781) for the MLP policy
// (models/embodiment/mlp_policy/mlp_policy.py:256-321) with the device-resident synthetic env (rollout.cu).
//
// Environments are independent for the whole rollout and the policy is frozen, so nothing has to cross SMs: CTA c owns
// environments [c*E, c*E+E) for all T steps (E = ceil(B / #SM) <= 32) and keeps their observation and every
// activation in shared memory.  Per step and CTA: 3+3 hidden layers (thread j = hidden unit j, all E environments in
// registers, weights streamed from L2 as transposed [in][256] rows -> one coalesced 1 KB load per input feature), the
// fused heads (Normal sample with Philox or supplied noise, log-prob, value), the env dynamics (s.W_s + a.W_a, tanh,
// reward, termination / truncation, auto-reset) and the truncation bootstrap r += gamma * V(final_obs), which needs
// an extra value-tower pass only in steps where one of the CTA's environments was flagged.
// The graph version of the same loop (rollout.py) launches ~16 kernels per step, each with B/128 tiles on 148 SMs:
// 105 us / step at B = 4096 and hardly less at B = 512 (8-GPU strong scaling); here a step costs E * 346k FMA per SM
// (B = 4096: E = 28) or the 1.3 MB weight stream from L2 (small E).
// Same random streams as the per-kernel path: policy Philox(seed_p, row*act + a, offset + c_p + t), env
// Philox(seed_e, row*32 + lane, (c_e + t) * 64) with the same draw order, so both paths generate the same episode
// up to fp32 summation order.
#include <curand_kernel.h>

#include "common.cuh"

namespace {

constexpr int kH = 256;
constexpr int kThreads = 256;
constexpr int kMaxAct = 32;
constexpr float kHalfLog2Pi = 0.91893853320467274178f;

struct FusedArgs {
  rb200_mlp_layout L;
  const float* params;   // flat fp32 parameters
  const float* wt;       // transposed hidden weights (rb200_rollout_fused_prepare)
  const float* w_s;      // [obs, obs]  ([in][out])
  const float* w_a;      // [act, obs]
  float* states;         // [T+1, B, obs]   row 0 = current observation (in), rows 1..T written
  float* actions;        // [T, B, act]
  float* logp;           // [T, B, act]
  float* values;         // [T+1, B, vdim]
  float* rewards;        // [T, B]
  uint8_t* term;         // [T+1, B]  rows 1..T written
  uint8_t* trunc;
  uint8_t* done;
  float* final_obs;      // [B, obs]   observation before the auto-reset of the LAST step (contract parity)
  float* final_values;   // [B]        V(final_obs) of the last flagged step (scratch, contract parity)
  int32_t* elapsed;      // [B] in/out
  const float* policy_noise;  // [T, B, act] or null
  const float* env_noise;     // [T, B, 2*obs+2] or null
  const uint64_t* counter_p;  // device step counters (read once; the caller adds T afterwards)
  const uint64_t* counter_e;
  uint64_t seed_p, seed_e, offset_p;
  int T, B, E, obs, act, vdim;
  int max_episode_steps, auto_reset, bootstrap_on_done;
  float gamma, p_term, noise_std, reward_noise_std;
};

__device__ __forceinline__ float tanh_fast(float x) {  // same formula as the tensor-core epilogue (tc_gemm_h.cu)
  const float t = __expf(-2.0f * fabsf(x));
  return copysignf(__fdividef(1.0f - t, 1.0f + t), x);
}

// out[e][j] = tanh(sum_k in[e][k] * Wt[k][j] + bias[j]) for the CTA's EMAX environment slots; thread j = column j.
// Wt rows are 1 KB coalesced loads (L2 resident), double-buffered in registers; in[e][k..k+3] are broadcast LDS.128.
// This one-k-step prefetch and its tiled twin below serve the K that the pipelined layers cannot (K % 16 != 0).
template <int EMAX>
__device__ __forceinline__ void layer(const float* __restrict__ in_s, int K, const float* __restrict__ Wt,
                                      const float* __restrict__ bias, float* __restrict__ out_s, int j) {
  float acc[EMAX];
#pragma unroll
  for (int e = 0; e < EMAX; ++e) acc[e] = 0.f;
  float w0 = __ldg(Wt + 0 * kH + j), w1 = __ldg(Wt + 1 * kH + j), w2 = __ldg(Wt + 2 * kH + j),
        w3 = __ldg(Wt + 3 * kH + j);
  for (int k = 0; k < K; k += 4) {
    float n0 = 0.f, n1 = 0.f, n2 = 0.f, n3 = 0.f;
    if (k + 4 < K) {
      n0 = __ldg(Wt + (size_t)(k + 4) * kH + j);
      n1 = __ldg(Wt + (size_t)(k + 5) * kH + j);
      n2 = __ldg(Wt + (size_t)(k + 6) * kH + j);
      n3 = __ldg(Wt + (size_t)(k + 7) * kH + j);
    }
#pragma unroll
    for (int e = 0; e < EMAX; ++e) {
      const float4 xv = *reinterpret_cast<const float4*>(in_s + e * K + k);
      acc[e] = fmaf(xv.x, w0, acc[e]);
      acc[e] = fmaf(xv.y, w1, acc[e]);
      acc[e] = fmaf(xv.z, w2, acc[e]);
      acc[e] = fmaf(xv.w, w3, acc[e]);
    }
    w0 = n0; w1 = n1; w2 = n2; w3 = n3;
  }
  const float b = bias[j];
#pragma unroll
  for (int e = 0; e < EMAX; ++e) out_s[e * kH + j] = tanh_fast(acc[e] + b);
}

// Register-tiled variant for many environments per CTA: thread = 4 consecutive columns x EMAX/4 environments
// (64 column groups x 4 environment groups), so one broadcast LDS.128 feeds 16 FMAs instead of 4 and the weight rows
// are read as LDG.128.  Same k-ascending fmaf order per output as layer<>: bit-identical results.
template <int EMAX>
__device__ __forceinline__ void layer_tiled(const float* __restrict__ in_s, int K, const float* __restrict__ Wt,
                                            const float* __restrict__ bias, float* __restrict__ out_s, int tid) {
  constexpr int ET = EMAX / 4;
  const int cg = tid & 63, eg = tid >> 6;
  const float* in_e = in_s + (size_t)eg * ET * K;
  const float4* W4 = reinterpret_cast<const float4*>(Wt) + cg;  // row k starts at W4[k * 64]
  float4 acc[ET];
#pragma unroll
  for (int e = 0; e < ET; ++e) acc[e] = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 w0 = __ldg(W4), w1 = __ldg(W4 + 64), w2 = __ldg(W4 + 128), w3 = __ldg(W4 + 192);
  for (int k = 0; k < K; k += 4) {
    float4 n0 = make_float4(0.f, 0.f, 0.f, 0.f), n1 = n0, n2 = n0, n3 = n0;
    if (k + 4 < K) {
      n0 = __ldg(W4 + (size_t)(k + 4) * 64);
      n1 = __ldg(W4 + (size_t)(k + 5) * 64);
      n2 = __ldg(W4 + (size_t)(k + 6) * 64);
      n3 = __ldg(W4 + (size_t)(k + 7) * 64);
    }
#pragma unroll
    for (int e = 0; e < ET; ++e) {
      const float4 xv = *reinterpret_cast<const float4*>(in_e + e * K + k);
      acc[e].x = fmaf(xv.x, w0.x, acc[e].x); acc[e].y = fmaf(xv.x, w0.y, acc[e].y);
      acc[e].z = fmaf(xv.x, w0.z, acc[e].z); acc[e].w = fmaf(xv.x, w0.w, acc[e].w);
      acc[e].x = fmaf(xv.y, w1.x, acc[e].x); acc[e].y = fmaf(xv.y, w1.y, acc[e].y);
      acc[e].z = fmaf(xv.y, w1.z, acc[e].z); acc[e].w = fmaf(xv.y, w1.w, acc[e].w);
      acc[e].x = fmaf(xv.z, w2.x, acc[e].x); acc[e].y = fmaf(xv.z, w2.y, acc[e].y);
      acc[e].z = fmaf(xv.z, w2.z, acc[e].z); acc[e].w = fmaf(xv.z, w2.w, acc[e].w);
      acc[e].x = fmaf(xv.w, w3.x, acc[e].x); acc[e].y = fmaf(xv.w, w3.y, acc[e].y);
      acc[e].z = fmaf(xv.w, w3.z, acc[e].z); acc[e].w = fmaf(xv.w, w3.w, acc[e].w);
    }
    w0 = n0; w1 = n1; w2 = n2; w3 = n3;
  }
  const float4 b = *reinterpret_cast<const float4*>(bias + 4 * cg);
#pragma unroll
  for (int e = 0; e < ET; ++e)
    *reinterpret_cast<float4*>(out_s + (size_t)(eg * ET + e) * kH + 4 * cg) =
        make_float4(tanh_fast(acc[e].x + b.x), tanh_fast(acc[e].y + b.y), tanh_fast(acc[e].z + b.z),
                    tanh_fast(acc[e].w + b.w));
}

// ---- deeper software pipelining -------------------------------------------------------------------------------------
// Same arithmetic, same k-ascending fmaf order (bit-identical results), but the weight rows of the next D k-steps
// are in flight instead of one: with 8 warps / SM the one-k-step prefetch leaves the L2 latency exposed (round 1:
// 45 us / env step at E = 4 although the FMA work is ~2 us; round 2 with D = 4: 23.1 -> 19.1 ms per 512-step rollout at
// 512 envs, bit-identical buffers).  Requires K % (4 * D) == 0.
template <int EMAX, int D>
__device__ __forceinline__ void layer_pf(const float* __restrict__ in_s, int K, const float* __restrict__ Wt,
                                         const float* __restrict__ bias, float* __restrict__ out_s, int j) {
  float acc[EMAX];
#pragma unroll
  for (int e = 0; e < EMAX; ++e) acc[e] = 0.f;
  float w[D][4];
#pragma unroll
  for (int d = 0; d < D; ++d)
#pragma unroll
    for (int i = 0; i < 4; ++i) w[d][i] = __ldg(Wt + (size_t)(4 * d + i) * kH + j);
  for (int k = 0; k < K; k += 4 * D) {
#pragma unroll
    for (int d = 0; d < D; ++d) {
      const int kk = k + 4 * d;
      const float w0 = w[d][0], w1 = w[d][1], w2 = w[d][2], w3 = w[d][3];
      if (kk + 4 * D < K) {
#pragma unroll
        for (int i = 0; i < 4; ++i) w[d][i] = __ldg(Wt + (size_t)(kk + 4 * D + i) * kH + j);
      }
#pragma unroll
      for (int e = 0; e < EMAX; ++e) {
        const float4 xv = *reinterpret_cast<const float4*>(in_s + e * K + kk);
        acc[e] = fmaf(xv.x, w0, acc[e]);
        acc[e] = fmaf(xv.y, w1, acc[e]);
        acc[e] = fmaf(xv.z, w2, acc[e]);
        acc[e] = fmaf(xv.w, w3, acc[e]);
      }
    }
  }
  const float b = bias[j];
#pragma unroll
  for (int e = 0; e < EMAX; ++e) out_s[e * kH + j] = tanh_fast(acc[e] + b);
}

template <int EMAX, int D>
__device__ __forceinline__ void layer_tiled_pf(const float* __restrict__ in_s, int K, const float* __restrict__ Wt,
                                               const float* __restrict__ bias, float* __restrict__ out_s, int tid) {
  constexpr int ET = EMAX / 4;
  const int cg = tid & 63, eg = tid >> 6;
  const float* in_e = in_s + (size_t)eg * ET * K;
  const float4* W4 = reinterpret_cast<const float4*>(Wt) + cg;
  float4 acc[ET];
#pragma unroll
  for (int e = 0; e < ET; ++e) acc[e] = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 w[D][4];
#pragma unroll
  for (int d = 0; d < D; ++d)
#pragma unroll
    for (int i = 0; i < 4; ++i) w[d][i] = __ldg(W4 + (size_t)(4 * d + i) * 64);
  for (int k = 0; k < K; k += 4 * D) {
#pragma unroll
    for (int d = 0; d < D; ++d) {
      const int kk = k + 4 * d;
      const float4 w0 = w[d][0], w1 = w[d][1], w2 = w[d][2], w3 = w[d][3];
      if (kk + 4 * D < K) {
#pragma unroll
        for (int i = 0; i < 4; ++i) w[d][i] = __ldg(W4 + (size_t)(kk + 4 * D + i) * 64);
      }
#pragma unroll
      for (int e = 0; e < ET; ++e) {
        const float4 xv = *reinterpret_cast<const float4*>(in_e + e * K + kk);
        acc[e].x = fmaf(xv.x, w0.x, acc[e].x); acc[e].y = fmaf(xv.x, w0.y, acc[e].y);
        acc[e].z = fmaf(xv.x, w0.z, acc[e].z); acc[e].w = fmaf(xv.x, w0.w, acc[e].w);
        acc[e].x = fmaf(xv.y, w1.x, acc[e].x); acc[e].y = fmaf(xv.y, w1.y, acc[e].y);
        acc[e].z = fmaf(xv.y, w1.z, acc[e].z); acc[e].w = fmaf(xv.y, w1.w, acc[e].w);
        acc[e].x = fmaf(xv.z, w2.x, acc[e].x); acc[e].y = fmaf(xv.z, w2.y, acc[e].y);
        acc[e].z = fmaf(xv.z, w2.z, acc[e].z); acc[e].w = fmaf(xv.z, w2.w, acc[e].w);
        acc[e].x = fmaf(xv.w, w3.x, acc[e].x); acc[e].y = fmaf(xv.w, w3.y, acc[e].y);
        acc[e].z = fmaf(xv.w, w3.z, acc[e].z); acc[e].w = fmaf(xv.w, w3.w, acc[e].w);
      }
    }
  }
  const float4 b = *reinterpret_cast<const float4*>(bias + 4 * cg);
#pragma unroll
  for (int e = 0; e < ET; ++e)
    *reinterpret_cast<float4*>(out_s + (size_t)(eg * ET + e) * kH + 4 * cg) =
        make_float4(tanh_fast(acc[e].x + b.x), tanh_fast(acc[e].y + b.y), tanh_fast(acc[e].z + b.z),
                    tanh_fast(acc[e].w + b.w));
}

// EMAX == 32 (up to 32 environments per CTA) uses the register-tiled layer, smaller slices the column-per-thread one.
// Weight rows of the next 4 k-steps in flight (2 in the register-tiled layer) when K allows it.
template <int EMAX>
__device__ __forceinline__ void layer_any(const float* __restrict__ in_s, int K, const float* __restrict__ Wt,
                                          const float* __restrict__ bias, float* __restrict__ out_s, int j) {
  if (K % 16 == 0) {  // uniform
    if constexpr (EMAX >= 32) layer_tiled_pf<EMAX, 2>(in_s, K, Wt, bias, out_s, j);
    else layer_pf<EMAX, 4>(in_s, K, Wt, bias, out_s, j);
    return;
  }
  if constexpr (EMAX >= 32) layer_tiled<EMAX>(in_s, K, Wt, bias, out_s, j);
  else layer<EMAX>(in_s, K, Wt, bias, out_s, j);
}

// value tower on in_s -> g3 in bufB (uses bufC as the middle buffer); every thread must call it
template <int EMAX>
__device__ __forceinline__ void value_tower(const FusedArgs& p, const float* in_s, float* bufB, float* bufC, int j) {
  const float* P = p.params;
  const float* wt_v = p.wt;  // value tower first
  const size_t n0 = (size_t)p.obs * kH, nn = (size_t)kH * kH;
  layer_any<EMAX>(in_s, p.obs, wt_v, P + p.L.vb0, bufB, j);
  __syncthreads();
  layer_any<EMAX>(bufB, kH, wt_v + n0, P + p.L.vb1, bufC, j);
  __syncthreads();
  layer_any<EMAX>(bufC, kH, wt_v + n0 + nn, P + p.L.vb2, bufB, j);
  __syncthreads();
}

// V = g3[e] . vw3 (vdim == 1): warp-level dot product, all lanes get the result
__device__ __forceinline__ float value_dot(const float* g3_row, const float* s_vw, int lane) {
  const float4 g0 = *reinterpret_cast<const float4*>(g3_row + lane * 4);
  const float4 g1 = *reinterpret_cast<const float4*>(g3_row + 128 + lane * 4);
  const float4 w0 = *reinterpret_cast<const float4*>(s_vw + lane * 4);
  const float4 w1 = *reinterpret_cast<const float4*>(s_vw + 128 + lane * 4);
  float s = g0.x * w0.x + g0.y * w0.y + g0.z * w0.z + g0.w * w0.w + g1.x * w1.x + g1.y * w1.y + g1.z * w1.z +
            g1.w * w1.w;
  return rb::warp_sum(s);
}

template <int EMAX>
__global__ void __launch_bounds__(kThreads, 1) rollout_fused_kernel(FusedArgs p) {
  extern __shared__ __align__(16) float sm[];
  const int obs = p.obs, act = p.act;
  float* x = sm;                        // [EMAX][obs]  current observation
  float* bufA = x + EMAX * obs;         // [EMAX][256]
  float* bufB = bufA + EMAX * kH;       // [EMAX][256]
  float* bufC = bufB + EMAX * kH;       // [EMAX][256]
  float* zs = bufC + EMAX * kH;         // [EMAX][obs]  env pre-activation -> final observation
  float* s_mw = zs + EMAX * obs;        // [act][256]
  float* s_vw = s_mw + kMaxAct * kH;    // [256]
  float* act_s = s_vw + kH;             // [EMAX][kMaxAct]
  float* rew_s = act_s + EMAX * kMaxAct;               // [EMAX]
  int* el_s = reinterpret_cast<int*>(rew_s + EMAX);    // [EMAX]
  int* flag_s = el_s + EMAX;                           // [EMAX] bootstrap flag of this step

  const int j = threadIdx.x, lane = j & 31, warp = j >> 5;
  const int e0 = blockIdx.x * p.E;
  int nE = p.B - e0;
  if (nE > p.E) nE = p.E;
  if (nE <= 0) return;
  const int T = p.T, B = p.B;
  const bool has_v = p.vdim > 0;
  const float* P = p.params;
  const size_t n0 = (size_t)obs * kH, nn = (size_t)kH * kH;
  const float* wt_b = p.wt + (n0 + 2 * nn);  // backbone tower after the value tower
  const uint64_t c_p = p.counter_p ? p.counter_p[0] : 0ull;
  const uint64_t c_e = p.counter_e ? p.counter_e[0] : 0ull;

  for (int i = j; i < act * kH; i += kThreads) s_mw[i] = P[p.L.mw + i];
  if (has_v) s_vw[j] = P[p.L.vw3 + j];
  for (int i = j; i < EMAX * obs; i += kThreads) {
    const int e = i / obs, c = i - e * obs;
    x[i] = e < nE ? p.states[(size_t)(e0 + e) * obs + c] : 0.f;
  }
  if (j < EMAX) {
    el_s[j] = j < nE ? p.elapsed[e0 + j] : 0;
    flag_s[j] = 0;
  }
  __syncthreads();

  for (int t = 0; t < T; ++t) {
    // ---- actor tower: x -> bufA -> bufB -> bufA (h3) ----
    layer_any<EMAX>(x, obs, wt_b, P + p.L.bb0, bufA, j);
    __syncthreads();
    layer_any<EMAX>(bufA, kH, wt_b + n0, P + p.L.bb1, bufB, j);
    __syncthreads();
    layer_any<EMAX>(bufB, kH, wt_b + n0 + nn, P + p.L.bb2, bufA, j);
    __syncthreads();
    // ---- value tower: x -> bufB -> bufC -> bufB (g3) ----
    if (has_v) value_tower<EMAX>(p, x, bufB, bufC, j);

    // ---- heads: one warp per environment (head_fwd_kernel, sample mode) ----
    for (int e = warp; e < nE; e += kThreads / 32) {
      const int64_t row = e0 + e;
      const float* h3 = bufA + e * kH;
      const float4 h0 = *reinterpret_cast<const float4*>(h3 + lane * 4);
      const float4 h1 = *reinterpret_cast<const float4*>(h3 + 128 + lane * 4);
      float my_mean = 0.f;
      for (int a = 0; a < act; ++a) {
        const float4 w0 = *reinterpret_cast<const float4*>(s_mw + a * kH + lane * 4);
        const float4 w1 = *reinterpret_cast<const float4*>(s_mw + a * kH + 128 + lane * 4);
        float s = h0.x * w0.x + h0.y * w0.y + h0.z * w0.z + h0.w * w0.w + h1.x * w1.x + h1.y * w1.y + h1.z * w1.z +
                  h1.w * w1.w;
        s = rb::warp_sum(s);
        if (lane == a) my_mean = s + P[p.L.mb + a];
      }
      if (lane < act) {
        const float ls = P[p.L.logstd + lane];
        const float sd = expf(ls);
        float z;
        if (p.policy_noise) {
          z = p.policy_noise[((size_t)t * B + row) * act + lane];
        } else {
          curandStatePhilox4_32_10_t st;
          curand_init(p.seed_p, (unsigned long long)(row * act + lane), p.offset_p + 4ull * (c_p + (uint64_t)t), &st);
          z = curand_normal(&st);
        }
        const float xa = my_mean + sd * z;
        const float d = xa - my_mean;
        const float var = sd * sd;
        const size_t o = ((size_t)t * B + row) * act + lane;
        p.actions[o] = xa;
        p.logp[o] = -(d * d) / (2.0f * var) - logf(sd) - kHalfLog2Pi;
        act_s[e * kMaxAct + lane] = xa;
      }
      if (has_v) {
        const float v = value_dot(bufB + e * kH, s_vw, lane);
        if (lane == 0) p.values[(size_t)t * B + row] = v;
      }
    }
    __syncthreads();

    // ---- env dynamics: zs[e][c] = x[e] . W_s[:, c]  (W_s is [in][out]) ----
    if (j < obs) {
      float acc[EMAX];
#pragma unroll
      for (int e = 0; e < EMAX; ++e) acc[e] = 0.f;
      for (int k = 0; k < obs; k += 4) {
        const float w0 = __ldg(p.w_s + (size_t)(k + 0) * obs + j), w1 = __ldg(p.w_s + (size_t)(k + 1) * obs + j),
                    w2 = __ldg(p.w_s + (size_t)(k + 2) * obs + j), w3 = __ldg(p.w_s + (size_t)(k + 3) * obs + j);
#pragma unroll
        for (int e = 0; e < EMAX; ++e) {
          const float4 xv = *reinterpret_cast<const float4*>(x + e * obs + k);
          acc[e] = fmaf(xv.x, w0, acc[e]);
          acc[e] = fmaf(xv.y, w1, acc[e]);
          acc[e] = fmaf(xv.z, w2, acc[e]);
          acc[e] = fmaf(xv.w, w3, acc[e]);
        }
      }
#pragma unroll
      for (int e = 0; e < EMAX; ++e) zs[e * obs + j] = acc[e];
    }
    __syncthreads();

    // ---- env finish: one warp per environment (env_finish_kernel) ----
    for (int e = warp; e < nE; e += kThreads / 32) {
      const int64_t row = e0 + e;
      curandStatePhilox4_32_10_t st;
      if (!p.env_noise) curand_init(p.seed_e, (unsigned long long)row * 32ull + lane, (c_e + (uint64_t)t) * 64ull, &st);
      const float* nz = p.env_noise ? p.env_noise + ((size_t)t * B + row) * (2 * obs + 2) : nullptr;
      float sq = 0.f;
      for (int c = lane; c < obs; c += 32) {
        float z = zs[e * obs + c];
        for (int a = 0; a < act; ++a) z = fmaf(act_s[e * kMaxAct + a], __ldg(p.w_a + a * obs + c), z);
        const float eps = nz ? nz[c] : curand_normal(&st);
        const float s = tanhf(z + p.noise_std * eps);
        zs[e * obs + c] = s;  // final observation (before any reset)
        sq += s * s;
      }
      sq = rb::warp_sum(sq);
      float eps_r = 0.f, u = 1.f;
      if (lane == 0) {
        eps_r = nz ? nz[obs] : curand_normal(&st);
        u = nz ? nz[obs + 1] : curand_uniform(&st);
      }
      eps_r = __shfl_sync(0xffffffffu, eps_r, 0);
      u = __shfl_sync(0xffffffffu, u, 0);
      const int el = el_s[e] + 1;
      const bool term = u < p.p_term;
      const bool trunc = p.max_episode_steps > 0 && el >= p.max_episode_steps;
      const bool done = term || trunc;
      const bool reset = done && p.auto_reset;
      __syncwarp();
      if (lane == 0) {
        rew_s[e] = -sq / (float)obs + p.reward_noise_std * eps_r;
        const size_t o = (size_t)(t + 1) * B + row;
        p.term[o] = term;
        p.trunc[o] = trunc;
        p.done[o] = done;
        el_s[e] = reset ? 0 : el;
        flag_s[e] = (p.bootstrap_on_done ? done : trunc) ? 1 : 0;
      }
      for (int c = lane; c < obs; c += 32) {
        float s = zs[e * obs + c];
        if (t == T - 1) p.final_obs[(size_t)row * obs + c] = s;
        if (reset) s = nz ? nz[obs + 2 + c] : curand_normal(&st);
        x[e * obs + c] = s;
        p.states[((size_t)(t + 1) * B + row) * obs + c] = s;
      }
    }
    __syncthreads();

    // ---- truncation bootstrap: rewards += gamma * V(final_obs) where flagged (compute_bootstrap_rewards) ----
    if (p.auto_reset && has_v) {
      int any = 0;
      if (j < nE) any = flag_s[j];
      any = __syncthreads_or(any);
      if (any) {
        value_tower<EMAX>(p, zs, bufB, bufC, j);
        for (int e = warp; e < nE; e += kThreads / 32) {
          if (!flag_s[e]) continue;
          const float v = value_dot(bufB + e * kH, s_vw, lane);
          if (lane == 0) {
            rew_s[e] = __fadd_rn(rew_s[e], __fmul_rn(p.gamma, v));
            p.final_values[e0 + e] = v;
          }
        }
        __syncthreads();
      }
    }
    if (j < nE) p.rewards[(size_t)t * B + e0 + j] = rew_s[j];
    // rew_s / flag_s / act_s are next written after later barriers of step t+1
  }

  // ---- bootstrap value row T (env_worker.py:1237-1306) ----
  if (has_v) {
    value_tower<EMAX>(p, x, bufB, bufC, j);
    for (int e = warp; e < nE; e += kThreads / 32) {
      const float v = value_dot(bufB + e * kH, s_vw, lane);
      if (lane == 0) p.values[(size_t)T * B + e0 + e] = v;
    }
  }
  if (j < nE) p.elapsed[e0 + j] = el_s[j];
}

__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int R,
                                                        int C) {
  // out[c][r] = in[r][c]
  __shared__ float tile[32][33];
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + tx;
    tile[i][tx] = (r < R && c < C) ? in[(size_t)r * C + c] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + tx;
    if (c < C && r < R) out[(size_t)c * R + r] = tile[tx][i];
  }
}

template <int EMAX>
size_t fused_smem(int obs) {
  return sizeof(float) * ((size_t)2 * EMAX * obs + (size_t)3 * EMAX * kH + (size_t)kMaxAct * kH + kH +
                          (size_t)EMAX * kMaxAct + EMAX) +
         sizeof(int) * 2 * EMAX;
}

template <int EMAX>
int launch_fused(const FusedArgs& a, int grid, cudaStream_t st) {
  const size_t smem = fused_smem<EMAX>(a.obs);
  if (smem > 227 * 1024) return RB200_E_UNSUPPORTED;
  cudaError_t ce = cudaFuncSetAttribute(rollout_fused_kernel<EMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem);
  if (ce != cudaSuccess) return (int)ce;
  rollout_fused_kernel<EMAX><<<grid, kThreads, smem, st>>>(a);
  rb::count_launch();
  ce = cudaPeekAtLastError();
  return ce == cudaSuccess ? 0 : (int)ce;
}

}  // namespace

// floats needed by rb200_rollout_fused_prepare's output
extern "C" int64_t rb200_rollout_fused_wt_floats(const rb200_mlp_layout* L) {
  if (!L) return 0;
  return 2 * ((int64_t)L->obs_dim * kH + 2 * (int64_t)kH * kH);
}

// 0 when the fused kernel supports this problem (else the caller keeps the per-kernel CUDA-graph rollout)
extern "C" int rb200_rollout_fused_supported(const rb200_mlp_layout* L, int B) {
  if (!L) return RB200_E_NULL;
  if (L->hidden != kH || L->act_dim <= 0 || L->act_dim > kMaxAct || L->value_dim < 0 || L->value_dim > 1)
    return RB200_E_UNSUPPORTED;
  if (L->obs_dim <= 0 || L->obs_dim > kH || (L->obs_dim & 3)) return RB200_E_UNSUPPORTED;
  if (B <= 0 || B > 32 * rb::sm_count()) return RB200_E_UNSUPPORTED;
  return RB200_OK;
}

// wt: per tower (value tower first, then backbone) W0^T [obs][256] | W1^T [256][256] | W2^T [256][256]
extern "C" int rb200_rollout_fused_prepare(const rb200_mlp_layout* L, const float* params, float* wt,
                                           rb200_stream_t stream) {
  if (!L || !params || !wt) return RB200_E_NULL;
  if (L->hidden != kH) return RB200_E_UNSUPPORTED;
  cudaStream_t st = rb::as_stream(stream);
  const int64_t n0 = (int64_t)L->obs_dim * kH, nn = (int64_t)kH * kH;
  const int64_t src[2][3] = {{L->vw0, L->vw1, L->vw2}, {L->bw0, L->bw1, L->bw2}};
  for (int v = 0; v < 2; ++v) {
    if (v == 0 && L->value_dim == 0) continue;
    float* dst = wt + v * (n0 + 2 * nn);
    for (int l = 0; l < 3; ++l) {
      const int R = kH, C = l == 0 ? L->obs_dim : kH;  // stored [out=256][in=C] -> [in][256]
      dim3 grid((C + 31) / 32, (R + 31) / 32);
      transpose_kernel<<<grid, 256, 0, st>>>(params + src[v][l], dst + (l == 0 ? 0 : n0 + (l - 1) * nn), R, C);
      rb::count_launch();
    }
  }
  cudaError_t ce = cudaPeekAtLastError();
  return ce == cudaSuccess ? 0 : (int)ce;
}

extern "C" int rb200_rollout_fused(const rb200_mlp_layout* L, const float* params, const float* wt, const float* w_s,
                                   const float* w_a, float* states, float* actions, float* logprobs, float* values,
                                   float* rewards, uint8_t* terminations, uint8_t* truncations, uint8_t* dones,
                                   float* final_obs, float* final_values, int32_t* elapsed,
                                   const float* policy_noise, const float* env_noise, const uint64_t* counter_policy,
                                   const uint64_t* counter_env, uint64_t seed_policy, uint64_t seed_env,
                                   uint64_t offset_policy, int T, int B, int max_episode_steps, int auto_reset,
                                   int bootstrap_on_done, double gamma, double p_term, double noise_std,
                                   double reward_noise_std, rb200_stream_t stream) {
  int e = rb200_rollout_fused_supported(L, B);
  if (e) return e;
  if (!params || !wt || !w_s || !w_a || !states || !actions || !logprobs || !rewards || !terminations ||
      !truncations || !dones || !final_obs || !elapsed)
    return RB200_E_NULL;
  if (L->value_dim > 0 && (!values || !final_values)) return RB200_E_NULL;
  if (T <= 0) return RB200_E_SHAPE;
  FusedArgs a{};
  a.L = *L; a.params = params; a.wt = wt; a.w_s = w_s; a.w_a = w_a; a.states = states; a.actions = actions;
  a.logp = logprobs; a.values = values; a.rewards = rewards; a.term = terminations; a.trunc = truncations;
  a.done = dones; a.final_obs = final_obs; a.final_values = final_values; a.elapsed = elapsed;
  a.policy_noise = policy_noise; a.env_noise = env_noise; a.counter_p = counter_policy; a.counter_e = counter_env;
  a.seed_p = seed_policy; a.seed_e = seed_env; a.offset_p = offset_policy; a.T = T; a.B = B; a.obs = L->obs_dim;
  a.act = L->act_dim; a.vdim = L->value_dim; a.max_episode_steps = max_episode_steps; a.auto_reset = auto_reset;
  a.bootstrap_on_done = bootstrap_on_done; a.gamma = (float)gamma; a.p_term = (float)p_term;
  a.noise_std = (float)noise_std; a.reward_noise_std = (float)reward_noise_std;
  const int sms = rb::sm_count();
  int E = (B + sms - 1) / sms;
  if (E < 1) E = 1;
  a.E = E;
  const int grid = (B + E - 1) / E;
  cudaStream_t st = rb::as_stream(stream);
  if (E <= 4) return launch_fused<4>(a, grid, st);
  if (E <= 8) return launch_fused<8>(a, grid, st);
  if (E <= 16) return launch_fused<16>(a, grid, st);
  return launch_fused<32>(a, grid, st);
}
