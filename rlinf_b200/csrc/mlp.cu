// K3 / K5: MLP policy + value head: forward, backward, rollout sampling.
// Reference: MLPPolicy.default_forward / _generate_actions, rlinf/models/embodiment/mlp_policy/mlp_policy.py:202-293
// (3x256 tanh backbone -> actor_mean; state-independent actor_logstd; Normal log_prob / entropy) and
// ValueHead, rlinf/models/embodiment/modules/value_head.py:18-67 (3x256 tanh MLP -> value_dim, last layer
// without bias); backward = what autograd derives from them.
//
// Hidden-layer GEMMs run on the fp16-split tensor-core kernels (tc_gemm_h.cu: tcgen05 kind::f16, a = a_hi + a_lo in fp16,
// three MMAs per product, fp32-level accuracy, both towers per launch), reading the weights from the packs that
// rb200_mlp_prepare_weights writes into the caller's wsplit buffer.  Layer 0 falls back to the fp32 SIMT GEMM (sgemm.cuh)
// when its operand cannot be TMA-tiled (obs_dim % 32 != 0, or rows gathered through idx; for its weight gradient also
// obs_dim > 256).  Activations and activation-gradients are stored once, as plain fp32 [n,256] (6 tanh outputs per
// forward, tanh' = 1 - h^2); the tensor-core kernels split them into (hi, lo) pairs on the fly in shared memory.
// The heads (256 -> act mean, 256 -> value) are fused with the Normal log-prob / entropy epilogue and their backward.
#include <curand_kernel.h>

#include <algorithm>

#include "common.cuh"
#include "sgemm.cuh"
#include "tc_gemm.cuh"

namespace {

using namespace rb::gemm;

// ------------------------------------------------------------------------------------------------
// Fused heads.  One warp per sample row; H = 256 hidden units -> 8 per lane (two float4).
// ------------------------------------------------------------------------------------------------
constexpr int kH = 256;
constexpr int kMaxAct = 32;
constexpr int kMaxVal = 8;
constexpr float kHalfLog2Pi = 0.91893853320467274178f;  // log(sqrt(2*pi))

struct HeadFwdArgs {
  const float* h3;      // [n,256] backbone features
  const float* g3;      // [n,256] value features (may be null -> no values)
  const float* mw;      // [act,256]
  const float* mb;      // [act]
  const float* logstd;  // [act]
  const float* vw3;     // [vdim,256]
  const float* action;  // [rows,act] given actions (gathered by idx) or null in sample mode
  const int64_t* idx;
  const float* noise;   // sample mode: [n,act] N(0,1) draws or null -> Philox
  uint64_t seed, offset;
  const uint64_t* counter;
  int sample_mode;
  float* mean_out;     // [n,act] or null
  float* action_out;   // sample mode
  float* logprobs;     // [n,act]
  float* entropy;      // [n,act] or null
  float* values;       // [n,vdim] or null
  int64_t n;
  int act, vdim;
};

__global__ void __launch_bounds__(256) head_fwd_kernel(HeadFwdArgs p) {
  extern __shared__ float sm[];  // mw [act][256] | vw3 [vdim][256]
  float* s_mw = sm;
  float* s_vw = sm + p.act * kH;
  for (int i = threadIdx.x; i < p.act * kH; i += blockDim.x) s_mw[i] = p.mw[i];
  if (p.g3 && p.values)
    for (int i = threadIdx.x; i < p.vdim * kH; i += blockDim.x) s_vw[i] = p.vw3[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const bool want_v = p.g3 && p.values;
  const int64_t row_stride = (int64_t)gridDim.x * nwarp;
  // one warp per row; the NEXT row's 2 KB are requested before this row's dot products and shuffles (round 2: without
  // the prefetch a warp alternated between a DRAM round trip and ~150 dependent instructions: 193 us for 537 MB)
  float4 nh0 = make_float4(0.f, 0.f, 0.f, 0.f), nh1 = nh0, ng0 = nh0, ng1 = nh0;
  auto fetch = [&](int64_t r) {
    if (r < p.n) {
      nh0 = __ldg(reinterpret_cast<const float4*>(p.h3 + r * kH + lane * 4));
      nh1 = __ldg(reinterpret_cast<const float4*>(p.h3 + r * kH + 128 + lane * 4));
      if (want_v) {
        ng0 = __ldg(reinterpret_cast<const float4*>(p.g3 + r * kH + lane * 4));
        ng1 = __ldg(reinterpret_cast<const float4*>(p.g3 + r * kH + 128 + lane * 4));
      }
    }
  };
  fetch((int64_t)blockIdx.x * nwarp + warp);
  for (int64_t row = (int64_t)blockIdx.x * nwarp + warp; row < p.n; row += row_stride) {
    const float4 h0 = nh0, h1 = nh1, pg0 = ng0, pg1 = ng1;
    fetch(row + row_stride);
    float my_mean = 0.f;
    for (int a = 0; a < p.act; ++a) {
      const float4 w0 = *reinterpret_cast<const float4*>(s_mw + a * kH + lane * 4);
      const float4 w1 = *reinterpret_cast<const float4*>(s_mw + a * kH + 128 + lane * 4);
      float s = h0.x * w0.x + h0.y * w0.y + h0.z * w0.z + h0.w * w0.w + h1.x * w1.x + h1.y * w1.y + h1.z * w1.z +
                h1.w * w1.w;
      s = rb::warp_sum(s);
      if (lane == a) my_mean = s + p.mb[a];
    }
    if (lane < p.act) {
      const float ls = p.logstd[lane];
      const float sd = expf(ls);
      float x;
      if (p.sample_mode) {
        float z;
        if (p.noise) {
          z = p.noise[row * p.act + lane];
        } else {
          curandStatePhilox4_32_10_t st;
          // the Philox offset counts 32-bit outputs and curand_normal consumes two (Box-Muller): stride 4 per env step so
          // that consecutive steps never share a word (round 1 used stride 1: the angle word of step t was the radius
          // word of step t+1)
          curand_init(p.seed, (unsigned long long)(row * p.act + lane), p.offset + 4ull * (p.counter ? p.counter[0] : 0ull), &st);
          z = curand_normal(&st);
        }
        x = my_mean + sd * z;
        p.action_out[row * p.act + lane] = x;
      } else {
        const int64_t src = p.idx ? p.idx[row] : row;
        x = p.action[src * p.act + lane];
      }
      // torch.distributions.Normal.log_prob: -((x-mu)^2)/(2 var) - log(sd) - log(sqrt(2 pi))
      const float d = x - my_mean;
      const float var = sd * sd;
      p.logprobs[row * p.act + lane] = -(d * d) / (2.0f * var) - logf(sd) - kHalfLog2Pi;
      if (p.entropy) p.entropy[row * p.act + lane] = 0.5f + kHalfLog2Pi + logf(sd);
      if (p.mean_out) p.mean_out[row * p.act + lane] = my_mean;
    }
    if (want_v) {
      const float4 g0 = pg0, g1 = pg1;
      for (int c = 0; c < p.vdim; ++c) {
        const float4 w0 = *reinterpret_cast<const float4*>(s_vw + c * kH + lane * 4);
        const float4 w1 = *reinterpret_cast<const float4*>(s_vw + c * kH + 128 + lane * 4);
        float s = g0.x * w0.x + g0.y * w0.y + g0.z * w0.z + g0.w * w0.w + g1.x * w1.x + g1.y * w1.y + g1.z * w1.z +
                  g1.w * w1.w;
        s = rb::warp_sum(s);
        if (lane == 0) p.values[row * p.vdim + c] = s;
      }
    }
  }
}

struct HeadBwdArgs {
  const float* h3;   // layer-3 activations of the backbone / value tower
  const float* g3;
  const float* mean;    // [n,act] saved by forward
  const float* mw;
  const float* logstd;
  const float* vw3;
  const float* action;
  const int64_t* idx;
  const float* d_logprobs;  // [n,act]
  const float* d_entropy;   // [n,act] or null
  const float* d_values;    // [n,vdim] or null
  float* dz3;               // [n,256] out: grad wrt backbone layer-3 pre-activation
  float* dy3;               // [n,256] out: grad wrt value layer-3 pre-activation (if d_values)
  float* g_mw;              // [act,256] +=
  float* g_mb;              // [act] +=
  float* g_logstd;          // [act] +=
  float* g_vw3;             // [vdim,256] +=
  float* g_b2;              // [256] += column sums of dz3 (bias gradient of backbone layer 3)
  float* g_vb2;             // [256] += column sums of dy3 (value layer 3)
  float* amax_dz3;          // [1] atomicMax |dz3| (operand scaling of the fp16-split gradient GEMMs), or null
  float* amax_dy3;          // [1] atomicMax |dy3|, or null
  float* part;              // [grid][row] per-block gradient sums (row: see the end of the kernel), added in order by rb::sum_partials
  int64_t n;
  int act, vdim;
};

// REG = true: act <= 8 and vdim <= 2 -> weight-gradient partials live in registers for the whole row loop
// (one shared-memory flush per warp); REG = false: generic path through shared-memory atomics.
template <bool REG>
__global__ void __launch_bounds__(256) head_bwd_kernel(HeadBwdArgs p) {
  extern __shared__ float sm[];
  // layout: mw [act][256] | vw [vdim][256] | acc_mw [act][256] | acc_vw [vdim][256] | acc_mb[32] | acc_ls[32] |
  //         acc_b2[256] | acc_vb2[256]
  float* s_mw = sm;
  float* s_vw = s_mw + p.act * kH;
  float* a_mw = s_vw + p.vdim * kH;
  float* a_vw = a_mw + p.act * kH;
  float* a_mb = a_vw + p.vdim * kH;
  float* a_ls = a_mb + 32;
  float* a_b2 = a_ls + 32;
  float* a_vb2 = a_b2 + kH;
  const bool has_v = p.d_values != nullptr;
  for (int i = threadIdx.x; i < p.act * kH; i += blockDim.x) {
    s_mw[i] = p.mw[i];
    a_mw[i] = 0.f;
  }
  for (int i = threadIdx.x; i < p.vdim * kH; i += blockDim.x) {
    s_vw[i] = has_v ? p.vw3[i] : 0.f;
    a_vw[i] = 0.f;
  }
  if (threadIdx.x < 64) a_mb[threadIdx.x] = 0.f;  // a_mb and a_ls are contiguous
  for (int i = threadIdx.x; i < 2 * kH; i += blockDim.x) a_b2[i] = 0.f;  // a_b2 and a_vb2 are contiguous
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  float cb[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, cv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float mz = 0.f, my = 0.f;  // running max |dz3|, |dy3|
  float rmb = 0.f, rls = 0.f;  // this lane's sums of the mean / log-std gradients (lane < act)
  float rm[REG ? 8 : 1][8], rv[REG ? 2 : 1][8];
#pragma unroll
  for (int a = 0; a < (REG ? 8 : 1); ++a)
#pragma unroll
    for (int j = 0; j < 8; ++j) rm[a][j] = 0.f;
#pragma unroll
  for (int c = 0; c < (REG ? 2 : 1); ++c)
#pragma unroll
    for (int j = 0; j < 8; ++j) rv[c][j] = 0.f;
  // One warp per row, 152 registers in the REG variant -> 8 warps / SM: without help every row pays a full DRAM
  // round trip (ncu round 1: 565 us for 1.05 GB).  The row inputs are therefore fetched two rows ahead.
  struct RowIn {
    float4 h0, h1, g0, g1;
    float x, mu, dlp, den, dv0, dv1;
  };
  auto load_row = [&](int64_t row) -> RowIn {
    RowIn r;
    r.h0 = r.h1 = r.g0 = r.g1 = make_float4(0.f, 0.f, 0.f, 0.f);
    r.x = r.mu = r.dlp = r.den = r.dv0 = r.dv1 = 0.f;
    if (row < p.n) {
      r.h0 = __ldg(reinterpret_cast<const float4*>(p.h3 + row * kH + lane * 4));
      r.h1 = __ldg(reinterpret_cast<const float4*>(p.h3 + row * kH + 128 + lane * 4));
      if (has_v) {
        r.g0 = __ldg(reinterpret_cast<const float4*>(p.g3 + row * kH + lane * 4));
        r.g1 = __ldg(reinterpret_cast<const float4*>(p.g3 + row * kH + 128 + lane * 4));
        if (REG) {
          r.dv0 = __ldg(p.d_values + row * p.vdim);
          if (p.vdim > 1) r.dv1 = __ldg(p.d_values + row * p.vdim + 1);
        }
      }
      if (lane < p.act) {
        const int64_t src = p.idx ? p.idx[row] : row;
        r.x = __ldg(p.action + src * p.act + lane);
        r.mu = __ldg(p.mean + row * p.act + lane);
        r.dlp = __ldg(p.d_logprobs + row * p.act + lane);
        if (p.d_entropy) r.den = __ldg(p.d_entropy + row * p.act + lane);
      }
    }
    return r;
  };
  const int64_t row_stride = (int64_t)gridDim.x * nwarp;
  const int64_t row_first = (int64_t)blockIdx.x * nwarp + warp;
  const float sd_l = lane < p.act ? expf(p.logstd[lane]) : 1.f;
  const float var_l = sd_l * sd_l;
  RowIn nxt0 = load_row(row_first), nxt1 = load_row(row_first + row_stride);
  // Every warp of the block runs the same number of iterations (the generic path adds into shared memory in warp order at
  // each one, between barriers); a row past the end loads zeros, contributes zeros and stores nothing.
  for (int64_t base = (int64_t)blockIdx.x * nwarp; base < p.n; base += row_stride) {
    const int64_t row = base + warp;
    const bool live = row < p.n;
    const RowIn cur = nxt0;
    nxt0 = nxt1;
    nxt1 = load_row(row + 2 * row_stride);
    const float4 h0 = cur.h0, h1 = cur.h1;
    float dmu = 0.f;
    if (lane < p.act) {
      const float d = cur.x - cur.mu;
      dmu = cur.dlp * d / var_l;
      const float dls = cur.dlp * (d * d / var_l - 1.0f) + cur.den;
      rmb += dmu;
      rls += dls;
    }
    float4 dh0 = make_float4(0.f, 0.f, 0.f, 0.f), dh1 = dh0;
#pragma unroll
    for (int a = 0; a < (REG ? 8 : kMaxAct); ++a) {
      if (a >= p.act) break;
      const float g = __shfl_sync(0xffffffffu, dmu, a);
      const float4 w0 = *reinterpret_cast<const float4*>(s_mw + a * kH + lane * 4);
      const float4 w1 = *reinterpret_cast<const float4*>(s_mw + a * kH + 128 + lane * 4);
      dh0.x += g * w0.x; dh0.y += g * w0.y; dh0.z += g * w0.z; dh0.w += g * w0.w;
      dh1.x += g * w1.x; dh1.y += g * w1.y; dh1.z += g * w1.z; dh1.w += g * w1.w;
      if (REG) {
        const int ar = a < 8 ? a : 0;
        rm[ar][0] += g * h0.x; rm[ar][1] += g * h0.y; rm[ar][2] += g * h0.z; rm[ar][3] += g * h0.w;
        rm[ar][4] += g * h1.x; rm[ar][5] += g * h1.y; rm[ar][6] += g * h1.z; rm[ar][7] += g * h1.w;
      }
    }
    float4 o0, o1;
    o0.x = dh0.x * (1.f - h0.x * h0.x); o0.y = dh0.y * (1.f - h0.y * h0.y);
    o0.z = dh0.z * (1.f - h0.z * h0.z); o0.w = dh0.w * (1.f - h0.w * h0.w);
    o1.x = dh1.x * (1.f - h1.x * h1.x); o1.y = dh1.y * (1.f - h1.y * h1.y);
    o1.z = dh1.z * (1.f - h1.z * h1.z); o1.w = dh1.w * (1.f - h1.w * h1.w);
    if (live) {
      *reinterpret_cast<float4*>(p.dz3 + row * kH + lane * 4) = o0;
      *reinterpret_cast<float4*>(p.dz3 + row * kH + 128 + lane * 4) = o1;
    }
    cb[0] += o0.x; cb[1] += o0.y; cb[2] += o0.z; cb[3] += o0.w;
    cb[4] += o1.x; cb[5] += o1.y; cb[6] += o1.z; cb[7] += o1.w;
    mz = fmaxf(mz, fmaxf(fmaxf(fmaxf(fabsf(o0.x), fabsf(o0.y)), fmaxf(fabsf(o0.z), fabsf(o0.w))),
                         fmaxf(fmaxf(fabsf(o1.x), fabsf(o1.y)), fmaxf(fabsf(o1.z), fabsf(o1.w)))));

    if (has_v) {
      const float4 g0 = cur.g0, g1 = cur.g1;
      float4 dg0 = make_float4(0.f, 0.f, 0.f, 0.f), dg1 = dg0;
#pragma unroll
      for (int c = 0; c < (REG ? 2 : kMaxVal); ++c) {
        if (c >= p.vdim) break;
        const float g = REG ? (c == 0 ? cur.dv0 : cur.dv1) : (live ? p.d_values[row * p.vdim + c] : 0.f);
        const float4 w0 = *reinterpret_cast<const float4*>(s_vw + c * kH + lane * 4);
        const float4 w1 = *reinterpret_cast<const float4*>(s_vw + c * kH + 128 + lane * 4);
        dg0.x += g * w0.x; dg0.y += g * w0.y; dg0.z += g * w0.z; dg0.w += g * w0.w;
        dg1.x += g * w1.x; dg1.y += g * w1.y; dg1.z += g * w1.z; dg1.w += g * w1.w;
        if (REG) {
          const int cr = c < 2 ? c : 0;
          rv[cr][0] += g * g0.x; rv[cr][1] += g * g0.y; rv[cr][2] += g * g0.z; rv[cr][3] += g * g0.w;
          rv[cr][4] += g * g1.x; rv[cr][5] += g * g1.y; rv[cr][6] += g * g1.z; rv[cr][7] += g * g1.w;
        }
      }
      float4 q0, q1;
      q0.x = dg0.x * (1.f - g0.x * g0.x); q0.y = dg0.y * (1.f - g0.y * g0.y);
      q0.z = dg0.z * (1.f - g0.z * g0.z); q0.w = dg0.w * (1.f - g0.w * g0.w);
      q1.x = dg1.x * (1.f - g1.x * g1.x); q1.y = dg1.y * (1.f - g1.y * g1.y);
      q1.z = dg1.z * (1.f - g1.z * g1.z); q1.w = dg1.w * (1.f - g1.w * g1.w);
      if (live) {
        *reinterpret_cast<float4*>(p.dy3 + row * kH + lane * 4) = q0;
        *reinterpret_cast<float4*>(p.dy3 + row * kH + 128 + lane * 4) = q1;
      }
      cv[0] += q0.x; cv[1] += q0.y; cv[2] += q0.z; cv[3] += q0.w;
      cv[4] += q1.x; cv[5] += q1.y; cv[6] += q1.z; cv[7] += q1.w;
      my = fmaxf(my, fmaxf(fmaxf(fmaxf(fabsf(q0.x), fabsf(q0.y)), fmaxf(fabsf(q0.z), fabsf(q0.w))),
                           fmaxf(fmaxf(fabsf(q1.x), fabsf(q1.y)), fmaxf(fabsf(q1.z), fabsf(q1.w)))));
    }
    if (!REG) {  // generic path: the warps add this row's weight-gradient terms into shared memory one after another
      for (int w = 0; w < nwarp; ++w) {
        if (warp == w) {
          for (int a = 0; a < p.act; ++a) {
            const float g = __shfl_sync(0xffffffffu, dmu, a);
            float* am = a_mw + a * kH;
            am[lane * 4 + 0] += g * h0.x; am[lane * 4 + 1] += g * h0.y;
            am[lane * 4 + 2] += g * h0.z; am[lane * 4 + 3] += g * h0.w;
            am[128 + lane * 4 + 0] += g * h1.x; am[128 + lane * 4 + 1] += g * h1.y;
            am[128 + lane * 4 + 2] += g * h1.z; am[128 + lane * 4 + 3] += g * h1.w;
          }
          if (has_v)
            for (int c = 0; c < p.vdim; ++c) {
              const float g = live ? p.d_values[row * p.vdim + c] : 0.f;
              const float4 g0 = cur.g0, g1 = cur.g1;
              float* av = a_vw + c * kH;
              av[lane * 4 + 0] += g * g0.x; av[lane * 4 + 1] += g * g0.y;
              av[lane * 4 + 2] += g * g0.z; av[lane * 4 + 3] += g * g0.w;
              av[128 + lane * 4 + 0] += g * g1.x; av[128 + lane * 4 + 1] += g * g1.y;
              av[128 + lane * 4 + 2] += g * g1.z; av[128 + lane * 4 + 3] += g * g1.w;
            }
        }
        __syncthreads();
      }
    }
  }
  if (p.amax_dz3 != nullptr) {  // non-negative floats order like their bit patterns
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mz = fmaxf(mz, __shfl_xor_sync(0xffffffffu, mz, o));
      my = fmaxf(my, __shfl_xor_sync(0xffffffffu, my, o));
    }
    if (lane == 0) {
      if (mz > 0.f) atomicMax(reinterpret_cast<unsigned int*>(p.amax_dz3), __float_as_uint(mz));
      if (has_v && my > 0.f && p.amax_dy3) atomicMax(reinterpret_cast<unsigned int*>(p.amax_dy3), __float_as_uint(my));
    }
  }
  // The warps add their register sums into the block's shared sums one after another (warp 0 first): within a warp
  // every lane owns distinct entries, so the order of every addition is fixed.
  for (int w = 0; w < nwarp; ++w) {
    if (warp == w) {
      if (lane < p.act) {
        a_mb[lane] += rmb;
        a_ls[lane] += rls;
      }
      // bias gradients of the two layer-3 pre-activations (lane owns columns lane*4..+3 and 128+lane*4..+3)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        a_b2[lane * 4 + j] += cb[j];
        a_b2[128 + lane * 4 + j] += cb[4 + j];
        if (has_v) {
          a_vb2[lane * 4 + j] += cv[j];
          a_vb2[128 + lane * 4 + j] += cv[4 + j];
        }
      }
      if (REG) {
#pragma unroll
        for (int a = 0; a < 8; ++a) {
          if (a >= p.act) break;
          float* am = a_mw + a * kH;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            am[lane * 4 + j] += rm[a][j];
            am[128 + lane * 4 + j] += rm[a][4 + j];
          }
        }
        if (has_v) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            if (c >= p.vdim) break;
            float* av = a_vw + c * kH;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              av[lane * 4 + j] += rv[c][j];
              av[128 + lane * 4 + j] += rv[c][4 + j];
            }
          }
        }
      }
    }
    __syncthreads();
  }
  // the block's sums: one row of the partials buffer, laid out like the shared accumulators from a_mw on
  const int row_floats = (p.act + p.vdim) * kH + 64 + 2 * kH;
  for (int i = threadIdx.x; i < row_floats; i += blockDim.x) p.part[(int64_t)blockIdx.x * row_floats + i] = a_mw[i];
}

int head_grid(int64_t n) {
  int64_t blocks = (n + 7) / 8;
  const int64_t cap = (int64_t)rb::sm_count() * 4;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

// ---------------------------------------------------------------------------------------------------------
// Towers.  Activation / gradient tensors are plain fp32 [n,256].
// ---------------------------------------------------------------------------------------------------------
struct TowerW {           // fp32 weights and biases as stored in the parameters
  const float *w0, *b0, *w1, *b1, *w2, *b2;
};

// one hidden layer forward on the SIMT GEMM: out = tanh(in . W^T + b)
int layer_forward(const float* in, const int64_t* idx, int64_t n, int in_dim, const float* w, const float* b,
                  float* out, cudaStream_t st) {
  GemmArgs g{};
  g.M = n; g.N = kH; g.ldc = kH; g.k_per_split = 1 << 30;
  g.A = in; g.lda = in_dim; g.a_rows = idx; g.B = w; g.ldb = in_dim; g.K = in_dim; g.bias = b; g.C = out;
  return launch_gemm<A_KCONTIG, B_KCONTIG, EPI_BIAS_TANH>(g, 1, st);
}

struct TowerWH {  // packed fp16 (hi, lo) tiles of w * 2^10 (rb::tch::split_weights); typed float* (they live in the wsplit buffer)
  const float *w0f, *w1f, *w2f;  // forward packs of layers 0..2
  const float *w1d, *w2d;        // dgrad packs of the square layers
};

struct TowerIO {  // one tower of a grouped forward / backward
  TowerW w;
  TowerWH wh;
  float *H1, *H2, *H3;                               // activations (forward: outputs)
  float *g_w0, *g_b0, *g_w1, *g_b1, *g_w2, *g_b2;    // parameter gradients (backward)
  const float* dZ3;                                  // backward: gradient wrt the layer-3 pre-activation
  float *tA, *tB;                                    // backward: dZ2, dZ1 scratch
  float* amax;                                       // backward: [3] max|dZ3|, max|dZ2|, max|dZ1| (device)
};

// X -> H1 -> H2 -> H3 for `nt` towers sharing the input X
int towers_forward_h(const float* X, const int64_t* idx, int64_t n, int in_dim, TowerIO* t, int nt, cudaStream_t st) {
  int e;
  const bool l0_tc = idx == nullptr && (in_dim % rb::tc::BK == 0);
  rb::tch::GemmLaunch g[2];
  if (l0_tc) {
    for (int i = 0; i < nt; ++i) g[i] = rb::tch::GemmLaunch{X, t[i].wh.w0f, nullptr, t[i].H1, t[i].w.b0, nullptr, nullptr, nullptr, nullptr};
    if ((e = rb::tch::launch(g, nt, n, in_dim, rb::tc::EPI_BIAS_TANH, 0, nullptr, st))) return e;
  } else {
    for (int i = 0; i < nt; ++i)
      if ((e = layer_forward(X, idx, n, in_dim, t[i].w.w0, t[i].w.b0, t[i].H1, st))) return e;
  }
  for (int i = 0; i < nt; ++i) g[i] = rb::tch::GemmLaunch{t[i].H1, t[i].wh.w1f, nullptr, t[i].H2, t[i].w.b1, nullptr, nullptr, nullptr, nullptr};
  if ((e = rb::tch::launch(g, nt, n, kH, rb::tc::EPI_BIAS_TANH, 0, nullptr, st))) return e;
  for (int i = 0; i < nt; ++i) g[i] = rb::tch::GemmLaunch{t[i].H2, t[i].wh.w2f, nullptr, t[i].H3, t[i].w.b2, nullptr, nullptr, nullptr, nullptr};
  return rb::tch::launch(g, nt, n, kH, rb::tc::EPI_BIAS_TANH, 0, nullptr, st);
}

// backward through the hidden layers of `nt` towers given their dZ3 (and max|dZ3| in amax[0]); part: partial-sum rows
// of the gradient GEMMs (part_floats)
int towers_backward_h(const float* X, const int64_t* idx, int64_t n, int in_dim, TowerIO* t, int nt, float* part,
                      cudaStream_t st) {
  int e;
  rb::tch::WgradLaunch w[2];
  rb::tch::GemmLaunch g[2];
  // layer 2: dW2 += dZ3^T . H2 ; dZ2 = (dZ3 . W2) * (1 - H2^2)  (+ column sums -> g_b1, max|dZ2| -> amax[1])
  for (int i = 0; i < nt; ++i) w[i] = rb::tch::WgradLaunch{t[i].dZ3, t[i].H2, t[i].g_w2, t[i].amax};
  if ((e = rb::tch::wgrad(w, nt, n, kH, part, st))) return e;
  for (int i = 0; i < nt; ++i)
    g[i] = rb::tch::GemmLaunch{t[i].dZ3, t[i].wh.w2d, nullptr, t[i].tA, nullptr, t[i].H2, t[i].g_b1, t[i].amax, t[i].amax + 1};
  if ((e = rb::tch::launch(g, nt, n, kH, rb::tc::EPI_TANHGRAD, 1, part, st))) return e;
  // layer 1
  for (int i = 0; i < nt; ++i) w[i] = rb::tch::WgradLaunch{t[i].tA, t[i].H1, t[i].g_w1, t[i].amax + 1};
  if ((e = rb::tch::wgrad(w, nt, n, kH, part, st))) return e;
  for (int i = 0; i < nt; ++i)
    g[i] = rb::tch::GemmLaunch{t[i].tA, t[i].wh.w1d, nullptr, t[i].tB, nullptr, t[i].H1, t[i].g_b0, t[i].amax + 1, t[i].amax + 2};
  if ((e = rb::tch::launch(g, nt, n, kH, rb::tc::EPI_TANHGRAD, 1, part, st))) return e;
  // layer 0: dW0 += dZ1^T . X
  if (idx == nullptr && (in_dim % rb::tc::BK == 0) && in_dim <= 256) {
    for (int i = 0; i < nt; ++i) w[i] = rb::tch::WgradLaunch{t[i].tB, X, t[i].g_w0, t[i].amax + 2};
    return rb::tch::wgrad(w, nt, n, in_dim, part, st);
  }
  const int64_t rows_per_split = 4096;
  const int splits = (int)((n + rows_per_split - 1) / rows_per_split);
  for (int i = 0; i < nt; ++i) {
    GemmArgs a{};
    a.A = t[i].tB; a.lda = kH; a.B = X; a.ldb = in_dim; a.b_rows = idx; a.C = t[i].g_w0;
    a.ldc = in_dim; a.M = kH; a.N = in_dim; a.K = n; a.k_per_split = rows_per_split;
    if ((e = launch_gemm<A_MCONTIG, B_NCONTIG, EPI_ATOMIC>(a, splits, st))) return e;
  }
  return 0;
}

}  // namespace

extern "C" int rb200_mlp_layout_init(rb200_mlp_layout* L, int obs_dim, int act_dim, int value_dim, int hidden) {
  if (!L) return RB200_E_NULL;
  if (obs_dim <= 0 || act_dim <= 0 || value_dim < 0) return RB200_E_SHAPE;
  if (hidden != kH || act_dim > kMaxAct || value_dim > kMaxVal) return RB200_E_UNSUPPORTED;
  L->obs_dim = obs_dim; L->act_dim = act_dim; L->value_dim = value_dim; L->hidden = hidden;
  int64_t o = 0;
  // every tensor starts on a 16-byte boundary (vector loads, TMA); the <=3 pad floats between tensors stay
  // zero forever (zero grad, zero Adam state, decay of zero)
  auto take = [&](int64_t n) { o = (o + 3) & ~int64_t(3); const int64_t at = o; o += n; return at; };
  // named_parameters() order of the reference MLPPolicy: own Parameter first, then children in construction
  // order (value_head, backbone, actor_mean) - mlp_policy.py:28-105
  L->logstd = take(act_dim);
  L->vw0 = take((int64_t)hidden * obs_dim); L->vb0 = take(hidden);
  L->vw1 = take((int64_t)hidden * hidden); L->vb1 = take(hidden);
  L->vw2 = take((int64_t)hidden * hidden); L->vb2 = take(hidden);
  L->vw3 = take((int64_t)value_dim * hidden);
  L->bw0 = take((int64_t)hidden * obs_dim); L->bb0 = take(hidden);
  L->bw1 = take((int64_t)hidden * hidden); L->bb1 = take(hidden);
  L->bw2 = take((int64_t)hidden * hidden); L->bb2 = take(hidden);
  L->mw = take((int64_t)act_dim * hidden); L->mb = take(act_dim);
  L->total = (o + 3) & ~int64_t(3);
  return RB200_OK;
}

// acts layout (floats): H1 H2 H3 G1 G2 G3, each [n,256] | mean [n,act]
// work layout (backward): 6 gradient tensors of [n,256] | 64 floats (max|dZ| slots) | partial-sum rows (part_floats)
static inline int64_t act_floats(int64_t n) { return n * kH; }

static inline int64_t head_row_floats(const rb200_mlp_layout* L) { return (int64_t)(L->act_dim + L->value_dim) * kH + 64 + 2 * kH; }

// partial-sum rows of one backward: the head kernel's per-block sums, then (reusing the same rows, stream-ordered) the
// per-chunk / per-CTA sums of the gradient GEMMs
static int64_t part_floats(const rb200_mlp_layout* L, int64_t n) {
  int64_t f = (int64_t)head_grid(n) * head_row_floats(L);
  for (int ng = 1; ng <= 2; ++ng) {
    f = std::max(f, rb::tch::wgrad_part_floats(ng, n, kH));
    f = std::max(f, rb::tch::wgrad_part_floats(ng, n, L->obs_dim % rb::tc::BK == 0 && L->obs_dim <= kH ? L->obs_dim : kH));
    f = std::max(f, rb::tch::launch_part_floats(ng, n));
  }
  return f;
}

extern "C" int64_t rb200_mlp_fwd_scratch_floats(const rb200_mlp_layout* L, int64_t n) {
  if (!L || n <= 0) return 0;
  return 6 * act_floats(n) + 64 + std::max(n * L->act_dim, part_floats(L, n));
}

// wsplit layout, per tower (value tower first, then backbone): packed fp16 (hi, lo) tiles (rb::tch::split_weights), one
// float of storage per weight: forward packs of w0 [256*obs], w1, w2 [65536 each], then the dgrad packs of w1, w2
static inline int64_t wsplit_tower_floats(int obs) { return (int64_t)kH * obs + 4ll * kH * kH; }

extern "C" int64_t rb200_mlp_wsplit_floats(const rb200_mlp_layout* L) {
  if (!L) return 0;
  return 2 * wsplit_tower_floats(L->obs_dim);
}

static int check_layout(const rb200_mlp_layout* L) {
  if (!L) return RB200_E_NULL;
  if (L->hidden != kH || L->act_dim <= 0 || L->act_dim > kMaxAct || L->value_dim < 0 || L->value_dim > kMaxVal)
    return RB200_E_UNSUPPORTED;
  return RB200_OK;
}

namespace {
TowerW tower_w(const rb200_mlp_layout* L, const float* P, bool value) {
  TowerW w;
  if (value) {
    w.w0 = P + L->vw0; w.b0 = P + L->vb0; w.w1 = P + L->vw1; w.b1 = P + L->vb1; w.w2 = P + L->vw2; w.b2 = P + L->vb2;
  } else {
    w.w0 = P + L->bw0; w.b0 = P + L->bb0; w.w1 = P + L->bw1; w.b1 = P + L->bb1; w.w2 = P + L->bw2; w.b2 = P + L->bb2;
  }
  return w;
}
TowerWH tower_wh(const rb200_mlp_layout* L, const float* ws, bool value) {
  const int64_t n0 = (int64_t)kH * L->obs_dim, nn = (int64_t)kH * kH;
  const float* b = ws + (value ? 0 : wsplit_tower_floats(L->obs_dim));
  TowerWH t;
  t.w0f = b;
  t.w1f = b + n0;
  t.w2f = b + n0 + nn;
  t.w1d = b + n0 + 2 * nn;
  t.w2d = b + n0 + 3 * nn;
  return t;
}
}  // namespace

// Refresh the weight packs the tensor-core GEMMs read: fp16 (hi, lo) of w * 2^10 for all hidden matrices in ONE launch.
// Call after every parameter update (once per optimiser step / once per rollout).
extern "C" int rb200_mlp_prepare_weights(const rb200_mlp_layout* L, const float* params, float* wsplit,
                                         rb200_stream_t stream) {
  int e = check_layout(L);
  if (e) return e;
  if (!params || !wsplit) return RB200_E_NULL;
  rb::tch::SplitSpec sp[6];
  int cnt = 0;
  for (int v = 0; v < 2; ++v) {
    if (v == 0 && L->value_dim == 0) continue;
    const TowerW w = tower_w(L, params, v == 0);
    const TowerWH t = tower_wh(L, wsplit, v == 0);
    const int64_t n0 = (int64_t)kH * L->obs_dim, nn = (int64_t)kH * kH;
    if (L->obs_dim % rb::tc::BK == 0)  // layer 0 runs on the tensor cores only then
      sp[cnt++] = rb::tch::SplitSpec{w.w0, const_cast<float*>(t.w0f), nullptr, n0};
    sp[cnt++] = rb::tch::SplitSpec{w.w1, const_cast<float*>(t.w1f), const_cast<float*>(t.w1d), nn};
    sp[cnt++] = rb::tch::SplitSpec{w.w2, const_cast<float*>(t.w2f), const_cast<float*>(t.w2d), nn};
  }
  return rb::tch::split_weights(sp, cnt, rb::as_stream(stream));
}

extern "C" int rb200_mlp_forward(const rb200_mlp_layout* L, const float* params, const float* wsplit,
                                 const float* states, const float* action, const int64_t* idx, int64_t n,
                                 float* logprobs, float* entropy, float* values, float* acts, float* work,
                                 rb200_stream_t stream) {
  int e = check_layout(L);
  if (e) return e;
  if (!params || !wsplit || !states || !action || !logprobs || !acts || !work) return RB200_E_NULL;
  if (n <= 0) return RB200_E_SHAPE;
  if (values && L->value_dim == 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  const int64_t PF = act_floats(n);
  float *H1 = acts, *H2 = H1 + PF, *H3 = H2 + PF, *G1 = H3 + PF, *G2 = G1 + PF, *G3 = G2 + PF;
  float* mean = G3 + PF;
  const float* P = params;
  TowerIO t[2] = {};
  t[0].w = tower_w(L, P, false); t[0].wh = tower_wh(L, wsplit, false); t[0].H1 = H1; t[0].H2 = H2; t[0].H3 = H3;
  t[1].w = tower_w(L, P, true);  t[1].wh = tower_wh(L, wsplit, true);  t[1].H1 = G1; t[1].H2 = G2; t[1].H3 = G3;
  if ((e = towers_forward_h(states, idx, n, L->obs_dim, t, values ? 2 : 1, st))) return e;
  HeadFwdArgs h{};
  h.h3 = H3; h.g3 = values ? G3 : nullptr; h.mw = P + L->mw; h.mb = P + L->mb;
  h.logstd = P + L->logstd; h.vw3 = P + L->vw3; h.action = action; h.idx = idx; h.sample_mode = 0; h.mean_out = mean;
  h.logprobs = logprobs; h.entropy = entropy; h.values = values; h.n = n; h.act = L->act_dim; h.vdim = L->value_dim;
  const size_t smem = sizeof(float) * (size_t)(L->act_dim + L->value_dim) * kH;
  head_fwd_kernel<<<head_grid(n), 256, smem, st>>>(h);
  rb::count_launch();
  RB_RETURN_LAUNCH();
}

extern "C" int rb200_mlp_backward(const rb200_mlp_layout* L, const float* params, const float* wsplit,
                                  const float* states, const float* action, const int64_t* idx, int64_t n,
                                  const float* d_logprobs, const float* d_entropy, const float* d_values,
                                  const float* acts, float* work, float* grads, rb200_stream_t stream) {
  int e = check_layout(L);
  if (e) return e;
  if (!params || !wsplit || !states || !action || !d_logprobs || !acts || !work || !grads) return RB200_E_NULL;
  if (n <= 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  const int64_t PF = act_floats(n);
  const float *H1 = acts, *H2 = H1 + PF, *H3 = H2 + PF, *G1 = H3 + PF, *G2 = G1 + PF, *G3 = G2 + PF;
  const float* mean = G3 + PF;
  float *dZ3 = work, *tA = dZ3 + PF, *tB = tA + PF, *dY3 = tB + PF, *uA = dY3 + PF, *uB = uA + PF;
  const float* P = params;
  float* G = grads;
  HeadBwdArgs h{};
  h.h3 = H3; h.g3 = G3; h.mean = mean; h.mw = P + L->mw;
  h.logstd = P + L->logstd; h.vw3 = P + L->vw3; h.action = action; h.idx = idx; h.d_logprobs = d_logprobs;
  h.d_entropy = d_entropy; h.d_values = d_values; h.dz3 = dZ3; h.dy3 = dY3;
  h.g_mw = G + L->mw; h.g_mb = G + L->mb; h.g_logstd = G + L->logstd; h.g_vw3 = G + L->vw3;
  h.g_b2 = G + L->bb2; h.g_vb2 = G + L->vb2;
  h.n = n; h.act = L->act_dim; h.vdim = L->value_dim;
  float* amax = work + 6 * PF;  // 8 floats of the scratch tail: max|dZ3|,|dZ2|,|dZ1| of the policy tower, then the value tower
  float* part = work + 6 * PF + 64;
  {
    cudaError_t ce = cudaMemsetAsync(amax, 0, 8 * sizeof(float), st);
    if (ce != cudaSuccess) return (int)ce;
  }
  h.amax_dz3 = amax;
  h.amax_dy3 = amax + 3;
  const size_t smem = sizeof(float) * ((size_t)2 * (L->act_dim + L->value_dim) * kH + 64 + 2 * kH);
  const bool reg = L->act_dim <= 8 && L->value_dim <= 2;
  if (smem > 48 * 1024) {
    cudaError_t ce = cudaFuncSetAttribute(head_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem);
    if (ce != cudaSuccess) return (int)ce;
  }
  const int grid = head_grid(n);
  const int64_t row = head_row_floats(L), va = (int64_t)L->act_dim * kH;
  h.part = part;
  if (reg)
    head_bwd_kernel<true><<<grid, 256, smem, st>>>(h);
  else
    head_bwd_kernel<false><<<grid, 256, smem, st>>>(h);
  rb::count_launch();
  {
    cudaError_t ce = cudaPeekAtLastError();
    if (ce != cudaSuccess) return (int)ce;
    const int64_t o = va + (int64_t)L->value_dim * kH;  // a_mb | a_ls | a_b2 | a_vb2 follow the weight sums
    rb::PartialSeg segs[6] = {{h.g_mw, 0, va}, {h.g_mb, o, L->act_dim}, {h.g_logstd, o + 32, L->act_dim},
                              {h.g_b2, o + 64, kH}, {h.g_vw3, va, (int64_t)L->value_dim * kH}, {h.g_vb2, o + 64 + kH, kH}};
    if ((e = rb::sum_partials(h.part, grid, row, segs, d_values ? 6 : 4, st))) return e;
  }
  TowerIO t[2] = {};
  t[0].w = tower_w(L, P, false); t[0].wh = tower_wh(L, wsplit, false);
  t[0].H1 = const_cast<float*>(H1); t[0].H2 = const_cast<float*>(H2); t[0].dZ3 = dZ3; t[0].tA = tA; t[0].tB = tB;
  t[0].g_w0 = G + L->bw0; t[0].g_b0 = G + L->bb0; t[0].g_w1 = G + L->bw1; t[0].g_b1 = G + L->bb1;
  t[0].g_w2 = G + L->bw2; t[0].g_b2 = G + L->bb2; t[0].amax = amax;
  t[1].w = tower_w(L, P, true); t[1].wh = tower_wh(L, wsplit, true);
  t[1].H1 = const_cast<float*>(G1); t[1].H2 = const_cast<float*>(G2); t[1].dZ3 = dY3; t[1].tA = uA; t[1].tB = uB;
  t[1].g_w0 = G + L->vw0; t[1].g_b0 = G + L->vb0; t[1].g_w1 = G + L->vw1; t[1].g_b1 = G + L->vb1;
  t[1].g_w2 = G + L->vw2; t[1].g_b2 = G + L->vb2; t[1].amax = amax + 3;
  return towers_backward_h(states, idx, n, L->obs_dim, t, d_values ? 2 : 1, part, st);
}

// work: 6 activation tensors; rb200_mlp_fwd_scratch_floats(L, n) floats is always enough
extern "C" int rb200_mlp_sample(const rb200_mlp_layout* L, const float* params, const float* wsplit,
                                const float* states, const float* noise, uint64_t seed, uint64_t offset,
                                const uint64_t* counter_dev, int64_t n, float* action, float* logprobs, float* values,
                                float* work, rb200_stream_t stream) {
  int e = check_layout(L);
  if (e) return e;
  if (!params || !wsplit || !states || !action || !logprobs || !work) return RB200_E_NULL;
  if (n <= 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  const int64_t PF = act_floats(n);
  float *H1 = work, *H2 = H1 + PF, *H3 = H2 + PF, *G1 = H3 + PF, *G2 = G1 + PF, *G3 = G2 + PF;
  const float* P = params;
  TowerIO t[2] = {};  // both towers in one grouped launch per layer
  t[0].w = tower_w(L, P, false); t[0].wh = tower_wh(L, wsplit, false); t[0].H1 = H1; t[0].H2 = H2; t[0].H3 = H3;
  t[1].w = tower_w(L, P, true);  t[1].wh = tower_wh(L, wsplit, true);  t[1].H1 = G1; t[1].H2 = G2; t[1].H3 = G3;
  if ((e = towers_forward_h(states, nullptr, n, L->obs_dim, t, values ? 2 : 1, st))) return e;
  HeadFwdArgs h{};
  h.h3 = H3; h.g3 = values ? G3 : nullptr; h.mw = P + L->mw; h.mb = P + L->mb;
  h.logstd = P + L->logstd; h.vw3 = P + L->vw3; h.noise = noise; h.seed = seed; h.offset = offset;
  h.counter = counter_dev; h.sample_mode = 1; h.action_out = action; h.logprobs = logprobs; h.values = values; h.n = n;
  h.act = L->act_dim; h.vdim = L->value_dim;
  const size_t smem = sizeof(float) * (size_t)(L->act_dim + L->value_dim) * kH;
  head_fwd_kernel<<<head_grid(n), 256, smem, st>>>(h);
  rb::count_launch();
  RB_RETURN_LAUNCH();
}

// value tower + last linear layer only (no bias on the last layer: value_head.py:46)
namespace {
__global__ void __launch_bounds__(256) value_head_kernel(const float* __restrict__ g3, const float* __restrict__ vw3, float* __restrict__ values,
                                                         int64_t n, int vdim) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int64_t row = (int64_t)blockIdx.x * nwarp + warp; row < n; row += (int64_t)gridDim.x * nwarp) {
    const float4 g0 = *reinterpret_cast<const float4*>(g3 + row * kH + lane * 4);
    const float4 g1 = *reinterpret_cast<const float4*>(g3 + row * kH + 128 + lane * 4);
    for (int c = 0; c < vdim; ++c) {
      const float4 w0 = *reinterpret_cast<const float4*>(vw3 + c * kH + lane * 4);
      const float4 w1 = *reinterpret_cast<const float4*>(vw3 + c * kH + 128 + lane * 4);
      float s = g0.x * w0.x + g0.y * w0.y + g0.z * w0.z + g0.w * w0.w + g1.x * w1.x + g1.y * w1.y + g1.z * w1.z +
                g1.w * w1.w;
      s = rb::warp_sum(s);
      if (lane == 0) values[row * vdim + c] = s;
    }
  }
}
}  // namespace

// work: 3 activation tensors
extern "C" int rb200_mlp_value(const rb200_mlp_layout* L, const float* params, const float* wsplit,
                               const float* states, int64_t n, float* values, float* work, rb200_stream_t stream) {
  int e = check_layout(L);
  if (e) return e;
  if (!params || !wsplit || !states || !values || !work) return RB200_E_NULL;
  if (n <= 0 || L->value_dim <= 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  const int64_t PF = act_floats(n);
  float *G1 = work, *G2 = G1 + PF, *G3 = G2 + PF;
  TowerIO t[1] = {};
  t[0].w = tower_w(L, params, true); t[0].wh = tower_wh(L, wsplit, true); t[0].H1 = G1; t[0].H2 = G2; t[0].H3 = G3;
  if ((e = towers_forward_h(states, nullptr, n, L->obs_dim, t, 1, st))) return e;
  value_head_kernel<<<head_grid(n), 256, 0, st>>>(G3, params + L->vw3, values, n, L->value_dim);
  rb::count_launch();
  RB_RETURN_LAUNCH();
}

// actor tower + mean head only (mode="eval": the action is the mean, mlp_policy.py:268-271)
namespace {
// the dot products and the bias add of head_fwd_kernel, written the same way so the mean is bit-identical
__global__ void __launch_bounds__(256) mean_head_kernel(const float* __restrict__ h3, const float* __restrict__ mw,
                                                        const float* __restrict__ mb, float* __restrict__ mean, int64_t n,
                                                        int act) {
  extern __shared__ float s_mw[];  // [act][256]
  for (int i = threadIdx.x; i < act * kH; i += blockDim.x) s_mw[i] = mw[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int64_t row = (int64_t)blockIdx.x * nwarp + warp; row < n; row += (int64_t)gridDim.x * nwarp) {
    const float4 h0 = __ldg(reinterpret_cast<const float4*>(h3 + row * kH + lane * 4));
    const float4 h1 = __ldg(reinterpret_cast<const float4*>(h3 + row * kH + 128 + lane * 4));
    float my_mean = 0.f;
    for (int a = 0; a < act; ++a) {
      const float4 w0 = *reinterpret_cast<const float4*>(s_mw + a * kH + lane * 4);
      const float4 w1 = *reinterpret_cast<const float4*>(s_mw + a * kH + 128 + lane * 4);
      float s = h0.x * w0.x + h0.y * w0.y + h0.z * w0.z + h0.w * w0.w + h1.x * w1.x + h1.y * w1.y + h1.z * w1.z +
                h1.w * w1.w;
      s = rb::warp_sum(s);
      if (lane == a) my_mean = s + mb[a];
    }
    if (lane < act) mean[row * act + lane] = my_mean;
  }
}
}  // namespace

extern "C" int rb200_mlp_mean(const rb200_mlp_layout* L, const float* params, const float* wsplit, const float* states,
                              int64_t n, float* mean, float* work, rb200_stream_t stream) {
  int e = check_layout(L);
  if (e) return e;
  if (!params || !wsplit || !states || !mean || !work) return RB200_E_NULL;
  if (n <= 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  const int64_t PF = act_floats(n);
  float *H1 = work, *H2 = H1 + PF, *H3 = H2 + PF;
  TowerIO t[1] = {};
  t[0].w = tower_w(L, params, false); t[0].wh = tower_wh(L, wsplit, false); t[0].H1 = H1; t[0].H2 = H2; t[0].H3 = H3;
  if ((e = towers_forward_h(states, nullptr, n, L->obs_dim, t, 1, st))) return e;
  mean_head_kernel<<<head_grid(n), 256, sizeof(float) * (size_t)L->act_dim * kH, st>>>(H3, params + L->mw,
                                                                                      params + L->mb, mean, n,
                                                                                      L->act_dim);
  rb::count_launch();
  RB_RETURN_LAUNCH();
}
