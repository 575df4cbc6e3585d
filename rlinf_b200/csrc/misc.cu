// Small path kernels: reward filter (a10), kl_penalty (a18), masked statistics for rollout metrics (a24).
#include "common.cuh"

namespace {

// ---- a10: reward filter -----------------------------------------------------------------------------------------
// Reference: EmbodiedFSDPActor._process_received_rollout_batch, workers/actor/embodied_fsdp_actor_worker.py:236-282
// (duplicate: preprocess_embodied_batch, rlinf/utils/utils.py:803-830): per-env sum of (masked) rewards over all
// steps, mean over the group of G consecutive envs, keep the group iff lower <= mean <= upper.
// One warp per group.
__global__ void __launch_bounds__(256) reward_filter_kernel(const float* __restrict__ rewards,
                                                            const uint8_t* __restrict__ mask, uint8_t* __restrict__ keep,
                                                            int nc, int B, int C, int G, float lower, float upper) {
  const int lane = threadIdx.x & 31;
  const int grp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (grp * G >= B) return;
  // per-env sums in fp32 (as the reference's .sum(dim=-1)), then the group mean
  float gsum = 0.f;
  for (int e = 0; e < G; ++e) {
    const int b = grp * G + e;
    float s = 0.f;
    for (int i = lane; i < nc * C; i += 32) {
      const int ch = i / C, c = i - ch * C;
      const size_t o = ((size_t)ch * B + b) * C + c;
      s += mask ? rewards[o] * (mask[o] ? 1.0f : 0.0f) : rewards[o];
    }
    gsum += rb::warp_sum(s);
  }
  const float mean = gsum / (float)G;
  const uint8_t k = (mean >= lower && mean <= upper) ? 1 : 0;
  for (int e = lane; e < G; e += 32) keep[grp * G + e] = k;
}

// out[ch,b,c] = keep[b] & (mask ? mask[ch,b,c] : 1); Cm = C when mask given, else 1
__global__ void __launch_bounds__(256) apply_keep_kernel(const uint8_t* __restrict__ keep,
                                                         const uint8_t* __restrict__ mask, uint8_t* __restrict__ out,
                                                         int nc, int B, int Cm) {
  const int64_t n = (int64_t)nc * B * Cm;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int b = (int)((i / Cm) % B);
    out[i] = (uint8_t)(keep[b] && (mask ? mask[i] != 0 : true));
  }
}

// ---- a18: kl_penalty, rlinf/algorithms/utils.py:26-64 -------------------------------------------------------------
// mode 0: k1 (lp-ref), 1: abs, 2: k2 (0.5 d^2), 3: k3 (low_var_kl with clamps +-20 / +-10). d_out = d kl / d logprob.
__global__ void __launch_bounds__(256) kl_penalty_kernel(const float* __restrict__ lp, const float* __restrict__ ref,
                                                         float* __restrict__ out, float* __restrict__ dlp, int64_t n,
                                                         int mode) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float a = lp[i], b = ref[i];
    float v, g;
    if (mode == 0) {
      v = __fsub_rn(a, b);
      g = 1.0f;
    } else if (mode == 1) {
      const float d = __fsub_rn(a, b);
      v = fabsf(d);
      g = d > 0.f ? 1.0f : (d < 0.f ? -1.0f : 0.0f);
    } else if (mode == 2) {
      const float d = __fsub_rn(a, b);
      v = __fmul_rn(0.5f, __fmul_rn(d, d));
      g = d;
    } else {
      const float raw = __fsub_rn(b, a);
      const float kl = fminf(fmaxf(raw, -20.0f), 20.0f);
      const float ratio = expf(kl);
      const float kld = __fsub_rn(__fsub_rn(ratio, kl), 1.0f);
      v = fminf(fmaxf(kld, -10.0f), 10.0f);
      const bool pass = (raw >= -20.0f && raw <= 20.0f) && (kld >= -10.0f && kld <= 10.0f);
      g = pass ? -(ratio - 1.0f) : 0.0f;  // d kld / d lp = (ratio - 1) * d kl / d lp, d kl / d lp = -1
    }
    out[i] = v;
    if (dlp) dlp[i] = g;
  }
}

// ---- a24: masked count / sum / min / max (compute_rollout_metrics, rlinf/utils/metric_utils.py:422-506) ------------
__global__ void __launch_bounds__(256) masked_stats_kernel(const float* __restrict__ x, const uint8_t* __restrict__ mask,
                                                           int64_t n, int64_t mask_div, double* __restrict__ out) {
  __shared__ double red[2 * 32];
  __shared__ float rmin[32], rmax[32];
  double v[2] = {0.0, 0.0};
  float mn = INFINITY, mx = -INFINITY;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (mask && !mask[i / mask_div]) continue;
    const float xi = x[i];
    v[0] += 1.0;
    v[1] += (double)xi;
    mn = fminf(mn, xi);
    mx = fmaxf(mx, xi);
  }
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
    rmin[warp] = mn;
    rmax[warp] = mx;
  }
  rb::block_sum<2>(v, red);  // contains a __syncthreads
  if (threadIdx.x == 0) {
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
      mn = fminf(mn, rmin[w]);
      mx = fmaxf(mx, rmax[w]);
    }
    if (v[0] > 0.0) {
      atomicAdd(&out[0], v[0]);
      atomicAdd(&out[1], v[1]);
      // double min/max through CAS on the bit pattern (values are finite floats widened to double)
      unsigned long long* pmin = reinterpret_cast<unsigned long long*>(&out[2]);
      unsigned long long* pmax = reinterpret_cast<unsigned long long*>(&out[3]);
      unsigned long long old = *pmin, assumed;
      do {
        assumed = old;
        if (__longlong_as_double((long long)assumed) <= (double)mn) break;
        old = atomicCAS(pmin, assumed, (unsigned long long)__double_as_longlong((double)mn));
      } while (old != assumed);
      old = *pmax;
      do {
        assumed = old;
        if (__longlong_as_double((long long)assumed) >= (double)mx) break;
        old = atomicCAS(pmax, assumed, (unsigned long long)__double_as_longlong((double)mx));
      } while (old != assumed);
    }
  }
}

__global__ void stats_init_kernel(double* out) {
  if (threadIdx.x == 0) {
    out[0] = 0.0;
    out[1] = 0.0;
    out[2] = INFINITY;
    out[3] = -INFINITY;
  }
}

int grid_for(int64_t n) {
  int64_t b = (n + 255) / 256;
  const int64_t cap = (int64_t)rb::sm_count() * 8;
  if (b > cap) b = cap;
  return (int)(b < 1 ? 1 : b);
}

}  // namespace

extern "C" int rb200_reward_filter(const float* rewards, const uint8_t* loss_mask, uint8_t* out_mask, uint8_t* keep_env,
                                   int nc, int B, int C, int group_size, float lower, float upper,
                                   rb200_stream_t stream) {
  if (!rewards || !out_mask || !keep_env) return RB200_E_NULL;
  if (nc <= 0 || B <= 0 || C <= 0 || group_size <= 0 || B % group_size != 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  const int n_groups = B / group_size;
  reward_filter_kernel<<<(n_groups + 7) / 8, 256, 0, st>>>(rewards, loss_mask, keep_env, nc, B, C, group_size, lower,
                                                            upper);
  rb::count_launch();
  const int Cm = loss_mask ? C : 1;
  apply_keep_kernel<<<grid_for((int64_t)nc * B * Cm), 256, 0, st>>>(keep_env, loss_mask, out_mask, nc, B, Cm);
  rb::count_launch();
  RB_RETURN_LAUNCH();
}

extern "C" int rb200_kl_penalty(const float* logprob, const float* ref_logprob, float* out, float* d_logprob, int64_t n,
                                int mode, rb200_stream_t stream) {
  if (!logprob || !ref_logprob || !out) return RB200_E_NULL;
  if (n <= 0) return RB200_E_SHAPE;
  if (mode < 0 || mode > 3) return RB200_E_ARG;
  kl_penalty_kernel<<<grid_for(n), 256, 0, rb::as_stream(stream)>>>(logprob, ref_logprob, out, d_logprob, n, mode);
  rb::count_launch();
  RB_RETURN_LAUNCH();
}

extern "C" int rb200_masked_stats(const float* x, const uint8_t* mask, int64_t n, int64_t mask_div, double* out4,
                                  rb200_stream_t stream) {
  if (!x || !out4) return RB200_E_NULL;
  if (n < 0 || mask_div <= 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  stats_init_kernel<<<1, 32, 0, st>>>(out4);
  rb::count_launch();
  if (n > 0) {
    masked_stats_kernel<<<grid_for(n), 256, 0, st>>>(x, mask, n, mask_div, out4);
    rb::count_launch();
  }
  RB_RETURN_LAUNCH();
}

namespace rb {
namespace {
constexpr int kMaxSegs = 8;
struct Segs {
  PartialSeg s[kMaxSegs];
};

// block = 32 outputs x 32 row phases; grid = (ceil(max K / 32), nseg).  Row phase r sums rows r, r+32, ... in order,
// then one thread adds the 32 phase sums in order: the same order on every run.
__global__ void __launch_bounds__(1024) sum_partials_kernel(const float* __restrict__ part, int nparts, int64_t stride,
                                                            Segs segs) {
  __shared__ float s[32][33];
  const PartialSeg g = segs.s[blockIdx.y];
  const int kx = threadIdx.x & 31, ph = threadIdx.x >> 5;
  const int64_t k = (int64_t)blockIdx.x * 32 + kx;
  float acc = 0.f;
  if (k < g.K)
    for (int b = ph; b < nparts; b += 32) acc += part[(int64_t)b * stride + g.off + k];
  s[ph][kx] = acc;
  __syncthreads();
  if (ph == 0 && k < g.K) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) t += s[i][kx];
    g.out[k] += t;
  }
}
}  // namespace

int sum_partials(const float* part, int nparts, int64_t stride, const PartialSeg* segs, int nseg, cudaStream_t st) {
  if (nseg < 1 || nseg > kMaxSegs || nparts < 1) return RB200_E_SHAPE;
  Segs S{};
  int64_t kmax = 0;
  for (int i = 0; i < nseg; ++i) {
    S.s[i] = segs[i];
    if (segs[i].K > kmax) kmax = segs[i].K;
  }
  sum_partials_kernel<<<dim3((unsigned)((kmax + 31) / 32), (unsigned)nseg), 1024, 0, st>>>(part, nparts, stride, S);
  count_launch();
  cudaError_t ce = cudaPeekAtLastError();
  return ce == cudaSuccess ? 0 : (int)ce;
}
}  // namespace rb
