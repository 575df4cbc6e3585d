// Policy evaluation: the eval env step with per-episode bookkeeping, and the reduction of the episode records.
// Reference: EnvWorker.evaluate / env_evaluate_step, rlinf/workers/env/env_worker.py:1374-1460, 557-620;
// ManiskillEnv.step / chunk_step / _record_metrics / _reset_metrics / _handle_auto_reset,
// rlinf/envs/maniskill/maniskill_env.py:232-391; compute_evaluate_metrics, rlinf/utils/metric_utils.py:372-420.
//
// The dynamics, the noise layout and the Philox streams are those of rb200_synth_env_step (C = 1) and
// rb200_synth_env_chunk_step (C > 1) in rollout.cu; the synthetic env's termination draw (u < p_term) is its "success"
// info.  Per sub-step and env (ManiSkill order): returns += r (fp32); success_once |= success; episode_len =
// elapsed; with ignore_terminations the termination is dropped after recording and success_at_end = success.  The
// sub-steps of a chunk run past a done; the chunk's done is the OR of its sub-steps' flags, its episode record is the
// bookkeeping of its last sub-step (the infos `final_info` holds), and one auto-reset follows the chunk.
#include <curand_kernel.h>

#include "common.cuh"
#include "sgemm.cuh"

namespace {

using namespace rb::gemm;

// ep_flags bits (per env, carried across sub-steps, chunk steps and epochs)
constexpr uint8_t kSuccessOnce = 1, kPrevDone = 2, kChunkTerm = 4, kChunkTrunc = 8;

struct EvalArgs {
  const float* z;         // [B,obs] = s . W_s
  const float* action;    // [B, C*act]: sub-step c uses columns [c*act, (c+1)*act)
  const float* w_a;       // [act,obs]
  const float* noise;     // optional [B, C*(obs+2) + obs]: per sub-step eps[obs] | eps_r | u_term, then reset[obs]
  float* out_state;       // [B,obs] state after this sub-step (the chunk's last sub-step: after the auto-reset)
  int32_t* elapsed;       // [B]
  float* ep_return;       // [B]
  uint8_t* ep_flags;      // [B]
  uint8_t* rec_flags;     // [B] record row of this chunk step (bit 0 reported, 1 success_once, 2 success_at_end)
  float* rec_return;      // [B]
  int32_t* rec_len;       // [B]
  uint64_t seed, ctr;
  int B, obs, act, C, c, max_episode_steps, auto_reset, ignore_terminations;
  float p_term, noise_std, reward_noise_std;
};

// one warp per env; draws in the order of env_finish_kernel (C = 1) / env_substep_kernel + chunk_finish_kernel (C > 1)
__global__ void __launch_bounds__(256) eval_env_substep_kernel(EvalArgs p) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= p.B) return;
  curandStatePhilox4_32_10_t st;
  if (!p.noise) curand_init(p.seed, (unsigned long long)row * 32ull + lane, (p.ctr * (uint64_t)p.C + p.c) * 64ull, &st);
  const size_t nrow = (size_t)p.C * (p.obs + 2) + p.obs;
  const float* nz = p.noise ? p.noise + (size_t)row * nrow + (size_t)p.c * (p.obs + 2) : nullptr;
  const float* act = p.action + (size_t)row * p.C * p.act + (size_t)p.c * p.act;
  float sq = 0.f;
  for (int j = lane; j < p.obs; j += 32) {
    float z = p.z[(size_t)row * p.obs + j];
    for (int a = 0; a < p.act; ++a) z = fmaf(act[a], p.w_a[a * p.obs + j], z);
    const float eps = nz ? nz[j] : curand_normal(&st);
    const float s = tanhf(z + p.noise_std * eps);
    p.out_state[(size_t)row * p.obs + j] = s;
    sq += s * s;
  }
  sq = rb::warp_sum(sq);
  const bool last = p.c == p.C - 1;
  int reset = 0;
  if (lane == 0) {
    const float eps_r = nz ? nz[p.obs] : curand_normal(&st);
    const float u = nz ? nz[p.obs + 1] : curand_uniform(&st);
    const float r = -sq / (float)p.obs + p.reward_noise_std * eps_r;
    int el = p.elapsed[row] + 1;
    const bool success = u < p.p_term;
    bool term = success;
    const bool trunc = p.max_episode_steps > 0 && el >= p.max_episode_steps;
    float ret = p.ep_return[row] + r;  // _record_metrics: self.returns += step_reward
    uint8_t f = p.ep_flags[row];
    if (success) f |= kSuccessOnce;
    if (p.ignore_terminations) term = false;  // step(): terminations[:] = False after recording
    if (p.c == 0) f &= (uint8_t)~(kChunkTerm | kChunkTrunc);
    if (term) f |= kChunkTerm;
    if (trunc) f |= kChunkTrunc;
    if (last) {
      const bool done = (f & (kChunkTerm | kChunkTrunc)) != 0;
      const bool reported = p.auto_reset ? done : (done && !(f & kPrevDone));  // env_evaluate_step: newly_done
      p.rec_flags[row] = (uint8_t)((reported ? 1 : 0) | ((f & kSuccessOnce) ? 2 : 0) | (success ? 4 : 0));
      p.rec_return[row] = ret;
      p.rec_len[row] = el;
      f &= (uint8_t)~(kChunkTerm | kChunkTrunc);
      if (!p.auto_reset && done) f |= kPrevDone;
      reset = done && p.auto_reset;
      if (reset) {  // _handle_auto_reset -> reset(env_idx) -> _reset_metrics(env_idx)
        el = 0;
        ret = 0.f;
        f &= (uint8_t)~kSuccessOnce;
      }
    }
    p.elapsed[row] = el;
    p.ep_return[row] = ret;
    p.ep_flags[row] = f;
  }
  if (!last) return;
  reset = __shfl_sync(0xffffffffu, reset, 0);
  if (!reset) return;
  if (!p.noise && p.C > 1)  // chunk_finish_kernel's reset window: 32 outputs behind the last sub-step's window
    curand_init(p.seed, (unsigned long long)row * 32ull + lane, (p.ctr * (uint64_t)p.C + (p.C - 1)) * 64ull + 32ull, &st);
  const float* rz = p.noise ? p.noise + (size_t)row * nrow + (size_t)p.C * (p.obs + 2) : nullptr;
  for (int j = lane; j < p.obs; j += 32) p.out_state[(size_t)row * p.obs + j] = rz ? rz[j] : curand_normal(&st);
}

constexpr int kRedThreads = 256;
constexpr int kRedMaxBlocks = RB200_EVAL_MAX_PARTS;

// per block: {sum return, sum len, sum reward, sum success_once, sum success_at_end, count} of the reported records
// in its fixed slice, in a fixed order (no atomics)
__global__ void __launch_bounds__(kRedThreads) eval_metrics_part_kernel(const uint8_t* __restrict__ flags,
                                                                        const float* __restrict__ ret,
                                                                        const int32_t* __restrict__ len, int64_t n,
                                                                        int64_t per_block, double* __restrict__ part) {
  __shared__ double sm[6 * 32];
  double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  const int64_t lo = (int64_t)blockIdx.x * per_block;
  const int64_t hi = lo + per_block < n ? lo + per_block : n;
  for (int64_t i = lo + threadIdx.x; i < hi; i += kRedThreads) {
    const uint8_t f = flags[i];
    if (!(f & 1)) continue;
    const float r = ret[i];
    const int32_t l = len[i];
    v[0] += (double)r;
    v[1] += (double)l;
    v[2] += (double)(r / (float)l);  // _record_metrics: reward = return / episode_len, fp32
    v[3] += (f & 2) ? 1.0 : 0.0;
    v[4] += (f & 4) ? 1.0 : 0.0;
    v[5] += 1.0;
  }
  rb::block_sum<6>(v, sm);
  if (threadIdx.x == 0)
    for (int k = 0; k < 6; ++k) part[blockIdx.x * 6 + k] = v[k];
}

__global__ void __launch_bounds__(kRedThreads) eval_metrics_final_kernel(const double* __restrict__ part, int nparts,
                                                                         double* __restrict__ out6) {
  __shared__ double sm[6 * 32];
  double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (int b = threadIdx.x; b < nparts; b += kRedThreads)
    for (int k = 0; k < 6; ++k) v[k] += part[b * 6 + k];
  rb::block_sum<6>(v, sm);
  if (threadIdx.x == 0)
    for (int k = 0; k < 6; ++k) out6[k] = v[k];
}

}  // namespace

extern "C" int rb200_synth_env_eval_step(const float* w_s, const float* w_a, float* state, const float* chunk_actions,
                                         const float* noise, int32_t* elapsed, float* ep_return, uint8_t* ep_flags,
                                         uint8_t* rec_flags, float* rec_return, int32_t* rec_len, float* scratch, int B,
                                         int obs, int act, int C, int max_episode_steps, int auto_reset,
                                         int ignore_terminations, float p_term, float noise_std, float reward_noise_std,
                                         uint64_t seed, uint64_t step, rb200_stream_t stream) {
  if (!w_s || !w_a || !state || !chunk_actions || !elapsed || !ep_return || !ep_flags || !rec_flags || !rec_return ||
      !rec_len || !scratch)
    return RB200_E_NULL;
  if (B <= 0 || obs <= 0 || act <= 0 || C <= 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  const size_t n = (size_t)B * obs;
  float* z = scratch;
  float* ping[2] = {scratch + n, scratch + 2 * n};
  const float* cur = state;
  for (int c = 0; c < C; ++c) {
    GemmArgs g{};
    g.A = cur; g.lda = obs; g.B = w_s; g.ldb = obs; g.C = z; g.ldc = obs;
    g.M = B; g.N = obs; g.K = obs; g.k_per_split = 1 << 30;
    int e = launch_gemm<A_KCONTIG, B_NCONTIG, EPI_STORE>(g, 1, st);  // z = s . W_s
    if (e) return e;
    EvalArgs p{};
    p.z = z; p.action = chunk_actions; p.w_a = w_a; p.noise = noise;
    p.out_state = c == C - 1 ? state : ping[c & 1];
    p.elapsed = elapsed; p.ep_return = ep_return; p.ep_flags = ep_flags;
    p.rec_flags = rec_flags; p.rec_return = rec_return; p.rec_len = rec_len;
    p.seed = seed; p.ctr = step; p.B = B; p.obs = obs; p.act = act; p.C = C; p.c = c;
    p.max_episode_steps = max_episode_steps; p.auto_reset = auto_reset; p.ignore_terminations = ignore_terminations;
    p.p_term = p_term; p.noise_std = noise_std; p.reward_noise_std = reward_noise_std;
    eval_env_substep_kernel<<<(B + 7) / 8, 256, 0, st>>>(p); rb::count_launch();
    cudaError_t ce = cudaPeekAtLastError();
    if (ce != cudaSuccess) return (int)ce;
    cur = p.out_state;
  }
  return RB200_OK;
}

extern "C" int rb200_eval_metrics(const uint8_t* rec_flags, const float* rec_return, const int32_t* rec_len, int64_t n,
                                  double* part, double* out6, rb200_stream_t stream) {
  if (!rec_flags || !rec_return || !rec_len || !part || !out6) return RB200_E_NULL;
  if (n <= 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  // the slice of each block depends on n only, so the summation order is the same on every call
  int64_t blocks = (n + 4 * kRedThreads - 1) / (4 * kRedThreads);
  if (blocks > kRedMaxBlocks) blocks = kRedMaxBlocks;
  const int64_t per_block = (n + blocks - 1) / blocks;
  eval_metrics_part_kernel<<<(int)blocks, kRedThreads, 0, st>>>(rec_flags, rec_return, rec_len, n, per_block, part);
  rb::count_launch();
  eval_metrics_final_kernel<<<1, kRedThreads, 0, st>>>(part, (int)blocks, out6);
  rb::count_launch();
  RB_RETURN_LAUNCH();
}
