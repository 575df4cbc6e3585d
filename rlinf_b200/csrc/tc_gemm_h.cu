// K3 tensor-core path: fp32-accurate GEMMs on tcgen05 `kind::f16` through a 2-way fp16 split.
//     a = a_hi + a_lo, b = b_hi + b_lo (fp16 numbers, 11 significant bits each; operands pre-scaled by a power of two so
//     that both halves stay in fp16's normal range);  a.b ~= a_lo.b_hi + a_hi.b_lo + a_hi.b_hi   (dropped a_lo.b_lo ~ 2^-22)
// This is the three-MMA compensation of a 3xTF32 GEMM with the same 2^-22 truncation, but
//   * kind::f16 issues at twice the kind::tf32 rate, so an fp32-accurate product costs peak/3 instead of peak/6;
//   * operands are 2 bytes in shared memory: the three MMAs re-read 72 KB per 128x256x32 k-block instead of 147 KB and
//     the weight tiles TMA-fill 32 KB instead of 64 KB (a 3xTF32 version, measured in round 1, was bound by exactly this
//     shared-memory traffic);
//   * the weights are packed per k-block as pre-swizzled fp16 (hi | lo) tiles - a K-major forward pack and an MN-major dgrad
//     pack per matrix, written by one pack kernel - and fetched with ONE 32 KB bulk copy per k-block;
//   * one launch serves BOTH towers (policy backbone + value MLP have identical shapes): grouped tile scheduling halves
//     the launches and fills the tail wave of small per-rank batches.
// Activations / activation gradients stay plain fp32 in HBM (one copy); the streamed operand is TMA-landed as fp32
// (SWIZZLE_128B) and split by transform warps into two fp16 SWIZZLE_64B tiles.  Gradients are tiny (1e-6 .. 1e-10):
// their producer publishes max|x| and the consumer scales by 2^s (exact) so that the maximum sits at 2^13; the fp32
// accumulator is scaled back in the epilogue (exact).
// Reference op chains replaced: nn.Linear + tanh of MLPPolicy.backbone / ValueHead.mlp
// (rlinf/models/embodiment/mlp_policy/mlp_policy.py:91-98, modules/value_head.py:37-45) and autograd's dgrad / wgrad.
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc_gemm.cuh"
#include "tma.cuh"

namespace rb {
namespace tch {

using rb::tc::BK;
using rb::tc::BM;
using rb::tc::BN;

// Two rings (round 2, second half).  The first version kept the fp32 landing tile, its fp16 halves and the weight
// tile in ONE 64 KB stage, 3 stages deep: a stage stayed busy for load latency (~3000 clk under HBM load) + transform
// (~700) + MMA (768), i.e. ~1500 clk per k-block against 768 of MMA (tools/gemm_role_probe.py).  Now the fp32 landing
// tiles have their own deep ring (freed as soon as the transform has read them: 6 x 16 KB of activations in flight per
// SM) and the MMA operands (A hi | lo written by the transform, weight hi | lo landed by TMA) a shallow one.
constexpr int kAStages = 4;         // fp32 landing ring of the streamed operand
constexpr int kBStages = 2;         // fp16 A hi | lo slots (written by the transform)
constexpr int kWStages = 3;         // weight tile ring (one 32 KB bulk copy each): with two slots the MMA waited ~650 clk
                                    // per k-block for the weight tile (32 KB over L2 -> SM take ~2000 clk to arrive)
constexpr int kA32 = BM * BK * 4;   // 16 KB fp32 landing tile of the streamed operand
constexpr int kA16 = BM * BK * 2;   //  8 KB per fp16 half
constexpr int kB16 = BN * BK * 2;   // 16 KB per fp16 half of the weight tile
constexpr int kOpBytes = 2 * kA16;  // 16 KB: A hi | A lo
constexpr int kWBytes = 2 * kB16;   // 32 KB: W hi | W lo
constexpr int kRingBytes = kAStages * kA32 + kBStages * kOpBytes + kWStages * kWBytes;  // 64 + 32 + 96 = 192 KB
constexpr int kXfWarps = 4;   // transform warps of the forward / dgrad kernel, one per scheduler (8 measured no faster:
                              // DESIGN.md section 4)
constexpr int kEpiWarps = 8;  // two per TMEM lane quarter, 128 of the 256 output columns each: the bias+tanh / (1-h^2)
                              // epilogue of one warp per scheduler took 7.8 k cycles per tile against 6.1 k of MMA
constexpr int kThreads = 32 * (2 + kXfWarps + kEpiWarps);  // producer, MMA, transform, epilogue
constexpr int kStagingBytes = kEpiWarps * 4096;  // one [32 x 32] fp32 staging tile per epilogue warp
constexpr int kTmemCols = 512;
constexpr int kWeightScaleLog2 = 10;  // weights are stored as fp16 (hi, lo) of w * 2^10 (|w| <~ 1: both halves normal)

// ---- PTX wrappers -----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tma::smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tma::smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
      ::"r"(d_tmem), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, "
      "%24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 1-D bulk copy global -> shared, completion counted on an mbarrier
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   tma::smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(tma::smem_u32(bar))
               : "memory");
}

// ---- UMMA shared-memory descriptors (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp; canonical layouts in
//      cute/atom/mma_traits_sm100.hpp:167-203).  start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) |
//      layout_type [61,64): 2 = SWIZZLE_128B, 4 = SWIZZLE_64B ------------------------------------------------------------
// K-major, SWIZZLE_64B: rows of 32 fp16 (64 B), 8-row groups 512 B apart (LBO unused for swizzled K-major).
__device__ __forceinline__ uint64_t desc_k_sw64(uint32_t addr) {
  return (uint64_t)((addr & 0x3ffffu) >> 4) | (1ull << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
// MN-major, SWIZZLE_128B: ((8,n),(8,k)) in 16-byte units = 64 fp16 along MN per row (128 B), 8 K-rows per atom (SBO = 1024 B
// between atoms along K), MN groups of 64 elements LBO bytes apart.
__device__ __forceinline__ uint64_t desc_mn_sw128(uint32_t addr, uint32_t lbo) {
  return (uint64_t)((addr & 0x3ffffu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
         (2ull << 61);
}
// MN-major, SWIZZLE_64B: ((4,n),(8,k)) = 32 fp16 along MN per row (64 B), 8 K-rows per atom (SBO = 512 B), MN groups LBO apart.
__device__ __forceinline__ uint64_t desc_mn_sw64(uint32_t addr, uint32_t lbo) {
  return (uint64_t)((addr & 0x3ffffu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) |
         (4ull << 61);
}
// kind::f16 instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 [4,6)=1, a/b format F16 = 0 [7,10),[10,13),
// a_major bit 15, b_major bit 16 (0 = K, 1 = MN), N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ float tanh_fast(float x) {
  const float t = __expf(-2.0f * fabsf(x));
  return copysignf(__fdividef(1.0f - t, 1.0f + t), x);
}

// 2^s as a float (s in [-126, 127])
__device__ __forceinline__ float pow2i(int s) { return __int_as_float((s + 127) << 23); }
// power-of-two scale that brings max|x| = amax to [2^13, 2^14): fp16 keeps 11 bits for every |x| >= amax * 2^-27
__device__ __forceinline__ int scale_log2_for(float amax) {
  const int e = (int)((__float_as_uint(amax) >> 23) & 0xffu) - 127;
  if (!(amax > 0.0f) || e < -120) return 0;
  int s = 13 - e;
  return s > 100 ? 100 : (s < -100 ? -100 : s);
}

// fp32 [R rows x 32 floats] SWIZZLE_128B tile -> fp16 hi / lo [R rows x 32 halfs] SWIZZLE_64B tiles; item = (row, 8 floats)
template <int NT>
__device__ __forceinline__ void split_tile(const uint8_t* __restrict__ src, uint8_t* __restrict__ hi, uint8_t* __restrict__ lo,
                                           int rows, int t, float scale) {
  const int items = rows * 4;
#pragma unroll 2
  for (int i = t; i < items; i += NT) {
    const int r = i >> 2, cp = i & 3;
    const uint8_t* srow = src + r * 128;
    const float4 x0 = *reinterpret_cast<const float4*>(srow + (((2 * cp) ^ (r & 7)) << 4));
    const float4 x1 = *reinterpret_cast<const float4*>(srow + (((2 * cp + 1) ^ (r & 7)) << 4));
    const float v[8] = {x0.x * scale, x0.y * scale, x0.z * scale, x0.w * scale,
                        x1.x * scale, x1.y * scale, x1.z * scale, x1.w * scale};
    uint32_t h[4], l[4];  // packed half2 words (no 16-byte reinterpretation of a 4-byte-aligned local array)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __half2 hh = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
      const float2 hf = __half22float2(hh);
      const __half2 ll = __floats2half2_rn(v[2 * j] - hf.x, v[2 * j + 1] - hf.y);
      h[j] = *reinterpret_cast<const uint32_t*>(&hh);
      l[j] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    const int doff = r * 64 + ((cp ^ ((r >> 1) & 3)) << 4);
    *reinterpret_cast<uint4*>(hi + doff) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + doff) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// PROF instantiations (tools/gemm_role_probe.py): cycles each role of CTA 0 spends waiting / working
template <bool PROF>
__device__ __forceinline__ void wait_bar(uint64_t* bar, uint32_t parity, long long& acc) {
  if constexpr (PROF) {
    const long long t0 = clock64();
    tma::mbar_wait(bar, parity);
    acc += clock64() - t0;
  } else {
    tma::mbar_wait(bar, parity);
  }
}

struct __align__(16) Barriers {
  uint64_t full_a[kAStages];   // fp32 landing tile arrived (TMA tx bytes)
  uint64_t empty_a[kAStages];  // transform warps have read it
  uint64_t xf[kBStages];       // transform warps have written A hi | lo
  uint64_t empty_b[kBStages];  // MMAs reading the A slot have completed (tcgen05.commit)
  uint64_t full_w[kWStages];   // weight tile arrived (bulk-copy tx bytes)
  uint64_t empty_w[kWStages];  // MMAs reading the weight slot have completed (tcgen05.commit)
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
  uint32_t pad_[3];
  alignas(16) float bias[BN];  // (read as float4) forward: the layer bias; dgrad: this CTA's column sums of the output
};

struct Group {
  const float* bias;    // [256]                         (EPI_BIAS_TANH)
  const float* h;       // [M,256] previous activation   (EPI_TANHGRAD)
  float* colsum;        // [256] += column sums of the output (per-CTA rows of the partials buffer, summed in order), or NULL
  const float* amax_in; // [1] max|A| published by A's producer (gradient GEMMs), or NULL = no scaling
  float* amax_out;      // [1] atomicMax of |output| for the next gradient GEMM, or NULL
};

struct GemmParams {
  CUtensorMap a[2], c[2];
  const uint8_t* wpack[2];  // packed weight tiles of each group (32 KB per k-block: hi | lo)
  Group g[2];
  int64_t M;
  int K;
  int epi;
  int b_mn;  // 0: weights K-major (forward), 1: MN-major (dgrad: B(n = in, k = out) = W[out][in])
  int ngroups;
  float* part;      // [CTAs per group][ngroups][256] column sums (EPI_TANHGRAD with colsum)
  long long* prof;  // [16] (PROF instantiation only)
};

template <bool PROF>
__global__ void __launch_bounds__(kThreads, 1) tc_h_gemm_kernel(const __grid_constant__ GemmParams P) {
  long long pc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  const long long t_start = PROF ? clock64() : 0;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (tma::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ring_a = smem;                       // kAStages x [128 rows x 32 fp32] SWIZZLE_128B
  uint8_t* ring_w = smem + kAStages * kA32;                 // kWStages x (W hi | W lo), 1024-aligned (MN-major SWIZZLE_128B)
  uint8_t* ring_b = ring_w + kWStages * kWBytes;            // kBStages x (A hi | A lo)
  uint8_t* staging = smem + kRingBytes;
  Barriers* bars = reinterpret_cast<Barriers*>(staging + kStagingBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = blockIdx.x % P.ngroups;
  const int cta = blockIdx.x / P.ngroups, n_cta = gridDim.x / P.ngroups;
  const Group& G = P.g[grp];
  const int64_t n_tiles = (P.M + BM - 1) / BM;
  const int n_kb = P.K / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kAStages; ++s) {
      tma::mbar_init(&bars->full_a[s], 1);
      tma::mbar_init(&bars->empty_a[s], kXfWarps);
    }
    for (int s = 0; s < kBStages; ++s) {
      tma::mbar_init(&bars->xf[s], kXfWarps);
      tma::mbar_init(&bars->empty_b[s], 1);
    }
    for (int s = 0; s < kWStages; ++s) {
      tma::mbar_init(&bars->full_w[s], 1);
      tma::mbar_init(&bars->empty_w[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      tma::mbar_init(&bars->tmem_full[b], 1);
      tma::mbar_init(&bars->tmem_empty[b], kEpiWarps);
    }
    tma::fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(&bars->tmem_base, kTmemCols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < BN; i += kThreads) bars->bias[i] = (P.epi == rb::tc::EPI_BIAS_TANH) ? G.bias[i] : 0.f;
  // dgrad column sums: each epilogue lane sums its column over the rows of its lane quarter of every tile (csum[i] for
  // columns c_lo + 32 i + lane); the quarters are added into bars->bias one after another at the end
  float csum[4] = {0.f, 0.f, 0.f, 0.f};
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = bars->tmem_base;
  // operand scaling: A by 2^sa (from the published amax), weights are stored * 2^kWeightScaleLog2
  const int sa = G.amax_in ? scale_log2_for(__ldg(G.amax_in)) : 0;
  const float a_scale = pow2i(sa);
  const float out_scale = pow2i(-(sa + kWeightScaleLog2));

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      tma::prefetch_desc(&P.a[grp]);
      const int64_t my_tiles = n_tiles > cta ? (n_tiles - cta + n_cta - 1) / n_cta : 0;
      const int64_t total = my_tiles * n_kb;
      // two independent streams issued by one thread: poll both rings, load whichever has a free slot
      int64_t ja = 0, jb = 0;
      uint32_t sa = 0, pa = 0, sb = 0, pb = 0;
      while (ja < total || jb < total) {
        if (ja < total && tma::mbar_try_wait(&bars->empty_a[sa], pa ^ 1u)) {
          const int kb = (int)(ja % n_kb);
          const int m0 = (int)((cta + (ja / n_kb) * n_cta) * BM);
          tma::mbar_arrive_expect_tx(&bars->full_a[sa], kA32);
          tma::load_2d(ring_a + sa * kA32, &P.a[grp], kb * BK, m0, &bars->full_a[sa]);  // rows >= M are zero-filled
          ++ja;
          if (++sa == kAStages) { sa = 0; pa ^= 1u; }
        }
        if (jb < total && tma::mbar_try_wait(&bars->empty_w[sb], pb ^ 1u)) {
          const int kb = (int)(jb % n_kb);
          tma::mbar_arrive_expect_tx(&bars->full_w[sb], kWBytes);
          bulk_load(ring_w + sb * kWBytes, P.wpack[grp] + (size_t)kb * kWBytes, kWBytes, &bars->full_w[sb]);  // hi | lo
          ++jb;
          if (++sb == kWStages) { sb = 0; pb ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0) {
      const uint32_t idesc = idesc_f16(BM, BN, 0, P.b_mn);
      uint32_t it = 0, tcount = 0;
      for (int64_t tile = cta; tile < n_tiles; tile += n_cta, ++tcount) {
        const uint32_t buf = tcount & 1u;
        const uint32_t bph = (tcount >> 1) & 1u;
        wait_bar<PROF>(&bars->tmem_empty[buf], bph ^ 1u, pc[1]);
        fence_after_sync();
        const uint32_t d_tmem = tmem_base + buf * BN;
        for (int kb = 0; kb < n_kb; ++kb, ++it) {
          const int s = it % kBStages;
          const uint32_t ph = (it / kBStages) & 1u;
          const int sw = it % kWStages;
          const uint32_t phw = (it / kWStages) & 1u;
          wait_bar<PROF>(&bars->full_w[sw], phw, pc[2]);
          wait_bar<PROF>(&bars->xf[s], ph, pc[3]);
          fence_after_sync();
          const uint32_t sa32 = tma::smem_u32(ring_b + s * kOpBytes);
          const uint64_t a_hi = desc_k_sw64(sa32), a_lo = desc_k_sw64(sa32 + kA16);
          const uint32_t sbase = tma::smem_u32(ring_w + sw * kWBytes);
          const uint64_t b_hi = P.b_mn ? desc_mn_sw128(sbase, 4096) : desc_k_sw64(sbase);
          const uint64_t b_lo = P.b_mn ? desc_mn_sw128(sbase + kB16, 4096) : desc_k_sw64(sbase + kB16);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t ka = (uint64_t)((k * 32) >> 4);                        // 16 fp16 = 32 B along a 64-B row
            const uint64_t kbo = P.b_mn ? (uint64_t)((k * 2048) >> 4) : ka;       // MN-major: 16 K-rows of 128 B
            const uint32_t acc = (kb > 0 || k > 0) ? 1u : 0u;
            mma_f16(d_tmem, a_lo + ka, b_hi + kbo, idesc, acc);  // small terms first
            mma_f16(d_tmem, a_hi + ka, b_lo + kbo, idesc, 1u);
            mma_f16(d_tmem, a_hi + ka, b_hi + kbo, idesc, 1u);
          }
          mma_commit(&bars->empty_b[s]);
          mma_commit(&bars->empty_w[sw]);
        }
        mma_commit(&bars->tmem_full[buf]);
      }
    }
  } else if (warp < 2 + kXfWarps) {
    // ================= transform warps: fp32 A tile -> (A_hi, A_lo) fp16 tiles =================
    const int t = threadIdx.x - 64;
    uint32_t sa = 0, pa = 0, sb = 0, pb = 0;
    for (int64_t tile = cta; tile < n_tiles; tile += n_cta) {
      for (int kb = 0; kb < n_kb; ++kb) {
        wait_bar<PROF>(&bars->full_a[sa], pa, pc[4]);           // the fp32 tile has landed
        wait_bar<PROF>(&bars->empty_b[sb], pb ^ 1u, pc[0]);     // the operand slot's previous MMAs are done
        const long long t_w0 = PROF ? clock64() : 0;
        uint8_t* dst = ring_b + sb * kOpBytes;
        split_tile<32 * kXfWarps>(ring_a + sa * kA32, dst, dst + kA16, BM, t, a_scale);
        tma::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma::mbar_arrive(&bars->xf[sb]);
          tma::mbar_arrive(&bars->empty_a[sa]);
        }
        if constexpr (PROF) pc[5] += clock64() - t_w0;
        if (++sa == kAStages) { sa = 0; pa ^= 1u; }
        if (++sb == kBStages) { sb = 0; pb ^= 1u; }
      }
    }
  } else {
    // ================= epilogue warps =================
    const int q = warp & 3;
    const int ew = warp - (2 + kXfWarps);
    const int c_lo = (ew >> 2) * (BN / 2);  // this warp's half of the output columns
    float4 (*sh)[8] = reinterpret_cast<float4 (*)[8]>(staging + ew * 4096);
    if (lane == 0) tma::prefetch_desc(&P.c[grp]);
    const int rs = lane >> 3, c4 = lane & 7;
    float4 hp[8];
    auto load_h = [&](int64_t r0, int cc) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int64_t gr = r0 + i * 4 + rs;
        hp[i] = gr < P.M ? __ldg(reinterpret_cast<const float4*>(G.h + gr * BN + cc) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    if (P.epi == rb::tc::EPI_TANHGRAD && (int64_t)cta < n_tiles) load_h((int64_t)cta * BM + q * 32, c_lo);
    float vmax = 0.f;
    uint32_t tcount = 0;
    for (int64_t tile = cta; tile < n_tiles; tile += n_cta, ++tcount) {
      const uint32_t buf = tcount & 1u;
      const uint32_t bph = (tcount >> 1) & 1u;
      wait_bar<PROF>(&bars->tmem_full[buf], bph, pc[6]);
      const long long t_e0 = PROF ? clock64() : 0;
      fence_after_sync();
      const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN;
      const int64_t row0 = tile * BM + q * 32;
#pragma unroll 1
      for (int c0 = c_lo; c0 < c_lo + BN / 2; c0 += 32) {
        if (lane == 0) tma::store_wait_read();  // the previous tile store has finished reading the staging tile
        __syncwarp();
        uint32_t r[32];
        tmem_ld32(taddr0 + c0, r);
        if (P.epi == rb::tc::EPI_TANHGRAD) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = i * 4 + rs;
            sh[rr][c4 ^ (rr & 7)] = hp[i];
          }
          __syncwarp();
          if (c0 + 32 < c_lo + BN / 2) load_h(row0, c0 + 32);
          else if (tile + n_cta < n_tiles) load_h((tile + n_cta) * BM + q * 32, c_lo);
        }
        tmem_ld_wait();
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          float4 v;
          const float a0 = __uint_as_float(r[j4 * 4 + 0]) * out_scale, a1 = __uint_as_float(r[j4 * 4 + 1]) * out_scale;
          const float a2 = __uint_as_float(r[j4 * 4 + 2]) * out_scale, a3 = __uint_as_float(r[j4 * 4 + 3]) * out_scale;
          if (P.epi == rb::tc::EPI_STORE) {
            v = make_float4(a0, a1, a2, a3);
          } else if (P.epi == rb::tc::EPI_BIAS_TANH) {
            const float4 b = *reinterpret_cast<const float4*>(&bars->bias[c0 + j4 * 4]);
            v = make_float4(tanh_fast(a0 + b.x), tanh_fast(a1 + b.y), tanh_fast(a2 + b.z), tanh_fast(a3 + b.w));
          } else {
            const float4 h = sh[lane][j4 ^ (lane & 7)];
            v = make_float4(a0 * (1.0f - h.x * h.x), a1 * (1.0f - h.y * h.y), a2 * (1.0f - h.z * h.z),
                            a3 * (1.0f - h.w * h.w));
            vmax = fmaxf(vmax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
          }
          sh[lane][j4 ^ (lane & 7)] = v;
        }
        tma::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma::store_2d(&P.c[grp], &sh[0][0], c0, (int)row0);  // rows >= M are clipped
          tma::store_commit();
        }
        if (G.colsum != nullptr && P.epi == rb::tc::EPI_TANHGRAD) {
          const int ch = lane >> 2, el = lane & 3;
          float cs = 0.f;
#pragma unroll 8
          for (int rr = 0; rr < 32; ++rr) cs += reinterpret_cast<const float*>(&sh[rr][ch ^ (rr & 7)])[el];
          csum[(c0 - c_lo) >> 5] += cs;
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) tma::mbar_arrive(&bars->tmem_empty[buf]);
      if constexpr (PROF) pc[7] += clock64() - t_e0;
    }
    if (G.amax_out != nullptr && P.epi == rb::tc::EPI_TANHGRAD) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
      if (lane == 0 && vmax > 0.f) atomicMax(reinterpret_cast<unsigned int*>(G.amax_out), __float_as_uint(vmax));
    }
    if (lane == 0) tma::store_wait_all();
  }

  if constexpr (PROF) {
    if (blockIdx.x == 0 && P.prof && lane == 0 && (warp == 0 || warp == 1 || warp == 2 || warp == 2 + kXfWarps)) {
      for (int i = 0; i < 8; ++i)
        if (pc[i]) atomicAdd(reinterpret_cast<unsigned long long*>(P.prof + i), (unsigned long long)pc[i]);
      if (warp == 0) atomicAdd(reinterpret_cast<unsigned long long*>(P.prof + 8), (unsigned long long)(clock64() - t_start));
    }
  }
  fence_before_sync();
  __syncthreads();
  if (G.colsum != nullptr && P.epi == rb::tc::EPI_TANHGRAD) {
    const int ew = warp - (2 + kXfWarps);
    for (int qq = 0; qq < 4; ++qq) {
      if (ew >= 0 && (warp & 3) == qq) {
        const int c_lo = (ew >> 2) * (BN / 2);
#pragma unroll
        for (int i = 0; i < 4; ++i) bars->bias[c_lo + 32 * i + lane] += csum[i];
      }
      __syncthreads();
    }
    for (int i = threadIdx.x; i < BN; i += kThreads) P.part[((size_t)cta * P.ngroups + grp) * BN + i] = bars->bias[i];
  }
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Weight-gradient GEMM:  dW[256, IN] += sum_m dZ[m, :]^T . H[m, :]     (IN % 32 == 0, <= 256), both operands MN-major.
// Per k-block of 32 samples: TMA lands fp32 boxes {32 floats, 32 samples} (SWIZZLE_128B), 8 transform warps split them
// into fp16 SWIZZLE_64B groups [32 samples x 32 features] = the canonical MN-major SW64 layout with LBO = 2048 B between
// 32-feature groups and SBO = 512 B between 8-sample atoms; one K=16 MMA step spans two atoms (1024 B).
// Grid = ngroups x 2 output tiles (128 rows of dW) x sample chunks; each chunk stores its partial dW in a row of the
// partials buffer and rb::sum_partials adds the chunks to dW in a fixed order (no float atomics: bit-reproducible).
// ---------------------------------------------------------------------------------------------------------------
// Two rings, as in the forward kernel: fp32 landing tiles (dZ 16 KB + H 32 KB per k-block of 32 samples) three deep,
// freed as soon as the transform has read them, and ONE fp16 operand slot (dZ hi | lo, H hi | lo: 48 KB) that transform
// and MMA take turns on.  The first version kept both in one 96 KB stage, two deep: a stage was held for load latency +
// transform + MMA and the period was (3000 + 500 + 768) / 2 clk per k-block.
constexpr int kWgLand = 3;
constexpr int kWgA32 = 128 * BK * 4, kWgA16 = 128 * BK * 2;  // 16 KB / 8 KB
constexpr int kWgB32 = 256 * BK * 4, kWgB16 = 256 * BK * 2;  // 32 KB / 16 KB (sized for IN = 256)
constexpr int kWgLandBytes = kWgA32 + kWgB32;                // 48 KB
constexpr int kWgOpBytes = 2 * kWgA16 + 2 * kWgB16;          // 48 KB
constexpr int kWgRingBytes = kWgLand * kWgLandBytes + kWgOpBytes;  // 192 KB
constexpr int kWgXfWarps = 16;  // four per scheduler: the fp32 -> fp16 split of 48 KB per k-block took 1025 clk with 8 (tools/gemm_role_probe.py)
constexpr int kWgThreads = 32 * (2 + 4 + kWgXfWarps);

struct WgBarriers {
  uint64_t full[kWgLand], empty[kWgLand];  // landing ring: TMA tx bytes / transform warps done reading
  uint64_t xf, op_free;                    // operand slot: written by the transform / its MMAs have completed
  uint64_t tmem_full;
  uint32_t tmem_base, pad_;
};

struct WgradParams {
  CUtensorMap z[2], h[2];
  float* dW[2];
  float* part;             // [chunks][ngroups][256 * IN] partial dW of each sample chunk
  const float* amax_z[2];  // max|dZ| per group (or NULL)
  int64_t n;
  int IN, kb_per_chunk, ngroups;
  long long* prof;  // [16] (PROF instantiation: slots 9..15)
};

template <bool PROF>
__global__ void __launch_bounds__(kWgThreads, 1) tc_h_wgrad_kernel(const __grid_constant__ WgradParams P) {
  long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long t_start = PROF ? clock64() : 0;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (tma::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* op = smem + kWgLand * kWgLandBytes;  // dZ hi | dZ lo | H hi | H lo
  WgBarriers* bars = reinterpret_cast<WgBarriers*>(smem + kWgRingBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = blockIdx.x % P.ngroups;
  const int rest = blockIdx.x / P.ngroups;
  const int out_tile = rest & 1, chunk = rest >> 1;
  const int IN = P.IN;
  const int n_kb_total = (int)((P.n + BK - 1) / BK);
  const int kb0 = chunk * P.kb_per_chunk;
  const int kb1 = (kb0 + P.kb_per_chunk < n_kb_total) ? kb0 + P.kb_per_chunk : n_kb_total;
  const int n_kb = kb1 - kb0;
  const uint32_t b32_bytes = (uint32_t)IN * BK * 4;
  const uint32_t tmem_cols = IN <= 32 ? 32u : (IN <= 64 ? 64u : (IN <= 128 ? 128u : 256u));

  if (threadIdx.x == 0) {
    for (int s = 0; s < kWgLand; ++s) {
      tma::mbar_init(&bars->full[s], 1);
      tma::mbar_init(&bars->empty[s], kWgXfWarps);
    }
    tma::mbar_init(&bars->xf, kWgXfWarps);
    tma::mbar_init(&bars->op_free, 1);
    tma::mbar_init(&bars->tmem_full, 1);
    tma::fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(&bars->tmem_base, tmem_cols);
    tmem_relinquish();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = bars->tmem_base;
  const int sz = P.amax_z[grp] ? scale_log2_for(__ldg(P.amax_z[grp])) : 0;
  const float z_scale = pow2i(sz), out_scale = pow2i(-sz);

  if (n_kb > 0) {
    if (warp == 0) {
      // boxes {32 floats, 32 samples} with SWIZZLE_128B, one lane per box (a single plain [32 x 128|IN] box per operand
      // was tried: 64 row requests instead of 384 per k-block, but the unswizzled landing tile costs more in the
      // transform than the requests save: 191 vs 163 us, profiles/r02_tc_h_unit_timings.txt)
      const int gB = IN / 32;
      const int n_box = 4 + gB;
      for (int it = 0; it < n_kb; ++it) {
        const int s = it % kWgLand;
        const uint32_t ph = (it / kWgLand) & 1u;
        if (lane == 0) {
          wait_bar<PROF>(&bars->empty[s], ph ^ 1u, pc[0]);
          tma::mbar_arrive_expect_tx(&bars->full[s], kWgA32 + b32_bytes);
        }
        __syncwarp();
        if (lane < n_box) {
          uint8_t* st = smem + s * kWgLandBytes;
          const int m0 = (kb0 + it) * BK;  // samples >= n are zero-filled
          if (lane < 4) tma::load_2d(st + lane * 4096, &P.z[grp], out_tile * 128 + lane * 32, m0, &bars->full[s]);
          else tma::load_2d(st + kWgA32 + (lane - 4) * 4096, &P.h[grp], (lane - 4) * 32, m0, &bars->full[s]);
        }
      }
    } else if (warp == 1) {
      if (lane == 0) {
        const uint32_t idesc = idesc_f16(128, IN, 1, 1);
        for (int it = 0; it < n_kb; ++it) {
          wait_bar<PROF>(&bars->xf, (uint32_t)it & 1u, pc[1]);  // the operand slot holds k-block `it`
          fence_after_sync();
          const uint32_t sa = tma::smem_u32(op);
          const uint32_t sb = sa + 2 * kWgA16;
          const uint64_t a_hi = desc_mn_sw64(sa, 2048), a_lo = desc_mn_sw64(sa + kWgA16, 2048);
          const uint64_t b_hi = desc_mn_sw64(sb, 2048), b_lo = desc_mn_sw64(sb + kWgB16, 2048);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t koff = (uint64_t)((k * 1024) >> 4);  // next 16 samples = two 8-sample atoms
            const uint32_t acc = (it > 0 || k > 0) ? 1u : 0u;
            mma_f16(tmem_base, a_lo + koff, b_hi + koff, idesc, acc);
            mma_f16(tmem_base, a_hi + koff, b_lo + koff, idesc, 1u);
            mma_f16(tmem_base, a_hi + koff, b_hi + koff, idesc, 1u);
          }
          mma_commit(&bars->op_free);
        }
        mma_commit(&bars->tmem_full);
      }
    } else if (warp < 6) {
      const int q = warp & 3;
      tma::mbar_wait(&bars->tmem_full, 0);
      fence_after_sync();
      const int row = out_tile * 128 + q * 32 + lane;
      const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16);
      float* dW = P.part + ((size_t)chunk * P.ngroups + grp) * 256 * IN;
      for (int c0 = 0; c0 < IN; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(taddr0 + c0, r);
        tmem_ld_wait();
        float* dst = dW + (size_t)row * IN + c0;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(dst + j) =
              make_float4(__uint_as_float(r[j]) * out_scale, __uint_as_float(r[j + 1]) * out_scale,
                          __uint_as_float(r[j + 2]) * out_scale, __uint_as_float(r[j + 3]) * out_scale);
      }
      fence_before_sync();
    } else {
      const int t = threadIdx.x - 6 * 32;
      for (int it = 0; it < n_kb; ++it) {
        const int s = it % kWgLand;
        const uint32_t ph = (it / kWgLand) & 1u;
        wait_bar<PROF>(&bars->full[s], ph, pc[2]);                       // the fp32 tiles have landed
        wait_bar<PROF>(&bars->op_free, ((uint32_t)it & 1u) ^ 1u, pc[3]);  // the MMAs of k-block it-1 have read the operand slot
        const long long t_w0 = PROF ? clock64() : 0;
        uint8_t* st = smem + s * kWgLandBytes;
        uint8_t* b32 = st + kWgA32;
        // groups of [32 samples x 32 floats] (4 KB) -> [32 samples x 32 halfs] (2 KB); consecutive groups are contiguous
        // on both sides, so "rows" simply runs over groups * 32
        split_tile<32 * kWgXfWarps>(st, op, op + kWgA16, 4 * 32, t, z_scale);
        split_tile<32 * kWgXfWarps>(b32, op + 2 * kWgA16, op + 2 * kWgA16 + kWgB16, (IN / 32) * 32, t, 1.0f);
        tma::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma::mbar_arrive(&bars->xf);
          tma::mbar_arrive(&bars->empty[s]);
        }
        if constexpr (PROF) pc[4] += clock64() - t_w0;
      }
    }
  }
  if constexpr (PROF) {
    if (blockIdx.x == 0 && P.prof && lane == 0 && (warp == 0 || warp == 1 || warp == 6)) {
      for (int i = 0; i < 5; ++i)
        if (pc[i]) atomicAdd(reinterpret_cast<unsigned long long*>(P.prof + 9 + i), (unsigned long long)pc[i]);
      if (warp == 0) {
        atomicAdd(reinterpret_cast<unsigned long long*>(P.prof + 14), (unsigned long long)(clock64() - t_start));
        atomicAdd(reinterpret_cast<unsigned long long*>(P.prof + 15), (unsigned long long)n_kb);
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ---- weights -> packed fp16 (hi, lo) tiles of w * 2^kWeightScaleLog2, all hidden matrices of the policy in ONE launch ----
struct SplitJob {
  const float* src;   // [256 out, K in]
  uint8_t* fwd;       // forward pack
  uint8_t* dgrad;     // dgrad pack or NULL
  int K;
};
struct SplitJobs {
  SplitJob j[8];
  int count;
};
// item = (out row o, 8 consecutive inputs): 16 bytes of hi and of lo in each pack
__global__ void __launch_bounds__(256) split_half_kernel(SplitJobs jobs) {
  const float scale = (float)(1 << kWeightScaleLog2);
  for (int q = 0; q < jobs.count; ++q) {
    const SplitJob& J = jobs.j[q];
    const int cpr = J.K / 8;  // 16-byte chunks per row
    const int64_t items = (int64_t)BN * cpr;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < items; i += stride) {
      const int o = (int)(i / cpr), c8 = (int)(i - (int64_t)o * cpr);  // inputs [8*c8, 8*c8+8)
      const float4 x0 = *reinterpret_cast<const float4*>(J.src + (size_t)o * J.K + 8 * c8);
      const float4 x1 = *reinterpret_cast<const float4*>(J.src + (size_t)o * J.K + 8 * c8 + 4);
      const float v[8] = {x0.x * scale, x0.y * scale, x0.z * scale, x0.w * scale,
                          x1.x * scale, x1.y * scale, x1.z * scale, x1.w * scale};
      uint32_t h[4], l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const __half2 hh = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
        const float2 hf = __half22float2(hh);
        const __half2 ll = __floats2half2_rn(v[2 * j] - hf.x, v[2 * j + 1] - hf.y);
        h[j] = *reinterpret_cast<const uint32_t*>(&hh);
        l[j] = *reinterpret_cast<const uint32_t*>(&ll);
      }
      {  // forward pack: k-block = 8*c8 / 32, tile row o (64 B), chunk (c8 & 3) swizzled by ((o >> 1) & 3)
        const int kb = c8 >> 2, ch = c8 & 3;
        uint8_t* d = J.fwd + (size_t)kb * (2 * kB16) + o * 64 + ((ch ^ ((o >> 1) & 3)) << 4);
        *reinterpret_cast<uint4*>(d) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(d + kB16) = make_uint4(l[0], l[1], l[2], l[3]);
      }
      if (J.dgrad != nullptr) {  // dgrad pack: k-block = o / 32, group = input / 64, row o % 32 (128 B), chunk swizzled by (row & 7)
        const int kb = o >> 5, r = o & 31, grp = c8 >> 3, ch = c8 & 7;
        uint8_t* d = J.dgrad + (size_t)kb * (2 * kB16) + grp * 4096 + r * 128 + ((ch ^ (r & 7)) << 4);
        *reinterpret_cast<uint4*>(d) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(d + kB16) = make_uint4(l[0], l[1], l[2], l[3]);
      }
    }
  }
}

// ---- host -----------------------------------------------------------------------------------------------------------
int encode_f32_sw128(CUtensorMap* out, const float* base, uint64_t rows, uint64_t cols, uint32_t box_rows);
int encode_f16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint32_t box_cols, uint32_t box_rows,
               int swizzle_bytes);

static long long* g_prof = nullptr;  // rb200_tc_h_debug

static int ctas_per_group(int ngroups, int64_t M) {
  const int64_t n_tiles = (M + BM - 1) / BM;
  int per_group = rb::sm_count() / ngroups;
  if (per_group > n_tiles) per_group = (int)n_tiles;
  return per_group < 1 ? 1 : per_group;
}

// sample chunks of the wgrad grid and k-blocks per chunk; every chunk owns at least one k-block (and writes its row)
static int wgrad_chunks(int ngroups, int64_t n, int* kb_per_chunk) {
  const int n_kb = (int)((n + BK - 1) / BK);
  int chunks = rb::sm_count() / (2 * ngroups);
  if (chunks < 1) chunks = 1;
  if (chunks > n_kb) chunks = n_kb;
  *kb_per_chunk = (n_kb + chunks - 1) / chunks;
  return (n_kb + *kb_per_chunk - 1) / *kb_per_chunk;
}

int64_t launch_part_floats(int ngroups, int64_t M) { return (int64_t)ctas_per_group(ngroups, M) * ngroups * BN; }

int64_t wgrad_part_floats(int ngroups, int64_t n, int IN) {
  int kpc = 0;
  return (int64_t)wgrad_chunks(ngroups, n, &kpc) * ngroups * 256 * IN;
}

int launch(const GemmLaunch* L, int ngroups, int64_t M, int K, int epi, int b_mn, float* part, cudaStream_t st) {
  if (ngroups < 1 || ngroups > 2 || K % BK != 0 || K <= 0 || M <= 0) return RB200_E_SHAPE;
  // Two towers in one launch: measured on B200 (profiles/r02_tc_h_gemm_grouping.txt) grouped is never slower than one
  // launch per tower (1.18 vs 1.21 ms per 6-GEMM forward at 262144 rows, 0.21 vs 0.24 ms at 32768 where it fills the
  // tail wave).
  GemmParams P{};
  P.M = M; P.K = K; P.epi = epi; P.b_mn = b_mn; P.ngroups = ngroups;
  for (int g = 0; g < ngroups; ++g) {
    const GemmLaunch& l = L[g];
    const uintptr_t al = reinterpret_cast<uintptr_t>(l.a) | reinterpret_cast<uintptr_t>(l.b_hi) |
                         reinterpret_cast<uintptr_t>(l.c) | reinterpret_cast<uintptr_t>(l.h);
    if (al & 15) return RB200_E_ALIGN;
    int e = encode_f32_sw128(&P.a[g], l.a, (uint64_t)M, (uint64_t)K, BM);
    P.wpack[g] = reinterpret_cast<const uint8_t*>(l.b_hi);
    if (!e) e = encode_f32_sw128(&P.c[g], l.c, (uint64_t)M, BN, 32);
    if (e) return RB200_E_UNSUPPORTED;
    P.g[g] = Group{l.bias, l.h, l.colsum, l.amax_in, l.amax_out};
  }
  static bool attr_done = false;
  constexpr int kSmem = kRingBytes + kStagingBytes + 1024 + (int)sizeof(Barriers);
  static_assert(kSmem <= 232448, "tc_h_gemm_kernel shared memory");
  if (!attr_done) {
    cudaError_t ce = cudaFuncSetAttribute(tc_h_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (ce == cudaSuccess)
      ce = cudaFuncSetAttribute(tc_h_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (ce != cudaSuccess) return (int)ce;
    attr_done = true;
  }
  P.prof = g_prof;
  const int per_group = ctas_per_group(ngroups, M);
  rb::PartialSeg segs[2];
  int nseg = 0;
  if (epi == rb::tc::EPI_TANHGRAD)
    for (int g = 0; g < ngroups; ++g)
      if (L[g].colsum != nullptr) segs[nseg++] = rb::PartialSeg{L[g].colsum, (int64_t)g * BN, BN};
  if (nseg > 0) {
    if (part == nullptr) return RB200_E_NULL;
    P.part = part;
  }
  if (g_prof) tc_h_gemm_kernel<true><<<per_group * ngroups, kThreads, kSmem, st>>>(P);
  else tc_h_gemm_kernel<false><<<per_group * ngroups, kThreads, kSmem, st>>>(P);
  rb::count_launch();
  cudaError_t ce = cudaPeekAtLastError();
  if (ce != cudaSuccess || nseg == 0) return (int)ce;
  return rb::sum_partials(P.part, per_group, (int64_t)ngroups * BN, segs, nseg, st);
}

int wgrad(const WgradLaunch* L, int ngroups, int64_t n, int IN, float* part, cudaStream_t st) {
  if (ngroups < 1 || ngroups > 2 || n <= 0 || IN <= 0 || IN > 256 || IN % 32 != 0) return RB200_E_SHAPE;
  WgradParams P{};
  P.n = n; P.IN = IN; P.ngroups = ngroups;
  for (int g = 0; g < ngroups; ++g) {
    const uintptr_t al = reinterpret_cast<uintptr_t>(L[g].z) | reinterpret_cast<uintptr_t>(L[g].h) |
                         reinterpret_cast<uintptr_t>(L[g].dW);
    if (al & 15) return RB200_E_ALIGN;
    int e = encode_f32_sw128(&P.z[g], L[g].z, (uint64_t)n, 256, 32);
    if (!e) e = encode_f32_sw128(&P.h[g], L[g].h, (uint64_t)n, (uint64_t)IN, 32);
    if (e) return RB200_E_UNSUPPORTED;
    P.dW[g] = L[g].dW;
    P.amax_z[g] = L[g].amax_z;
  }
  static bool attr_done = false;
  constexpr int kSmem = kWgRingBytes + 1024 + (int)sizeof(WgBarriers);
  static_assert(kSmem <= 232448, "tc_h_wgrad_kernel shared memory");
  if (!attr_done) {
    cudaError_t ce = cudaFuncSetAttribute(tc_h_wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (ce == cudaSuccess)
      ce = cudaFuncSetAttribute(tc_h_wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (ce != cudaSuccess) return (int)ce;
    attr_done = true;
  }
  if (part == nullptr) return RB200_E_NULL;
  const int chunks = wgrad_chunks(ngroups, n, &P.kb_per_chunk);
  const int64_t stride = (int64_t)ngroups * 256 * IN;
  P.part = part;
  P.prof = g_prof;
  if (g_prof) tc_h_wgrad_kernel<true><<<ngroups * 2 * chunks, kWgThreads, kSmem, st>>>(P);
  else tc_h_wgrad_kernel<false><<<ngroups * 2 * chunks, kWgThreads, kSmem, st>>>(P);
  rb::count_launch();
  cudaError_t ce = cudaPeekAtLastError();
  if (ce != cudaSuccess) return (int)ce;
  rb::PartialSeg segs[2];
  for (int g = 0; g < ngroups; ++g) segs[g] = rb::PartialSeg{L[g].dW, (int64_t)g * 256 * IN, 256ll * IN};
  return rb::sum_partials(P.part, chunks, stride, segs, ngroups, st);
}

int split_weights(const SplitSpec* specs, int count, cudaStream_t st) {
  if (count < 1 || count > 8) return RB200_E_SHAPE;
  SplitJobs jobs{};
  jobs.count = count;
  int64_t total = 0;
  for (int i = 0; i < count; ++i) {
    const int64_t K = specs[i].n / BN;
    if (K * BN != specs[i].n || K % BK != 0 || (specs[i].lo != nullptr && K != BN)) return RB200_E_SHAPE;
    jobs.j[i] = SplitJob{specs[i].src, reinterpret_cast<uint8_t*>(specs[i].hi), reinterpret_cast<uint8_t*>(specs[i].lo), (int)K};
    total = specs[i].n / 8 > total ? specs[i].n / 8 : total;
  }
  int64_t blocks = (total + 255) / 256;
  const int64_t cap = (int64_t)rb::sm_count() * 4;
  if (blocks > cap) blocks = cap;
  split_half_kernel<<<(int)blocks, 256, 0, st>>>(jobs);
  rb::count_launch();
  cudaError_t ce = cudaPeekAtLastError();
  return ce == cudaSuccess ? 0 : (int)ce;
}

}  // namespace tch
}  // namespace rb

// probe hook (tools/gemm_role_probe.py): 16 int64 receiving CTA 0's per-role wait / work cycles (forward / dgrad kernel:
// 0 producer-wait-empty, 1 mma-wait-tmem_empty, 2 mma-wait-full, 3 mma-wait-xf, 4 xf-wait-full, 5 xf-work,
// 6 epilogue-wait-tmem_full, 7 epilogue-work, 8 total); NULL restores the production kernels
extern "C" int rb200_tc_h_debug(void* prof16) {
  rb::tch::g_prof = static_cast<long long*>(prof16);
  return RB200_OK;
}

// ---- unit-test entries (tests/test_gpu_tc_gemm.py) --------------------------------------------------------------------
// C[M,256] = A[M,K] . B[256,K]^T (mode 0, forward) or A[M,256] . B[256,256] (mode 1, dgrad form: B is [out=K, in=N]);
// work: >= 256*K floats (fp16 hi/lo copies of B).  amax (device float, nullable) exercises the gradient scaling.
extern "C" int rb200_tc_gemm_h(const float* A, const float* B, float* C, int64_t M, int K, int mode, const float* amax,
                               float* work, rb200_stream_t stream) {
  if (!A || !B || !C || !work) return RB200_E_NULL;
  if (M <= 0 || K <= 0 || K % rb::tc::BK != 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  const int64_t nb = (int64_t)rb::tc::BN * K;
  if (mode && K != rb::tc::BN) return RB200_E_SHAPE;
  // forward pack always; the dgrad pack (square matrices only) behind it
  rb::tch::SplitSpec sp{B, work, mode ? work + nb : nullptr, nb};
  int e = rb::tch::split_weights(&sp, 1, st);
  if (e) return e;
  rb::tch::GemmLaunch l{};
  l.a = A; l.b_hi = mode ? sp.lo : sp.hi; l.b_lo = nullptr; l.c = C; l.amax_in = amax;
  return rb::tch::launch(&l, 1, M, K, rb::tc::EPI_STORE, mode ? 1 : 0, nullptr, st);
}

extern "C" int rb200_tc_wgrad_h(const float* Z, const float* H, float* dW, int64_t n, int IN, const float* amax,
                                rb200_stream_t stream) {
  if (!Z || !H || !dW) return RB200_E_NULL;
  if (n <= 0 || IN <= 0 || IN > 256 || IN % 32 != 0) return RB200_E_SHAPE;
  cudaStream_t st = rb::as_stream(stream);
  rb::tch::WgradLaunch l{Z, H, dW, amax};
  // the chunk partials live in a stream-ordered allocation of this call
  float* part = nullptr;
  cudaError_t ce = cudaMallocAsync(reinterpret_cast<void**>(&part), sizeof(float) * rb::tch::wgrad_part_floats(1, n, IN), st);
  if (ce != cudaSuccess) return (int)ce;
  const int e = rb::tch::wgrad(&l, 1, n, IN, part, st);
  ce = cudaFreeAsync(part, st);
  return e ? e : (int)ce;
}
