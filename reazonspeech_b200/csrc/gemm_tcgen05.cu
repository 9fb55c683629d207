// Persistent, warp-specialised bf16 GEMM for sm_100a:  out = epi(A[M,K] * W[N,K]^T)
//
//   warp 0      TMA producer   cp.async.bulk.tensor 2-D tiles (128B swizzle) -> smem ring
//   warp 1      MMA issuer     one elected lane issues tcgen05.mma (UMMA 128 x BN x 16), fp32
//                              accumulators in TMEM, two accumulator stages (2*BN columns)
//   warps 2..9  epilogue       tcgen05.ld TMEM -> registers -> bias / activation / GLU /
//                              residual -> vectorised global stores; overlaps the next tile's MMAs
//
// Covers every dense contraction of the FastConformer encoder (SURVEY.md App. A.3): FFN W1/W2,
// fused QKV, attention out-proj, conv pointwise 1/2, the subsampling 1x1 convs and out-linear,
// and the joint's encoder projection.  Replaces the cuBLAS fp32 GEMMs NeMo dispatches under
// model.transcribe (pkg/nemo-asr/src/transcribe.py:48-53).
#include <cuda.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/rs_engine.h"
#include "common.cuh"
#include "kernels.h"

namespace rs {

constexpr int BM = 128;
constexpr int BK = 64;                 // 64 bf16 = 128 B = one swizzle atom row
constexpr int UMMA_K = 16;
constexpr int kEpiWarps = 8;
constexpr int kGemmThreads = 32 * (2 + kEpiWarps);
constexpr int kABytes = BM * BK * 2;   // 16 KiB

struct GemmDev {
  const float* bias;
  const float* resid;
  void* out;
  int M, N, K;
  int epilogue;
  float alpha;
  int ldo;              // output (and residual) row stride in elements
  void* out2; int split, ld2;    // RS_EPI_QKV_VT
};
template <int BN>
struct GemmCfg {
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = BN == 128 ? 5 : 7;
  static constexpr int kTmemCols = 2 * BN;                       // power of two >= 32
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/ + kEpiWarps * (32 * 36 * 4 + 512) /*epilogue staging*/;
};

// Fused epilogue of one 32-row x 32-column chunk (one epilogue warp): bias, activation / GLU / residual, store.
// tcgen05.ld hands every lane one ROW of the chunk; storing that directly would touch 32 different cache
// lines per instruction.  The chunk is therefore transposed through a per-warp staging buffer in shared
// memory so that each global access instruction covers whole 128-byte lines (fp32: 4 rows x 128 B,
// bf16: 8 rows x 64 B), and the residual is read -- and prefetched during the MMAs -- in that same
// coalesced ownership.
constexpr int kStageLd = 36;                                   // floats per staged row (144 B: 16 B-aligned, conflict-free)
constexpr int kStageBytesPerWarp = 32 * kStageLd * 4 + 512;    // + the bias of the warp's (up to) four chunks of a tile

__device__ __forceinline__ void resid_prefetch(const GemmDev& p, bool on, int tile_row0, int lane, int col0, float4 (&rr)[8]) {
  if (on) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = tile_row0 + i * 4 + (lane >> 3);
      rr[i] = row < p.M ? *reinterpret_cast<const float4*>(p.resid + static_cast<size_t>(row) * p.ldo + col0 + (lane & 7) * 4)
                        : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

// EG: epilogue group compiled into a kernel instance -- 0: the common epilogues, 1: RS_EPI_QKV_VT.
// (One kernel with every path spilled registers in the common ones: 166 -> 168 registers + a stack frame, GEMMs 10-20 % slower.)
// kResid: the instance may be asked for RS_EPI_RESID_F32 with the residual in rr (otherwise rr is never read).
template <int EG, bool kResid>
__device__ __forceinline__ void epilogue_store(const GemmDev& p, const uint32_t (&r)[32], float* stage, int tile_row0, int lane,
                                               int col0, const float4 (&rr)[8], const float* bias_s = nullptr) {
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  if (bias_s != nullptr) {                                     // the chunk's bias from shared memory (broadcast reads; zeros without a bias)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b = *reinterpret_cast<const float4*>(bias_s + 4 * j);
      v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
    }
  } else if (p.bias != nullptr) {
    const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b = __ldg(b4 + j);
      v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
    }
  }
  uint32_t* stage_u = reinterpret_cast<uint32_t*>(stage);
  int epi = p.epilogue;
  if constexpr (EG == 1) {
    if (col0 < p.split) {
      epi = RS_EPI_BIAS_BF16;                                  // q | k columns: plain row-major bf16
    } else {
      // V columns: out2[col - split][row] = bf16(v).  Staged so that one store instruction covers 8 rows of out2
      // (= 8 head dims) x 64 B (= 32 consecutive frames).
      uint16_t* st16 = reinterpret_cast<uint16_t*>(stage);     // [32 dims][40] halves
#pragma unroll
      for (int j = 0; j < 32; ++j) st16[j * 40 + lane] = __bfloat16_as_ushort(__float2bfloat16_rn(v[j]));
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int dim = i * 8 + (lane >> 2), f0 = (lane & 3) * 8;
        const uint4 a = *reinterpret_cast<const uint4*>(st16 + dim * 40 + f0);
        if (tile_row0 + f0 < p.M)      // M is a multiple of 8 (checked at launch): frames beyond it belong to another row range of the same buffer
          *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out2) + static_cast<size_t>(col0 - p.split + dim) * p.ld2 + tile_row0 + f0) = a;
      }
      __syncwarp();
      return;
    }
  }
  switch (epi) {
    case RS_EPI_BIAS_F16: {                                    // same 16-bit store pattern as the bf16 epilogues
#pragma unroll
      for (int j = 0; j < 4; ++j)
        *reinterpret_cast<uint4*>(stage_u + lane * 20 + 4 * j) =
            make_uint4(pack_f16x2(v[8 * j], v[8 * j + 1]), pack_f16x2(v[8 * j + 2], v[8 * j + 3]),
                       pack_f16x2(v[8 * j + 4], v[8 * j + 5]), pack_f16x2(v[8 * j + 6], v[8 * j + 7]));
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rl = i * 8 + (lane >> 2), cw = (lane & 3) * 4;
        const int row = tile_row0 + rl;
        const uint4 a = *reinterpret_cast<const uint4*>(stage_u + rl * 20 + cw);
        if (row < p.M)
          *reinterpret_cast<uint4*>(static_cast<__half*>(p.out) + static_cast<size_t>(row) * p.ldo + col0 + cw * 2) = a;
      }
      break;
    }
    case RS_EPI_BIAS_BF16:
    case RS_EPI_BIAS_RELU_BF16:
    case RS_EPI_BIAS_SWISH_BF16: {
      if (epi == RS_EPI_BIAS_RELU_BF16) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
      } else if (epi == RS_EPI_BIAS_SWISH_BF16) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = swishf_fast(v[j]);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j)                              // staged row = 16 words, row stride 20 words
        *reinterpret_cast<uint4*>(stage_u + lane * 20 + 4 * j) =
            make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                       pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {                            // 8 rows x 64 B per instruction
        const int rl = i * 8 + (lane >> 2), cw = (lane & 3) * 4;
        const int row = tile_row0 + rl;
        const uint4 a = *reinterpret_cast<const uint4*>(stage_u + rl * 20 + cw);
        if (row < p.M)
          *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out) + static_cast<size_t>(row) * p.ldo + col0 + cw * 2) = a;
      }
      break;
    }
    case RS_EPI_BIAS_GLU_BF16: {
      // columns [0,16) of the chunk are values, [16,32) the matching gates (weights interleaved at pack time)
      float g[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) g[j] = v[j] * sigmoidf_fast(v[16 + j]);
#pragma unroll
      for (int j = 0; j < 2; ++j)                              // staged row = 8 words, row stride 12 words
        *reinterpret_cast<uint4*>(stage_u + lane * 12 + 4 * j) =
            make_uint4(pack_bf16x2(g[8 * j], g[8 * j + 1]), pack_bf16x2(g[8 * j + 2], g[8 * j + 3]),
                       pack_bf16x2(g[8 * j + 4], g[8 * j + 5]), pack_bf16x2(g[8 * j + 6], g[8 * j + 7]));
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 2; ++i) {                            // 16 rows x 32 B per instruction
        const int rl = i * 16 + (lane >> 1), cw = (lane & 1) * 4;
        const int row = tile_row0 + rl;
        const uint4 a = *reinterpret_cast<const uint4*>(stage_u + rl * 12 + cw);
        if (row < p.M)
          *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out) + static_cast<size_t>(row) * p.ldo + col0 / 2 + cw * 2) = a;
      }
      break;
    }
    default: {  // RS_EPI_RESID_F32 / RS_EPI_BIAS_F32
      constexpr int LD = kStageLd;
      for (int j = 0; j < 8; ++j)                              // (fully unrolled by the compiler: constant trip count)
        *reinterpret_cast<float4*>(stage + lane * LD + 4 * j) =
            make_float4(p.alpha * v[4 * j], p.alpha * v[4 * j + 1], p.alpha * v[4 * j + 2], p.alpha * v[4 * j + 3]);
      __syncwarp();
      const bool add = kResid && p.epilogue == RS_EPI_RESID_F32;
#pragma unroll
      for (int i = 0; i < 8; ++i) {                            // 4 rows x 128 B per instruction
        const int rl = i * 4 + (lane >> 3), cw = (lane & 7) * 4;
        const int row = tile_row0 + rl;
        float4 a = *reinterpret_cast<const float4*>(stage + rl * LD + cw);
        if (add) { a.x += rr[i].x; a.y += rr[i].y; a.z += rr[i].z; a.w += rr[i].w; }
        if (row < p.M)
          *reinterpret_cast<float4*>(static_cast<float*>(p.out) + static_cast<size_t>(row) * p.ldo + col0 + cw) = a;
      }
      break;
    }
  }
  __syncwarp();                                                // staging buffer reusable; reconverged for the next tcgen05.ld
}

template <int BN, int EG>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const GemmDev p) {
  using Cfg = GemmCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  // 128B-swizzled operand tiles need 1024 B alignment.
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + Cfg::kStages * Cfg::kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::kStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::kStages + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * Cfg::kStages + 4);
  uint8_t* stage_gen = smem_raw + ((bar_base + 256u) - smem_u32(smem_raw));   // generic pointer to the staging area
  auto smem_a = [&](int s) { return smem_base + s * Cfg::kStageBytes; };
  auto smem_b = [&](int s) { return smem_base + s * Cfg::kStageBytes + kABytes; };

  const int warp = warp_id_uniform();
  const int lane = lane_id();
  const int num_m = (p.M + BM - 1) / BM;
  const int num_n = (p.N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_k = p.K / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), kEpiWarps); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = (tile / num_n) * BM, n0 = (tile % num_n) * BN;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          mbar_arrive_expect_tx(full_bar(stage), Cfg::kStageBytes);
          tma_load_2d(smem_a(stage), &tm_a, kb * BK, m0, full_bar(stage));
          tma_load_2d(smem_b(stage), &tm_b, kb * BK, n0, full_bar(stage));
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM, BN);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);          // epilogue drained this accumulator
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint64_t da = umma_desc_k_sw128(smem_a(stage));
          const uint64_t db = umma_desc_k_sw128(smem_b(stage));
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            // advance 16 elements (32 B) along K inside the swizzle atom: +2 in the >>4 address field
            umma_bf16_ss(d_tmem, da + 2u * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(empty_bar(stage));                     // smem slot reusable when these MMAs retire
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1u; }
        }
        umma_commit(tfull_bar(acc));                         // accumulator complete
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps
    const int q = warp & 3;                                  // TMEM lane quarter this warp may read
    const int half = (warp - 2) >> 2;                        // which interleaved 32-column chunks
    float* stage = reinterpret_cast<float*>(stage_gen + (warp - 2) * kStageBytesPerWarp);
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1u;
      const int m0 = (tile / num_n) * BM, n0 = (tile % num_n) * BN;
      const int tile_row0 = m0 + q * 32;
      // residual of the first chunk is fetched while the tile's MMAs are still running
      const bool pre = p.epilogue == RS_EPI_RESID_F32;
      float4 rr[8], cur[8];
      resid_prefetch(p, pre && n0 + half * 32 < p.N, tile_row0, lane, n0 + half * 32, rr);
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
#pragma unroll 1
      for (int chunk = half; chunk < BN / 32; chunk += 2) {
        const int col0 = n0 + chunk * 32;
        if (col0 >= p.N) break;                              // warp-uniform
#pragma unroll
        for (int j = 0; j < 8; ++j) cur[j] = rr[j];
        resid_prefetch(p, pre && chunk + 2 < BN / 32 && col0 + 64 < p.N, tile_row0, lane, col0 + 64, rr);
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN + chunk * 32, r);
        tmem_ld_wait();
        epilogue_store<EG, true>(p, r, stage, tile_row0, lane, col0, cur);
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

// ---------------------------------------------------------------------------- 2-CTA variant
// Cluster of two CTAs (an SM pair) computes a 256 x BN tile with tcgen05.mma.cta_group::2: each CTA
// stages its own 128 rows of A and HALF of the W tile, the leader's single thread issues UMMA
// 256 x BN x 16 reading both halves.  Per CTA and k-block that is 32 KB of L2->smem traffic for the
// MACs the 1-CTA kernel feeds with 48 KB, which matters because at 128 x 256 tiles the 1-CTA kernel
// is bound by L2 bandwidth (87 FLOP/B against ~12 TB/s), not by the tensor pipe; it also leaves room
// for a 6-deep ring.  Barriers: full[] on the leader (both producers arrive, both TMAs credit it),
// empty[] / tmem_full[] per CTA (commit multicast to both), tmem_empty[] on the leader.
// EG 2 (in-place residual, out == resid): the epilogue never reads the residual.  Each warp writes alpha * (acc + bias) of
// a 32 x 32 chunk into a 128B-swizzled 4 KB buffer and one lane hands it to the TMA unit as a reduce-add
// (cp.reduce.async.bulk.tensor ... .add, fp32): the memory system performs x += tile at the destination, asynchronously.
// The register path it replaces fetched the residual 4 KB per warp at a time and was bound by that round trip
// (N = 1024, K = 1024: 39 us against a 20 us HBM floor).  Two buffers per warp, so a chunk is written while the
// previous one is still being read out.  The sum is the same fp32 add as before (each element is reduced exactly once).
constexpr int kReduceBufBytes = 32 * 32 * 4;

// Timeline of the last 2-CTA launch (SM clock of the leader CTA), first and last cluster: [0] roles start, per tile i < 3
// [1+4i] accumulator free, [2+4i] first operand stage landed, [3+4i] last MMA issued, [4+4i] accumulator complete as seen by
// the epilogue, [16+2i] that epilogue warp done with the tile, [30] kernel entry, [31] after the closing cluster sync.
__device__ long long g_gemm_prof[2][32];
template <int BN, int EG = 0>
struct Gemm2Cfg {
  static constexpr int kBHalfBytes = (BN / 2) * BK * 2;
  static constexpr int kStageBytes = kABytes + kBHalfBytes;
  static constexpr int kStages = (BN == 256) ? 5 : 7;
  static constexpr int kStagingPerWarp = EG == 2 ? 2 * kReduceBufBytes : kStageBytesPerWarp;
  static constexpr int kStagingBytes = kEpiWarps * kStagingPerWarp;      // multiple of 1024: follows the operand ring, 1024-aligned
  static constexpr int kTmemCols = 2 * BN;
  static constexpr int kSmemBytes = kStages * kStageBytes + kStagingBytes + 1024 /*align slack*/ + 256 /*barriers*/;
  static_assert(kStagingBytes % 1024 == 0 && kSmemBytes <= 227 * 1024, "shared memory layout");
};

template <int BN, int EG>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tn_2cta_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                         const __grid_constant__ CUtensorMap tm_o, const GemmDev p) {
  using Cfg = Gemm2Cfg<BN, EG>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t staging_base = smem_base + Cfg::kStages * Cfg::kStageBytes;
  const uint32_t bar_base = staging_base + Cfg::kStagingBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::kStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::kStages + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * Cfg::kStages + 4);
  uint8_t* stage_gen = smem_raw + (staging_base - smem_u32(smem_raw));        // generic pointer to the staging area
  auto smem_a = [&](int s) { return smem_base + s * Cfg::kStageBytes; };
  auto smem_b = [&](int s) { return smem_base + s * Cfg::kStageBytes + kABytes; };

  const int warp = warp_id_uniform();
  const int lane = lane_id();
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int num_m = (p.M + 2 * BM - 1) / (2 * BM);          // 256-row cluster tiles
  const int num_n = p.N / BN;
  const int num_tiles = num_m * num_n;
  const int num_k = p.K / BK;
  const int cid = static_cast<int>(cluster_id_x()), ncl = static_cast<int>(cluster_nctaid_x());
  const int prof_slot = !leader ? -1 : cid == 0 ? 0 : cid == ncl - 1 ? 1 : -1;
  // The stamps are compiled in only with -DRS_PROF (RS_BUILD_FLAGS=-DRS_PROF python -m reazonspeech_b200.build --force):
  // measured on one box, the shipped kernel is 2-3 % faster without them (12.5 vs 12.8 ms of GEMM per step, profiles/r02_ab.md).
#ifdef RS_PROF
  auto stamp = [&](int i) { if (prof_slot >= 0 && i < 32) g_gemm_prof[prof_slot][i] = clock64(); };
#else
  (void)prof_slot;
  auto stamp = [&](int) {};
#endif
  if (threadIdx.x == 0) stamp(30);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(full_bar(s), 2); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 2 * kEpiWarps); }
    fence_barrier_init();
  }
  cluster_sync_all();                                        // peer barriers exist before any remote arrive / 2-SM alloc
  // TMA producer state (lane 0 of warp 0, both CTAs).  (Issuing the first ring of loads between the two set-up barriers, to
  // hide ~0.5 us of the first operands' latency, was measured 2 % SLOWER on the same box and removed: profiles/r02_ab.md.)
  int p_tile = cid, p_kb = 0, p_stage = 0; uint32_t p_phase = 0;
  auto produce = [&]() {
    while (p_tile < num_tiles) {
      const int m0 = (p_tile / num_n) * 2 * BM + static_cast<int>(rank) * BM;
      const int n0 = (p_tile % num_n) * BN + static_cast<int>(rank) * (BN / 2);
      mbar_wait(empty_bar(p_stage), p_phase ^ 1u);
      tma_load_2d_2sm(smem_a(p_stage), &tm_a, p_kb * BK, m0, full_bar(p_stage));
      tma_load_2d_2sm(smem_b(p_stage), &tm_b, p_kb * BK, n0, full_bar(p_stage));
      if (leader) mbar_arrive_expect_tx(full_bar(p_stage), 2 * Cfg::kStageBytes);
      else mbar_arrive_remote(full_bar(p_stage), 0);
      if (++p_stage == Cfg::kStages) { p_stage = 0; p_phase ^= 1u; }
      if (++p_kb == num_k) { p_kb = 0; p_tile += ncl; }
    }
  };
  if (warp == 1) tmem_alloc_2sm<Cfg::kTmemCols>(tmem_slot);
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    if (lane == 0) produce();
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (leader && lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      stamp(0);
      for (int tile = cid; tile < num_tiles; tile += ncl, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        if (it < 3) stamp(1 + 4 * it);
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          if (kb == 0 && it < 3) stamp(2 + 4 * it);
          const uint64_t da = umma_desc_k_sw128(smem_a(stage));
          const uint64_t db = umma_desc_k_sw128(smem_b(stage));
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k)
            umma_bf16_ss_2sm(d_tmem, da + 2u * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit_2sm(empty_bar(stage));
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1u; }
        }
        umma_commit_2sm(tfull_bar(acc));
        if (it < 3) stamp(3 + 4 * it);
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ epilogue warps (both CTAs, own TMEM half)
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    float* stage = reinterpret_cast<float*>(stage_gen + (warp - 2) * Cfg::kStagingPerWarp);
    int it = 0;
    [[maybe_unused]] uint32_t nbuf = 0;
    for (int tile = cid; tile < num_tiles; tile += ncl, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1u;
      const int m0 = (tile / num_n) * 2 * BM + static_cast<int>(rank) * BM, n0 = (tile % num_n) * BN;
      const int tile_row0 = m0 + q * 32;
      if constexpr (EG == 2) {
        mbar_wait(tfull_bar(acc), acc_phase);
        tcgen05_fence_after();
        if (warp == 2 && lane == 0 && it < 3) stamp(4 + 4 * it);
#pragma unroll 1
        for (int chunk = half; chunk < BN / 32; chunk += 2, nbuf ^= 1u) {
          const int col0 = n0 + chunk * 32;
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN + chunk * 32, r);
          if (lane == 0) bulk_wait_group_read<1>();             // the buffer written two chunks ago has been read out
          __syncwarp();
          tmem_ld_wait();
          uint8_t* buf = reinterpret_cast<uint8_t*>(stage) + nbuf * kReduceBufBytes + lane * 128;
          const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
          for (int j = 0; j < 8; ++j) {                          // lane = row; 16-byte chunk j of the row sits at j ^ (row & 7)
            const float4 b = p.bias != nullptr ? __ldg(b4 + j) : make_float4(0.f, 0.f, 0.f, 0.f);   // (a register prefetch of the next chunk's bias measured slower)
            *reinterpret_cast<float4*>(buf + ((j ^ (lane & 7)) << 4)) =
                make_float4(p.alpha * (__uint_as_float(r[4 * j]) + b.x), p.alpha * (__uint_as_float(r[4 * j + 1]) + b.y),
                            p.alpha * (__uint_as_float(r[4 * j + 2]) + b.z), p.alpha * (__uint_as_float(r[4 * j + 3]) + b.w));
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_reduce_add_2d(&tm_o, smem_u32(stage) + nbuf * kReduceBufBytes, col0, tile_row0);
            bulk_commit_group();
          }
        }
      } else {
        [[maybe_unused]] float4 rr[8], cur[8];                                // EG 3 only: the residual, one chunk ahead
        if constexpr (EG == 3) resid_prefetch(p, true, tile_row0, lane, n0 + half * 32, rr);       // overlaps the tile's MMAs
        // the bias of the warp's four chunks -> its shared slot while the MMAs run, read back as broadcasts: with the loads inside
        // the chunk loop every chunk began with an L1 / L2 round trip (same box, three alternating runs: all GEMMs 12.12 ->
        // 11.94 ms per step, N = 4096 3.79 -> 3.62 ms; profiles/r02_ab.md)
        float* bias_s = stage + 32 * kStageLd;
#pragma unroll
        for (int c = 0; c < BN / 64; ++c) bias_s[c * 32 + lane] = p.bias != nullptr ? __ldg(p.bias + n0 + (half + 2 * c) * 32 + lane) : 0.f;
        __syncwarp();
        mbar_wait(tfull_bar(acc), acc_phase);
        tcgen05_fence_after();
        if (warp == 2 && lane == 0 && it < 3) stamp(4 + 4 * it);
        const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN + half * 32;
#pragma unroll 1
        for (int chunk = half; chunk < BN / 32; chunk += 2) {
          const int col0 = n0 + chunk * 32;
          if constexpr (EG == 3) {
#pragma unroll
            for (int j = 0; j < 8; ++j) cur[j] = rr[j];
            resid_prefetch(p, chunk + 2 < BN / 32, tile_row0, lane, col0 + 64, rr);
          }
          uint32_t r[32];
          tmem_ld_32x32(t_addr + (chunk - half) * 32, r);
          tmem_ld_wait();
          epilogue_store<EG, EG == 3>(p, r, stage, tile_row0, lane, col0, cur, bias_s + (chunk >> 1) * 32);
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(tempty_bar(acc));
        else mbar_arrive_remote(tempty_bar(acc), 0);
      }
      if (warp == 2 && lane == 0 && it < 3) stamp(16 + 2 * it);
    }
    if constexpr (EG == 2) {
      if (lane == 0) bulk_wait_group_read<0>();                  // shared memory stays valid until the last tile has been read out
      __syncwarp();
    }
  }
  tcgen05_fence_before();
  cluster_sync_all();                                        // both CTAs done with TMEM and with each other's barriers
  if (threadIdx.x == 0) stamp(31);
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_2sm<Cfg::kTmemCols>(tmem_base);
  }
}

// ---------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 row-major [rows, cols] -> 2-D map with a (box_rows x 64) box and 128B swizzle.
bool make_tmap_bf16(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, char* err) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) { snprintf(err, 256, "cuTensorMapEncodeTiled entry point unavailable"); return false; }
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { snprintf(err, 256, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu", (int)r, (unsigned long long)rows, (unsigned long long)cols); return false; }
  return true;
}

// fp32 row-major [rows, cols] -> 2-D map with a 32 x 32 box and 128B swizzle (one epilogue chunk; rows beyond `rows` are clipped).
static bool make_tmap_f32_chunk(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, char* err) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) { snprintf(err, 256, "cuTensorMapEncodeTiled entry point unavailable"); return false; }
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { snprintf(err, 256, "cuTensorMapEncodeTiled(f32) failed (%d) rows=%llu cols=%llu", (int)r, (unsigned long long)rows, (unsigned long long)cols); return false; }
  return true;
}

cudaError_t gemm_debug_cycles(long long* out64) { return cudaMemcpyFromSymbol(out64, g_gemm_prof, sizeof(long long) * 64); }

inline int epilogue_group(int epilogue) { return epilogue == RS_EPI_QKV_VT ? 1 : 0; }
// output (and residual) row stride: GLU writes one column per value / gate pair
inline int out_ld(const GemmArgs& g) { return g.epilogue == RS_EPI_BIAS_GLU_BF16 ? g.N / 2 : g.N; }

template <int BN, int EG>
static cudaError_t launch_bn_eg(const GemmArgs& g, int num_sms, cudaStream_t stream, char* err) {
  using Cfg = GemmCfg<BN>;
  static DeviceOnce attr_once;
  if (attr_once.pending()) {
    cudaError_t e = cudaFuncSetAttribute(gemm_bf16_tn_kernel<BN, EG>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) { snprintf(err, 256, "cudaFuncSetAttribute(smem=%d): %s", Cfg::kSmemBytes, cudaGetErrorString(e)); return e; }
    attr_once.set();
  }
  CUtensorMap tm_a, tm_b;
  if (!make_tmap_bf16(&tm_a, g.a, g.M, g.K, g.K, BM, err)) return cudaErrorInvalidValue;
  if (!make_tmap_bf16(&tm_b, g.w, g.N, g.K, g.K, BN, err)) return cudaErrorInvalidValue;
  const GemmDev p{g.bias, g.resid, g.out, g.M, g.N, g.K, g.epilogue, g.alpha, out_ld(g), g.out2, g.split, g.ld2};
  const int tiles = ((g.M + BM - 1) / BM) * ((g.N + BN - 1) / BN);
  const int grid = tiles < num_sms ? tiles : num_sms;
  gemm_bf16_tn_kernel<BN, EG><<<grid, kGemmThreads, Cfg::kSmemBytes, stream>>>(tm_a, tm_b, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) snprintf(err, 256, "gemm launch (M=%d N=%d K=%d BN=%d): %s", g.M, g.N, g.K, BN, cudaGetErrorString(e));
  return e;
}

template <int BN>
static cudaError_t launch_bn(const GemmArgs& g, int num_sms, cudaStream_t stream, char* err) {
  switch (epilogue_group(g.epilogue)) {
    case 1: return launch_bn_eg<BN, 1>(g, num_sms, stream, err);
    default: return launch_bn_eg<BN, 0>(g, num_sms, stream, err);
  }
}

template <int BN, int EG>
static cudaError_t launch_2cta_eg(const GemmArgs& g, int num_sms, cudaStream_t stream, char* err) {
  using Cfg = Gemm2Cfg<BN, EG>;
  static DeviceOnce attr_once;
  if (attr_once.pending()) {
    cudaError_t e = cudaFuncSetAttribute(gemm_bf16_tn_2cta_kernel<BN, EG>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) { snprintf(err, 256, "cudaFuncSetAttribute(2cta smem=%d): %s", Cfg::kSmemBytes, cudaGetErrorString(e)); return e; }
    attr_once.set();
  }
  CUtensorMap tm_a, tm_b, tm_o;
  if (!make_tmap_bf16(&tm_a, g.a, g.M, g.K, g.K, BM, err)) return cudaErrorInvalidValue;
  if (!make_tmap_bf16(&tm_b, g.w, g.N, g.K, g.K, BN / 2, err)) return cudaErrorInvalidValue;
  if (EG == 2) { if (!make_tmap_f32_chunk(&tm_o, g.out, g.M, g.N, out_ld(g), err)) return cudaErrorInvalidValue; }
  else memset(&tm_o, 0, sizeof(tm_o));
  const GemmDev p{g.bias, g.resid, g.out, g.M, g.N, g.K, g.epilogue, g.alpha, out_ld(g), g.out2, g.split, g.ld2};
  const int tiles = ((g.M + 2 * BM - 1) / (2 * BM)) * (g.N / BN);
  int clusters = num_sms / 2;
  if (tiles < clusters) clusters = tiles;
  gemm_bf16_tn_2cta_kernel<BN, EG><<<2 * clusters, kGemmThreads, Cfg::kSmemBytes, stream>>>(tm_a, tm_b, tm_o, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) snprintf(err, 256, "gemm 2cta launch (M=%d N=%d K=%d BN=%d): %s", g.M, g.N, g.K, BN, cudaGetErrorString(e));
  return e;
}

template <int BN>
static cudaError_t launch_2cta(const GemmArgs& g, int num_sms, cudaStream_t stream, char* err) {
  // residual added in place: handed to the memory system as a TMA reduce-add (see Gemm2Cfg)
  if (g.epilogue == RS_EPI_RESID_F32 && g.resid == g.out) return launch_2cta_eg<BN, 2>(g, num_sms, stream, err);
  if (g.epilogue == RS_EPI_RESID_F32) return launch_2cta_eg<BN, 3>(g, num_sms, stream, err);   // residual from another buffer: read into registers
  switch (epilogue_group(g.epilogue)) {
    case 1: return launch_2cta_eg<BN, 1>(g, num_sms, stream, err);
    default: return launch_2cta_eg<BN, 0>(g, num_sms, stream, err);
  }
}

cudaError_t launch_gemm(const GemmArgs& g, int num_sms, cudaStream_t stream, char* err) {
  if (g.M <= 0 || g.N <= 0 || g.K <= 0 || g.K % BK != 0 || g.N % 32 != 0) {
    snprintf(err, 256, "gemm shape unsupported: M=%d N=%d K=%d (need K%%64==0, N%%32==0)", g.M, g.N, g.K);
    return cudaErrorInvalidValue;
  }
  if ((reinterpret_cast<uintptr_t>(g.a) | reinterpret_cast<uintptr_t>(g.w) | reinterpret_cast<uintptr_t>(g.out)) & 15u) {
    snprintf(err, 256, "gemm operands must be 16-byte aligned");
    return cudaErrorInvalidValue;
  }
  if (g.epilogue == RS_EPI_RESID_F32 && g.resid == nullptr) { snprintf(err, 256, "gemm: residual epilogue without resid"); return cudaErrorInvalidValue; }
  if (g.epilogue == RS_EPI_QKV_VT && (g.out2 == nullptr || g.split % 32 || g.ld2 % 8 || g.M % 8 || g.ld2 < g.M)) {
    snprintf(err, 256, "gemm: RS_EPI_QKV_VT needs out2, split %% 32 == 0, ld2 %% 8 == 0, M %% 8 == 0, ld2 >= M");
    return cudaErrorInvalidValue;
  }
  // kernel choice depends on N only (never on M): a row's result must not depend on the batch it sits in
  if (g.N % 256 == 0) return launch_2cta<256>(g, num_sms, stream, err);   // 2-CTA pairs (cta_group::2), 256 x 256 tiles
  // 1-CTA kernel for N not divisible by 256: the widest tile that divides N
  if (g.N % 128 == 0) return launch_bn<128>(g, num_sms, stream, err);
  return launch_bn<64>(g, num_sms, stream, err);
}

}  // namespace rs
