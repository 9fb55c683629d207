// Windowed ("blank-run speculative") batched RNN-T greedy decode: NeMo GreedyRNNTInfer._greedy_decode, RNNTDecoder.predict
// and RNNTJoint.joint (the reference reaches them at pkg/nemo-asr/src/transcribe.py:48-53) as ONE persistent cooperative
// kernel, organised around two facts about greedy transducer decoding:
//
//  1. A blank leaves the prediction-network state untouched, so the joint of the NEXT frames can be
//     evaluated against the same state before the current decision is known.  Every iteration scores a
//     window of kFrames consecutive frames per utterance; the utterance then consumes the window up to and
//     including its first non-blank frame (all-blank window: kFrames frames in one iteration).  The decision
//     sequence is exactly the sequential one; the number of lock-step iterations drops from max(T + U) to
//     about max(U + (T - U)/kFrames).
//  2. With kFrames x B rows per iteration the joint is a real (small) GEMM.  The CTAs form a 2-D grid,
//     kGroups utterance groups x S vocabulary slices: a CTA keeps its ~82 rows of W_out in shared memory
//     for the whole decode and multiplies them with the relu(enc_proj + pred_proj) rows of its group
//     (32 rows per pass) on tcgen05 (see the kernel's comment).  Activations keep 22 mantissa bits: every fp32 value is
//     split into two IEEE-half terms (hi + lo), the bf16 weights are exact in half, accumulation is fp32.
//     The LSTM step and joint.pred of the utterances that emitted are the same kind of GEMM (rows =
//     utterances, K split over the warps, A fragments loaded straight from L2) on mma.sync m16n8k16.
//  3. The input half of the LSTM gates depends on the emitted token only: W_ih . embed[k] + b_ih + b_hh is a table
//     [V+1, 4*Hp] built once at load time (pred.gate_tab), so a step multiplies just the recurrent half W_hh . h -- half the
//     shared memory, half the MMAs, and half of what every CTA pulls through L2 per step (all 148 CTAs read every
//     emitting utterance's full input vector: that traffic, not the arithmetic, is what the phase costs).
//
//   phase J  kGroups x S CTAs: window logits of the CTA's vocabulary slice -> per (utterance, frame) a grid-wide
//            64-bit red.max of (ordered logit bits | ~row)
//   barrier  -> every CTA reads the window's tokens, advances (t, symbols), emits
//   phase L  utterances that emitted: LSTM gates of the CTA's units -> new h slice
//   barrier
//   phase P  utterances that emitted: pred_proj rows of the CTA from the new h
//   barrier
#include "common.cuh"
#include "kernels.h"

namespace rs {

constexpr int kSpThreads = 256;
constexpr int kSpWarps = kSpThreads / 32;
constexpr int kFrames = 4;                       // frames scored per utterance and iteration
constexpr int kGroups = 4;                       // utterance groups (utterance b belongs to group b % kGroups)
constexpr int kPassRows = 32;                    // (utterance, frame) rows per pass: two m16 tiles
constexpr int kPassUtts = kPassRows / kFrames;

struct SpecDev {
  const float* enc_proj; const int32_t* enc_len;
  const __nv_bfloat16* w_out; const float* b_out; const float* embed;
  const __nv_bfloat16* w_lstm; const float* gate_tab; const __nv_bfloat16* w_pred; const float* b_pred;
  int32_t* tokens; int32_t* frames; int32_t* n_tok;
  unsigned long long* best;   // [3][B][kFrames] packed (ordered logit bits << 32 | ~row), 3-deep ring
  float* hbuf;                // [2][B][Hp]
  float* ppbuf;               // [B][Hj]
  unsigned int* counter;      // grid barrier: kBarCounters arrival counters, one per 128-byte line
  long long* prof;            // [12] cycle counters of CTA 0
  int B, T_max, V, U_max, max_symbols;
  int S, rows_j, units, rows_p;
};

// Grid barrier over kBarCounters arrival counters, each in its own 128-byte line: CTA i arrives on counter i % kBarCounters,
// threads 0..kBarCounters-1 each poll one counter.  All 148 arrivals on ONE address are serialised by the L2 slice that
// owns it (the barrier then costs ~1.5 us, three times per decode iteration); spread over several lines they proceed in
// parallel.  `round` counts the barriers passed; counter c has seen round * (number of CTAs with i % kBarCounters == c) arrivals.
constexpr int kBarCounters = 8;
constexpr int kBarStride = 32;            // unsigned ints between counters
__device__ __forceinline__ void sp_grid_barrier(unsigned int* counters, unsigned int& round, unsigned int nblocks) {
  __syncthreads();
  ++round;
  if (threadIdx.x == 0)     // release at gpu scope: covers the other threads' writes too (they reached thread 0 through the CTA barrier above)
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counters + (blockIdx.x % kBarCounters) * kBarStride) : "memory");
  if (threadIdx.x < kBarCounters) {
    const unsigned int c = threadIdx.x;
    const unsigned int arrivals = (nblocks + kBarCounters - 1 - c) / kBarCounters;      // CTAs with index % kBarCounters == c
    const unsigned int target = round * arrivals;
    unsigned int v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counters + c * kBarStride) : "memory");
    } while (v < target);
  }
  __syncthreads();
}

__device__ __forceinline__ void mma_f16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// fp32 pair -> two IEEE-half pairs with hi + lo == x to 22 mantissa bits (11 + 11): the residual x - hi is exact in
// fp32 and is itself rounded to half.  The legacy tensor path issues one m16n8k16 per ~19 cycles and scheduler on
// sm_100, so the number of terms is what the joint costs; three bf16 terms (24 bits) were 1.5x slower.
// Magnitudes are clamped to the largest finite half before each conversion, which extends the exactly covered
// range to |x| <= 2 * 65504; a transducer joint / LSTM input beyond that is outside what NeMo itself runs in fp16 AMP.
__device__ __forceinline__ void split2(float2 x, uint32_t& hi, uint32_t& lo) {
  constexpr float kMax = 65504.f;
  const __half2 h = __floats2half2_rn(fminf(fmaxf(x.x, -kMax), kMax), fminf(fmaxf(x.y, -kMax), kMax));
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(fminf(fmaxf(x.x - hf.x, -kMax), kMax), fminf(fmaxf(x.y - hf.y, -kMax), kMax));
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// bf16 weight pair -> half pair.  Exact for 2^-14 <= |w| < 65504 (bf16 carries 8 mantissa bits, half 11); smaller
// magnitudes become half subnormals (absolute error < 2^-25), which is below the fp32 summation noise of a logit.
__device__ __forceinline__ uint32_t bf16x2_to_f16x2(uint32_t v) { return pack_f16x2(bf16_lo(v), bf16_hi(v)); }
__device__ __forceinline__ uint4 bf16x8_to_f16x8(uint4 v) {
  return make_uint4(bf16x2_to_f16x2(v.x), bf16x2_to_f16x2(v.y), bf16x2_to_f16x2(v.z), bf16x2_to_f16x2(v.w));
}

__device__ __forceinline__ float2 ldcg2(const float* p) { return __ldcg(reinterpret_cast<const float2*>(p)); }
__device__ __forceinline__ float4 ldcg4s(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

// The joint window runs on tcgen05.  A = the CTA's W_out rows as IEEE half in
// 128B-swizzled K-major slabs of 64 columns (88 rows stored per slab; the M = 128 instruction reads on into the next slab /
// region, whose rows land in accumulator lanes nobody looks at), B = the 32 (utterance, frame) activation rows as two half
// planes (hi, lo) staged one k-half at a time, D = [128 vocabulary rows x (32 hi | 32 lo)] fp32 in tensor memory.  40 UMMAs
// of 128x64x16 per pass replace 1760 mma.sync per CTA, which were issue-bound on the legacy path (~19 cycles each).
// The hi and lo planes of the activations sit side by side as ONE B tile of 64 rows (rows 0-31 hi, 32-63 lo), so a k16 step
// is one 128x64x16 UMMA and the two halves of D are added in the epilogue: small-N UMMAs cost about the same per
// instruction as wider ones, so 80 instructions of N=32 took twice as long as 40 of N=64.
constexpr uint32_t kIdescF16_128x64 = (1u << 4) | ((64u >> 3) << 17) | ((128u >> 4) << 24);   // D=f32, A=B=f16, K-major

__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  umma_bf16_ss(tmem_d, desc_a, desc_b, idesc, accumulate);      // same instruction (kind::f16); the operand formats live in idesc
}

template <int HJ, int HP>
__global__ void __launch_bounds__(kSpThreads, 1)
rnnt_greedy_spec_kernel(const SpecDev p) {
  constexpr int KH = HJ / 2;                 // joint k-half staged in shared memory at a time
  constexpr int LS = HP + 8;                 // W_hh row stride in halves
  constexpr int KS_H = KH / 16;              // k16 steps per joint half
  constexpr int KSW_L = (HP / 16) / kSpWarps;       // k16 steps per warp, LSTM (recurrent half only)
  constexpr int KSW_P = (HP / 16) / kSpWarps;       // k16 steps per warp, joint.pred
  constexpr int V4_ROW = KH / 4;             // float4 per staged row
  constexpr int ITEMS = kPassUtts * V4_ROW;  // loader items per k-half: (utterance, float4 column)
  constexpr int PERU = (ITEMS + kSpThreads - 1) / kSpThreads;
  static_assert(HJ % 32 == 0 && (HP / 16) % kSpWarps == 0, "shape");

  extern __shared__ __align__(16) uint8_t ssm[];
  const int G = gridDim.x, cta = blockIdx.x;
  const int NC = p.V + 1, blank = p.V, B = p.B;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gid = lane >> 2, tig = lane & 3;

  // ---- slices owned by this CTA
  const int grp = cta / p.S, slice = cta % p.S;
  const bool has_j = grp < kGroups;
  const int j0 = min(NC, slice * p.rows_j), j1 = min(NC, j0 + p.rows_j);
  const int nj = has_j ? j1 - j0 : 0;
  const int u0 = min(HP, cta * p.units), u1 = min(HP, u0 + p.units);
  const int nu = u1 - u0;
  const int p0 = min(HJ, cta * p.rows_p), p1 = min(HJ, p0 + p.rows_p);
  const int np = p1 - p0;

  // ---- shared memory carve-up.  B fragments of a partial last n8-tile read past the end of a weight array
  // into the next one; those columns are masked, and every array is followed by at least 8 more rows of bytes.
  constexpr int KSLABS = HJ / 64;                                  // 64-column slabs of A
  constexpr int NSLAB_H = KH / 64;                                 // slabs per staged k-half
  const int rows_a8 = (p.rows_j + 7) & ~7;
  const uint32_t a_slab = static_cast<uint32_t>(rows_a8) * 128u;   // bytes per A slab
  constexpr uint32_t kBSlab = 8192u;                               // B slab: 64 rows x 128 B = hi plane (rows 0-31) | lo plane (rows 32-63)
  constexpr uint32_t kBRegion = (NSLAB_H * kBSlab > 24576u) ? NSLAB_H * kBSlab : 24576u;   // >= what an M = 128 read of the last A slab overruns, and the LSTM reduction buffer
  // Order: [A slabs | W_lstm | W_pred | pad to 1024 | B slabs (also the L / P reduction buffer) | bias, state ...].  The mma.sync B fragments of the LSTM /
  // joint.pred phases read up to 8 rows past the end of their (5- or 20-row) arrays: those reads must land inside the
  // allocation, so the big B region follows the weight arrays (a 2-utterance batch otherwise read past the end of shared memory).
  const uint32_t wlp_bytes = static_cast<uint32_t>((static_cast<size_t>(4 * p.units) * LS + static_cast<size_t>(p.rows_p) * (HP + 8)) * 2);   // LS = HP + 8
  const uint32_t tc_base = (smem_u32(ssm) + 1023u) & ~1023u;
  const uint32_t b_off = (KSLABS * a_slab + wlp_bytes + 1023u) & ~1023u;
  uint8_t* gA = ssm + (tc_base - smem_u32(ssm));                   // generic pointers to the A slabs / B slabs
  uint8_t* gB = gA + b_off;
  __nv_bfloat16* s_wlstm = reinterpret_cast<__nv_bfloat16*>(gA + KSLABS * a_slab);    // [4*units][LS] gate-major
  __nv_bfloat16* s_wpred = s_wlstm + static_cast<size_t>(4 * p.units) * LS;           // [rows_p][HP + 8]
  float* s_g = reinterpret_cast<float*>(gB);                                          // B planes; also the L / P reduction buffer
  float* s_bout = reinterpret_cast<float*>(gB + kBRegion);                            // -inf beyond nj
  constexpr int n_bout = 128;
  float* s_c = s_bout + n_bout;                                                      // [B][units]
  unsigned long long* s_best = reinterpret_cast<unsigned long long*>(s_c + ((static_cast<size_t>(B) * p.units + 1) & ~static_cast<size_t>(1)));   // [32][4]
  int* s_t = reinterpret_cast<int*>(s_best + kPassRows * 4);
  int* s_sym = s_t + B; int* s_n = s_sym + B; int* s_par = s_n + B; int* s_tok = s_par + B;
  int* s_emit = s_tok + B; int* s_len = s_emit + B;
  int* s_act = s_len + B;                                                            // ordered list of the utterances with frames left
  int* s_cnt = s_act + B;                                                            // [0] n_emit, [1] n_active, [2..2+8) warp counts x2
  // one mbarrier (MMA completion) + the tensor-memory slot, 8-byte aligned after s_cnt
  const uint32_t tc_bar = (smem_u32(s_cnt + 2 + 2 * kSpWarps) + 7u) & ~7u;
  const uint32_t tc_slot = tc_bar + 8;

  {
    const uint32_t zero = 0;
    // W_out slice (rows beyond nj zero-filled)
    {
      for (int i = tid; i < rows_a8 * (HJ / 8); i += kSpThreads) {
        const int r = i / (HJ / 8), c = i % (HJ / 8);          // c: 16-byte chunk (8 columns) of the row
        uint4 v = make_uint4(zero, zero, zero, zero);
        if (r < nj) v = bf16x8_to_f16x8(reinterpret_cast<const uint4*>(p.w_out + static_cast<size_t>(j0 + r) * HJ)[c]);
        *reinterpret_cast<uint4*>(gA + (c >> 3) * a_slab + (r >> 3) * 1024 + (r & 7) * 128 + (((c & 7) ^ (r & 7)) << 4)) = v;
      }
      if (tid == 0) { mbar_init(tc_bar, 1); fence_barrier_init(); }
    }
    for (int i = tid; i < 4 * p.units * (HP / 8); i += kSpThreads) {      // the W_hh half of [W_ih | W_hh]
      const int r = i / (HP / 8), c = i % (HP / 8);
      const int gate = r / p.units, u = r % p.units;
      uint4 v = make_uint4(zero, zero, zero, zero);
      if (u < nu) v = bf16x8_to_f16x8(reinterpret_cast<const uint4*>(p.w_lstm + (static_cast<size_t>(gate) * HP + u0 + u) * 2 * HP + HP)[c]);
      *reinterpret_cast<uint4*>(s_wlstm + static_cast<size_t>(r) * LS + c * 8) = v;
    }
    for (int i = tid; i < p.rows_p * (HP / 8); i += kSpThreads) {
      const int r = i / (HP / 8), c = i % (HP / 8);
      uint4 v = make_uint4(zero, zero, zero, zero);
      if (r < np) v = bf16x8_to_f16x8(reinterpret_cast<const uint4*>(p.w_pred + static_cast<size_t>(p0 + r) * HP)[c]);
      *reinterpret_cast<uint4*>(s_wpred + static_cast<size_t>(r) * (HP + 8) + c * 8) = v;
    }
    for (int i = tid; i < n_bout; i += kSpThreads) s_bout[i] = i < nj ? p.b_out[j0 + i] : -INFINITY;
    for (int i = tid; i < B * p.units; i += kSpThreads) s_c[i] = 0.f;
    for (int b = tid; b < B; b += kSpThreads) {
      s_t[b] = 0; s_sym[b] = 0; s_n[b] = 0; s_par[b] = 0; s_tok[b] = blank; s_emit[b] = b; s_len[b] = p.enc_len[b];
    }
    if (tid == 0) { s_cnt[0] = B; s_cnt[1] = 0; }
  }
  uint32_t tmem_d = 0, mma_phase = 0;
  if (warp == 0) tmem_alloc<64>(tc_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_d) : "r"(tc_slot));

  unsigned int target = 0;
  int iter = 0;
  long long prof[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  // per-phase cycle counters of CTA 0 (rs_debug_decode_cycles).  They stay in the shipped kernel: on the same box, three alternating
  // runs each, the kernel compiled WITH them decodes the bench batch in 5.30-5.35 ms and the one without in 5.62-5.70 ms (238 against
  // 231 registers: the counters change the schedule ptxas picks, not the work; profiles/r02_ab.md).  -DRS_NO_DECODE_COUNTERS drops them.
#ifndef RS_NO_DECODE_COUNTERS
  auto tick = [&](int slot, long long& t0) { if (cta == 0 && tid == 0) { const long long t1 = clock64(); prof[slot] += t1 - t0; t0 = t1; } };
  long long tk = clock64();
#else
  auto tick = [&](int, long long&) {};
  long long tk = 0;
#endif

  // ------------------------------------------------------------------------------------------------
  // LSTM step + joint.pred for the utterances listed in s_emit[0..n_emit): token s_tok[b], state parity s_par[b]
  // ------------------------------------------------------------------------------------------------
  auto lstm_and_pred = [&]() {
    const int n_emit = s_cnt[0];
    float* red = s_g;                                  // [warps][32][24]: 24 KB of the B-plane region
    // ---- phase L: gates[utterance][4*units] = gate_tab[token] + h . W_hh[slice]^T, K split over the warps.  Both 16-row
    // tiles of a step (up to 32 emitting utterances) are loaded before the first MMA: one L2 round trip, one reduction.
    if (nu > 0) {
      const int kw = (warp + cta) % kSpWarps;          // which k-range this warp takes (rotated per CTA against L2 hot-spotting)
      for (int m0 = 0; m0 < n_emit; m0 += 32) {
        const bool two = m0 + 16 < n_emit;             // block-uniform
        float2 x[2][KSW_L][4];                         // [tile][k-step][row a lo, row b lo, row a hi, row b hi]
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          if (mt == 1 && !two) break;
          const int ea = m0 + 16 * mt + gid, eb = ea + 8;
          const bool va = ea < n_emit, vb = eb < n_emit;
          const int ba = va ? s_emit[ea] : 0, bb = vb ? s_emit[eb] : 0;
          const float* h_a = p.hbuf + (static_cast<size_t>(s_par[ba]) * B + ba) * HP;
          const float* h_b = p.hbuf + (static_cast<size_t>(s_par[bb]) * B + bb) * HP;
#pragma unroll
          for (int i = 0; i < KSW_L; ++i) {
            const int off = (kw * KSW_L + i) * 16 + tig * 2;
            x[mt][i][0] = va ? ldcg2(h_a + off) : make_float2(0.f, 0.f); x[mt][i][2] = va ? ldcg2(h_a + off + 8) : make_float2(0.f, 0.f);
            x[mt][i][1] = vb ? ldcg2(h_b + off) : make_float2(0.f, 0.f); x[mt][i][3] = vb ? ldcg2(h_b + off + 8) : make_float2(0.f, 0.f);
          }
        }
        // the table row of this thread's (utterance, unit) -- the reducer threads below -- is requested now as well
        float tab[4] = {0.f, 0.f, 0.f, 0.f};
        const int el_r = tid / nu, u_r = tid % nu, e_r = m0 + el_r;
        const bool red_on = tid < 32 * nu && e_r < n_emit;
        int b_r = 0;
        if (red_on) {
          b_r = s_emit[e_r];
          const float* tr = p.gate_tab + static_cast<size_t>(s_tok[b_r]) * 4 * HP + u0 + u_r;
#pragma unroll
          for (int gate = 0; gate < 4; ++gate) tab[gate] = __ldg(tr + gate * HP);
        }
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          if (mt == 1 && !two) break;
          float acc[3][4];
#pragma unroll
          for (int n = 0; n < 3; ++n) { acc[n][0] = acc[n][1] = acc[n][2] = acc[n][3] = 0.f; }
#pragma unroll
          for (int i = 0; i < KSW_L; ++i) {
            const int ks = kw * KSW_L + i;
            uint32_t ah[4], al[4];
            split2(x[mt][i][0], ah[0], al[0]); split2(x[mt][i][1], ah[1], al[1]);
            split2(x[mt][i][2], ah[2], al[2]); split2(x[mt][i][3], ah[3], al[3]);
#pragma unroll
            for (int n = 0; n < 3; ++n) {
              if (n * 8 < 4 * p.units) {                 // warp-uniform
                // rows beyond the CTA's 4 * units gate rows feed accumulator columns nobody reads: clamped so the fragment load stays
                // inside the array (it used to run on into the reduction buffer, which compute-sanitizer racecheck rightly flags)
                const __nv_bfloat16* wr = s_wlstm + static_cast<size_t>(min(n * 8 + gid, 4 * p.units - 1)) * LS + ks * 16 + tig * 2;
                const uint32_t b0 = *reinterpret_cast<const uint32_t*>(wr), b1 = *reinterpret_cast<const uint32_t*>(wr + 8);
                mma_f16_16816(acc[n], ah, b0, b1); mma_f16_16816(acc[n], al, b0, b1);
              }
            }
          }
#pragma unroll
          for (int n = 0; n < 3; ++n) {                  // red: [warps][32 utterances][24]
            float* r0 = red + ((warp * 32 + 16 * mt + gid) * 24) + n * 8 + tig * 2;
            r0[0] = acc[n][0]; r0[1] = acc[n][1]; r0[8 * 24] = acc[n][2]; r0[8 * 24 + 1] = acc[n][3];
          }
        }
        __syncthreads();
        if (red_on) {
          const int unit = u0 + u_r;
          float gsum[4];
#pragma unroll
          for (int gate = 0; gate < 4; ++gate) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kSpWarps; ++w) s += red[(w * 32 + el_r) * 24 + gate * p.units + u_r];
            gsum[gate] = s + tab[gate];
          }
          const float ig = sigmoidf_accurate(gsum[0]), fg = sigmoidf_accurate(gsum[1]);
          const float cg = tanhf(gsum[2]), og = sigmoidf_accurate(gsum[3]);
          const float c2 = fg * s_c[b_r * p.units + u_r] + ig * cg;
          s_c[b_r * p.units + u_r] = c2;
          __stcg(p.hbuf + (static_cast<size_t>(s_par[b_r] ^ 1) * B + b_r) * HP + unit, og * tanhf(c2));
        }
        __syncthreads();
      }
    }
    tick(3, tk);
    sp_grid_barrier(p.counter, target, G);
    tick(4, tk);
    // ---- phase P (state parity flips for the utterances that stepped)
    for (int e = tid; e < n_emit; e += kSpThreads) s_par[s_emit[e]] ^= 1;
    __syncthreads();
    if (np > 0) {
      const int kw = (warp + cta) % kSpWarps;
      for (int m0 = 0; m0 < n_emit; m0 += 32) {
        const bool two = m0 + 16 < n_emit;
        float2 x[2][KSW_P][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          if (mt == 1 && !two) break;
          const int ea = m0 + 16 * mt + gid, eb = ea + 8;
          const bool va = ea < n_emit, vb = eb < n_emit;
          const int ba = va ? s_emit[ea] : 0, bb = vb ? s_emit[eb] : 0;
          const float* h_a = p.hbuf + (static_cast<size_t>(s_par[ba]) * B + ba) * HP;
          const float* h_b = p.hbuf + (static_cast<size_t>(s_par[bb]) * B + bb) * HP;
#pragma unroll
          for (int i = 0; i < KSW_P; ++i) {
            const int off = (kw * KSW_P + i) * 16 + tig * 2;
            x[mt][i][0] = va ? ldcg2(h_a + off) : make_float2(0.f, 0.f); x[mt][i][2] = va ? ldcg2(h_a + off + 8) : make_float2(0.f, 0.f);
            x[mt][i][1] = vb ? ldcg2(h_b + off) : make_float2(0.f, 0.f); x[mt][i][3] = vb ? ldcg2(h_b + off + 8) : make_float2(0.f, 0.f);
          }
        }
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          if (mt == 1 && !two) break;
          float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int i = 0; i < KSW_P; ++i) {
            const int ks = kw * KSW_P + i;
            uint32_t ah[4], al[4];
            split2(x[mt][i][0], ah[0], al[0]); split2(x[mt][i][1], ah[1], al[1]);
            split2(x[mt][i][2], ah[2], al[2]); split2(x[mt][i][3], ah[3], al[3]);
            const __nv_bfloat16* wr = s_wpred + static_cast<size_t>(min(gid, p.rows_p - 1)) * (HP + 8) + ks * 16 + tig * 2;   // clamped like the LSTM rows
            const uint32_t b0 = *reinterpret_cast<const uint32_t*>(wr), b1 = *reinterpret_cast<const uint32_t*>(wr + 8);
            mma_f16_16816(acc, ah, b0, b1); mma_f16_16816(acc, al, b0, b1);
          }
          float* r0 = red + (warp * 32 + 16 * mt + gid) * 8 + tig * 2;
          r0[0] = acc[0]; r0[1] = acc[1]; r0[8 * 8] = acc[2]; r0[8 * 8 + 1] = acc[3];
        }
        __syncthreads();
        if (tid < 32 * np) {
          const int el = tid / np, r = tid % np, e = m0 + el;
          if (e < n_emit) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kSpWarps; ++w) s += red[(w * 32 + el) * 8 + r];
            __stcg(p.ppbuf + static_cast<size_t>(s_emit[e]) * HJ + p0 + r, s + __ldg(p.b_pred + p0 + r));
          }
        }
        __syncthreads();
      }
    }
    tick(5, tk);
    sp_grid_barrier(p.counter, target, G);
    tick(6, tk);
  };

  // ordered compaction of the utterances that emitted (s_emit) and of those with frames left (s_act)
  auto compact = [&]() {
    int run_e = 0, run_a = 0;
    for (int base = 0; base < B; base += kSpThreads) {
      const int b = base + tid;
      const bool em = b < B && s_tok[b] >= 0, ac = b < B && s_t[b] < s_len[b];
      const unsigned me = __ballot_sync(0xffffffffu, em), ma = __ballot_sync(0xffffffffu, ac);
      if (lane == 0) { s_cnt[2 + warp] = __popc(me); s_cnt[2 + kSpWarps + warp] = __popc(ma); }
      __syncthreads();
      int bef_e = 0, bef_a = 0, tot_e = 0, tot_a = 0;
#pragma unroll
      for (int w = 0; w < kSpWarps; ++w) {
        const int ce = s_cnt[2 + w], ca = s_cnt[2 + kSpWarps + w];
        if (w < warp) { bef_e += ce; bef_a += ca; }
        tot_e += ce; tot_a += ca;
      }
      const unsigned below = (1u << lane) - 1u;
      if (em) s_emit[run_e + bef_e + __popc(me & below)] = b;
      if (ac) s_act[run_a + bef_a + __popc(ma & below)] = b;
      run_e += tot_e; run_a += tot_a;
      __syncthreads();
    }
    if (tid == 0) { s_cnt[0] = run_e; s_cnt[1] = run_a; }
    __syncthreads();
  };

  lstm_and_pred();                                // SOS: every utterance steps once on the blank (zero) embedding
  for (int b = tid; b < B; b += kSpThreads) s_tok[b] = -1;
  __syncthreads();
  compact();


  for (;;) {
    // ---- phase J
    if (has_j) {
      // the active utterances are dealt round-robin to the groups every iteration (any group can serve any utterance:
      // all hold the full vocabulary), so the groups stay balanced while utterances finish at different times
      const int n_act = s_cnt[1];
      const int n_pass = ((n_act + kGroups - 1) / kGroups + kPassUtts - 1) / kPassUtts;
      for (int pass = 0; pass < n_pass; ++pass) {
        // row r = (utterance ul of the pass, frame j of its window); lane r evaluates row r's validity for the ballot
        int row_b, row_t;
        {
          const int e = pass * kPassUtts + lane / kFrames, ai = grp + kGroups * e, j = lane % kFrames;
          const int b = ai < n_act ? s_act[ai] : 0;
          const bool ok = ai < n_act && s_t[b] + j < s_len[b];
          row_b = ok ? b : -1; row_t = ok ? s_t[b] + j : 0;
        }
        const unsigned mask = __ballot_sync(0xffffffffu, row_b >= 0);
        if (mask == 0u) continue;                             // identical in every warp of the CTA
        // loader item = (utterance of the pass, float4 column): pred_proj is fetched once for the four frames of a window
        // and the item order is rotated by the vocabulary-slice index so the 37 CTAs of a group, which all need the same
        // rows, do not ask L2 for the same lines at the same instant
        float4 gv[PERU][kFrames];
        auto load_half = [&](int h) {
#pragma unroll
          for (int i = 0; i < PERU; ++i) {
            int it = tid + kSpThreads * i;
            const bool in_range = it < ITEMS;
            it = (it + slice * 29) % ITEMS;
            const int ul = it / V4_ROW, c4 = it % V4_ROW;
            int rb[kFrames], rt[kFrames];
#pragma unroll
            for (int j = 0; j < kFrames; ++j) {
              rb[j] = __shfl_sync(0xffffffffu, row_b, ul * kFrames + j);     // every warp holds the row table, lane r = row r
              rt[j] = __shfl_sync(0xffffffffu, row_t, ul * kFrames + j);
            }
#pragma unroll
            for (int j = 0; j < kFrames; ++j) gv[i][j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (in_range && rb[0] >= 0) {
              const float4 q4 = ldcg4s(p.ppbuf + static_cast<size_t>(rb[0]) * HJ + h * KH + 4 * c4);
#pragma unroll
              for (int j = 0; j < kFrames; ++j) {
                if (rb[j] >= 0) {
                  const float4 e4 = __ldg(reinterpret_cast<const float4*>(p.enc_proj + (static_cast<size_t>(rb[j]) * p.T_max + rt[j]) * HJ + h * KH) + c4);
                  gv[i][j] = make_float4(fmaxf(e4.x + q4.x, 0.f), fmaxf(e4.y + q4.y, 0.f), fmaxf(e4.z + q4.z, 0.f), fmaxf(e4.w + q4.w, 0.f));
                }
              }
            }
          }
        };
#ifndef RS_NO_DECODE_COUNTERS
        long long tj = 0;
        if (cta == 0 && tid == 0) tj = clock64();
        auto jtick = [&](int slot) { if (cta == 0 && tid == 0) { const long long t1 = clock64(); prof[slot] += t1 - tj; tj = t1; } };
#else
        auto jtick = [&](int) {};
#endif
        {
          // ---- tcgen05 joint: D[vocabulary row, (utterance, frame) row] in tensor memory
          auto write_planes = [&]() {                         // gv -> two IEEE-half planes, 128B-swizzled K-major, 32 rows per slab
#pragma unroll
            for (int i = 0; i < PERU; ++i) {
              int it = tid + kSpThreads * i;
              if (it < ITEMS) {
                it = (it + slice * 29) % ITEMS;
                const int ul = it / V4_ROW, c4 = it % V4_ROW;
                const int kcol = 4 * c4;                      // column inside the k-half
                const uint32_t off_k = static_cast<uint32_t>(kcol >> 6) * kBSlab, chunk = (kcol & 63) >> 3, sub = (kcol & 7) * 2;
#pragma unroll
                for (int j = 0; j < kFrames; ++j) {
                  const int row = ul * kFrames + j;
                  uint32_t h0, l0, h1, l1;
                  split2(make_float2(gv[i][j].x, gv[i][j].y), h0, l0);
                  split2(make_float2(gv[i][j].z, gv[i][j].w), h1, l1);
                  uint8_t* dst = gB + off_k + (row >> 3) * 1024 + (row & 7) * 128 + ((chunk ^ (row & 7)) << 4) + sub;
                  *reinterpret_cast<uint2*>(dst) = make_uint2(h0, h1);
                  *reinterpret_cast<uint2*>(dst + 4096) = make_uint2(l0, l1);       // row + 32 of the same slab
                }
              }
            }
          };
          auto issue_half = [&](int h) {                      // one thread: NSLAB_H slabs x 4 k16 steps, N = 64 (hi | lo)
            tcgen05_fence_after();
#pragma unroll 1
            for (int sl = 0; sl < NSLAB_H; ++sl) {
              const uint64_t da = umma_desc_k_sw128(tc_base + static_cast<uint32_t>(h * NSLAB_H + sl) * a_slab);
              const uint64_t db = umma_desc_k_sw128(tc_base + b_off + sl * kBSlab);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_f16_ss(tmem_d, da + 2u * k, db + 2u * k, kIdescF16_128x64, (h | sl | k) != 0 ? 1u : 0u);
            }
            umma_commit(tc_bar);
          };
          load_half(0);
          write_planes();
          fence_proxy_async();
          tcgen05_fence_before();
          __syncthreads();
          jtick(8);
          if (tid == 0) issue_half(0);
          __syncwarp();
          load_half(1);                                       // in flight under the MMAs of half 0
          mbar_wait(tc_bar, mma_phase); mma_phase ^= 1u;      // half 0 consumed: the planes may be rewritten
          write_planes();
          fence_proxy_async();
          tcgen05_fence_before();
          __syncthreads();
          if (tid == 0) issue_half(1);
          __syncwarp();
          mbar_wait(tc_bar, mma_phase); mma_phase ^= 1u;
          tcgen05_fence_after();
          jtick(9);
          // ---- argmax over the vocabulary rows (= TMEM lanes) per (utterance, frame) column: warp w holds rows 32w..32w+31
          if (warp < 4) {
            uint32_t v[32], vlo[32];
            tmem_ld_32x32(tmem_d + (static_cast<uint32_t>(warp * 32) << 16), v);          // A . hi
            tmem_ld_32x32(tmem_d + (static_cast<uint32_t>(warp * 32) << 16) + 32, vlo);   // A . lo
            tmem_ld_wait();
            const int rr = warp * 32 + lane;
            const bool rvalid = rr < nj;
            const float bias = s_bout[rr];
            unsigned my_key = 0; int my_row = 0x7fffffff;
#pragma unroll
            for (int c = 0; c < 32; ++c) {
              unsigned fb = __float_as_uint((__uint_as_float(v[c]) + __uint_as_float(vlo[c])) + bias);
              fb = (fb & 0x80000000u) ? ~fb : (fb | 0x80000000u);               // order-preserving
              const unsigned key = rvalid ? fb : 0u;
              const unsigned mk = __reduce_max_sync(0xffffffffu, key);
              const unsigned cand = (key == mk && rvalid) ? static_cast<unsigned>(rr) : 0x7fffffffu;
              const unsigned mr = __reduce_min_sync(0xffffffffu, cand);         // ties -> lower row
              if (lane == c) { my_key = mk; my_row = static_cast<int>(mr); }
            }
            s_best[lane * 4 + warp] = (my_row != 0x7fffffff && my_key != 0u)
                                          ? ((static_cast<unsigned long long>(my_key) << 32) | (0xffffffffu - static_cast<unsigned>(j0 + my_row)))
                                          : 0ull;
          }
          tcgen05_fence_before();
        }
        __syncthreads();
        if (warp == 0 && row_b >= 0) {
          unsigned long long m = s_best[lane * 4];
#pragma unroll
          for (int q = 1; q < 4; ++q) { const unsigned long long o = s_best[lane * 4 + q]; m = o > m ? o : m; }
          asm volatile("red.relaxed.gpu.global.max.u64 [%0], %1;" ::"l"(p.best + (static_cast<size_t>(iter % 3) * B + row_b) * kFrames + (lane % kFrames)), "l"(m) : "memory");
        }
        jtick(10);
        // s_best / s_g are rewritten only after the next pass's first __syncthreads pair; the reads above are by warp 0
        // before it reaches that barrier
      }
    }
    tick(0, tk);
    sp_grid_barrier(p.counter, target, G);
    tick(1, tk);
    // ---- consume the window (identically in every CTA): blanks advance t, the first non-blank emits and ends the window
    for (int b = tid; b < B; b += kSpThreads) {
      int t = s_t[b];
      const int len = s_len[b];
      int tok = -1;
      if (t < len) {
        const int nv = min(kFrames, len - t);
        int sym = s_sym[b];
        const ulonglong2* bp = reinterpret_cast<const ulonglong2*>(p.best + (static_cast<size_t>(iter % 3) * B + b) * kFrames);
        static_assert(kFrames == 4, "window read as two 16-byte loads");
        const ulonglong2 w01 = __ldcg(bp), w23 = __ldcg(bp + 1);
        const unsigned long long win[kFrames] = {w01.x, w01.y, w23.x, w23.y};
#pragma unroll
        for (int j = 0; j < kFrames; ++j) {
          if (j >= nv) break;
          const unsigned long long v = win[j];
          const int k = static_cast<int>(0xffffffffu - static_cast<unsigned int>(v & 0xffffffffull));
          if (k == blank) { t += 1; sym = 0; continue; }
          const int n = s_n[b];
          if (cta == 0 && n < p.U_max) {
            p.tokens[static_cast<size_t>(b) * p.U_max + n] = k;
            p.frames[static_cast<size_t>(b) * p.U_max + n] = t;
          }
          s_n[b] = n + 1;
          tok = k;
          if (++sym >= p.max_symbols) { t += 1; sym = 0; }
          break;
        }
        s_t[b] = t; s_sym[b] = sym;
      }
      s_tok[b] = tok;
    }
    // the slot that iteration iter+2 will use was last read two barriers ago: clear it now (visible through the
    // next barrier, which precedes that iteration's red.max)
    if (cta == 0) for (int i = tid; i < B * kFrames; i += kSpThreads) __stcg(p.best + static_cast<size_t>((iter + 2) % 3) * B * kFrames + i, 0ull);
    ++iter;
    __syncthreads();
    compact();
    const int n_active = s_cnt[1];
    tick(2, tk);
    prof[7] += 1;
    if (s_cnt[0] > 0) lstm_and_pred();
    if (n_active == 0) break;
  }
  if (cta == 0) for (int b = tid; b < B; b += kSpThreads) p.n_tok[b] = s_n[b];
  if (cta == 0 && tid == 0) for (int i = 0; i < 12; ++i) p.prof[i] = prof[i];
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) { tcgen05_fence_after(); tmem_dealloc<64>(tmem_d); }
}

// workspace: hbuf | ppbuf | pad to 128 | barrier counters (kBarCounters lines) | prof (128 B) | best
static size_t spec_counter_offset(int B, int Hj, int Hp) {
  return (static_cast<size_t>(2) * B * Hp * 4 + static_cast<size_t>(B) * Hj * 4 + 127) & ~static_cast<size_t>(127);
}
size_t rnnt_spec_prof_offset(int B, int Hj, int Hp) { return spec_counter_offset(B, Hj, Hp) + static_cast<size_t>(kBarCounters) * kBarStride * 4; }
size_t rnnt_spec_workspace_bytes(int B, int Hj, int Hp, int /*num_sms*/) {
  return rnnt_spec_prof_offset(B, Hj, Hp) + 128 + static_cast<size_t>(3) * B * kFrames * 8 + 128 /*base alignment slack*/;
}

template <int HJ, int HP>
static cudaError_t launch_sp(SpecDev p, int grid, size_t smem, cudaStream_t stream) {
  cudaError_t e = cudaFuncSetAttribute(rnnt_greedy_spec_kernel<HJ, HP>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rnnt_greedy_spec_kernel<HJ, HP>, kSpThreads, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorLaunchOutOfResources;
  void* args[] = {&p};
  return cudaLaunchCooperativeKernel(reinterpret_cast<void*>(rnnt_greedy_spec_kernel<HJ, HP>), dim3(grid), dim3(kSpThreads), args, smem, stream);
}

cudaError_t launch_rnnt_greedy_spec(const DecodeArgs& a, void* workspace, int num_sms, cudaStream_t stream) {
  if (a.B <= 0 || num_sms < kGroups) return cudaErrorInvalidValue;
  const int G = num_sms;
  SpecDev p;
  p.enc_proj = a.enc_proj; p.enc_len = a.enc_len;
  p.w_out = static_cast<const __nv_bfloat16*>(a.w_out); p.b_out = a.b_out; p.embed = a.embed;
  p.w_lstm = static_cast<const __nv_bfloat16*>(a.w_lstm); p.gate_tab = a.gate_tab;
  p.w_pred = static_cast<const __nv_bfloat16*>(a.w_pred); p.b_pred = a.b_pred;
  p.tokens = a.tokens; p.frames = a.frames; p.n_tok = a.n_tok;
  if (reinterpret_cast<uintptr_t>(workspace) & 15u) return cudaErrorInvalidValue;   // the window is read with 16-byte loads
  char* ws = static_cast<char*>(workspace);
  p.hbuf = reinterpret_cast<float*>(ws);
  p.ppbuf = reinterpret_cast<float*>(ws + static_cast<size_t>(2) * a.B * a.Hp * 4);
  p.counter = reinterpret_cast<unsigned int*>(ws + spec_counter_offset(a.B, a.Hj, a.Hp));
  p.prof = reinterpret_cast<long long*>(ws + rnnt_spec_prof_offset(a.B, a.Hj, a.Hp));
  p.best = reinterpret_cast<unsigned long long*>(ws + rnnt_spec_prof_offset(a.B, a.Hj, a.Hp) + 128);
  p.B = a.B; p.T_max = a.T_max; p.V = a.V; p.U_max = a.U_max; p.max_symbols = a.max_symbols;
  p.S = G / kGroups;
  p.rows_j = (a.V + 1 + p.S - 1) / p.S;
  p.units = (a.Hp + G - 1) / G;
  p.rows_p = (a.Hj + G - 1) / G;
  if (4 * p.units > 24 || p.rows_p > 8 || 32 * p.units > kSpThreads || 32 * p.rows_p > kSpThreads || a.gate_tab == nullptr) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(workspace, 0, rnnt_spec_workspace_bytes(a.B, a.Hj, a.Hp, num_sms), stream);
  if (e != cudaSuccess) return e;
  const size_t state = ((static_cast<size_t>(a.B) * p.units + 1) & ~static_cast<size_t>(1)) * 4 + kPassRows * 4 * 8 + static_cast<size_t>(a.B) * 8 * 4 +
                       (2 + 2 * kSpWarps) * 4 + 64;
  const size_t w_lp = (static_cast<size_t>(4 * p.units) * (a.Hp + 8) + static_cast<size_t>(p.rows_p) * (a.Hp + 8)) * 2;
  if (p.rows_j > 128) return cudaErrorInvalidValue;
  const size_t rows_a8 = (p.rows_j + 7) & ~7;
  const size_t b_bytes = static_cast<size_t>(a.Hj / 2 / 64) * 8192;
  const size_t b_region = b_bytes > 24576 ? b_bytes : 24576;     // also the [8 warps][32][24] fp32 reduction buffer of the LSTM phase
  const size_t ab = ((static_cast<size_t>(a.Hj / 64) * rows_a8 * 128 + w_lp + 1023) & ~static_cast<size_t>(1023));   // A slabs, W_lstm, W_pred, pad
  const size_t smem = 1024 + ab + b_region + 128 * 4 + state + 16;
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  if (a.Hj == 640 && a.Hp == 640) return launch_sp<640, 640>(p, G, smem, stream);
  if (a.Hj == 128 && a.Hp == 128) return launch_sp<128, 128>(p, G, smem, stream);
  return cudaErrorInvalidValue;
}

}  // namespace rs
