// RNN-T forced alignment of known token sequences (semantics: oracle/align_restated.py).  For utterance b with T encoder
// frames and targets y_1..y_U the lattice node (t, u), t < T, u <= U, carries
//   lb(t, u) = log_softmax(z)[blank],  ly(t, u) = log_softmax(z)[y_{u+1}],  z = W_out relu(f_t + g_u) + b_out,
// f_t = joint.enc(enc_t), g_u = joint.pred(h_u), h_u the predictor state after the SOS step and y_1..y_u (teacher-forced).
// Like the ALSD search (decode_alsd.cu) every matrix product meets its activations as three bf16 terms against tripled
// bf16-exact weights, so the log-probabilities are fp32-accurate.
//
//   align_check     targets outside [0, V) -> a flag the host reads before anything indexes with them
//   [GEMM] + align_pred (x U_max + 1)   LSTM gates of [embed[y_k] | h_{k-1}] -> cell -> h_k planes, next step's input
//   [GEMM]          g = joint.pred of every h_u at once
//   per chunk of kAlignChunkRows nodes:
//     align_rows      relu(f_t + g_u) -> three bf16 planes, target column
//     align_lattice   persistent TMA -> tcgen05.mma -> TMEM kernel: one CTA owns a 128-row block across all N blocks and
//                     reduces the logits to (log p(blank), log p(target)) in its epilogue; no logit reaches HBM
//   align_dp        anti-diagonal sweep per utterance: Viterbi (max) and forward (logaddexp) in float64, backtrace
//
// rs_rnnt_align_spans runs the same kernels over K frame windows of the encoder rows (semantics:
// oracle/align_spans_restated.py): the predictor over the K items, align_rows reading joint.enc rows from a per-item row
// base (src * T_max + lo; b * T_max for whole utterances), align_dp<kSpan = true> letting the path start and end anywhere.
#include <cuda.h>

#include <cfloat>
#include <cmath>
#include <cstdio>

#include "align.h"
#include "common.cuh"
#include "kernels.h"
#include "rnnt_cell.cuh"

namespace rs {

namespace {

// ---------------------------------------------------------------------------------------------- argument check
__global__ void align_check_kernel(const int32_t* __restrict__ targets, const int32_t* __restrict__ tgt_len, int B, int U_max, int V,
                                   int* __restrict__ bad) {
  const int64_t n = static_cast<int64_t>(B) * U_max;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(i / U_max), u = static_cast<int>(i % U_max);
    const int y = targets[i];
    if (u < tgt_len[b] && (y < 0 || y >= V)) atomicOr(bad, 1);
  }
}

// ---------------------------------------------------------------------------------------------- teacher-forced predictor
// grid (B), block 128.  Rows whose utterance has fewer than k targets are zero-filled (the GEMMs read them, nothing uses them).
__global__ void __launch_bounds__(128)
align_pred_kernel(const float* __restrict__ gates, float* __restrict__ c_state, const int32_t* __restrict__ targets,
                  const int32_t* __restrict__ tgt_len, int U_max, int U1, int k, const float* __restrict__ embed, int Hp,
                  __nv_bfloat16* __restrict__ in_planes, __nv_bfloat16* __restrict__ h_planes) {
  const int b = blockIdx.x;
  const int U = tgt_len[b];
  const bool active = k <= U, next = k < U;
  const float* g = gates + static_cast<size_t>(b) * 4 * Hp;
  const float* e = embed + static_cast<size_t>(next ? targets[static_cast<size_t>(b) * U_max + k] : 0) * Hp;
  __nv_bfloat16* hrow = h_planes + (static_cast<size_t>(b) * U1 + k) * 3 * Hp;
  __nv_bfloat16* irow = in_planes + static_cast<size_t>(b) * 6 * Hp;
  for (int j = threadIdx.x; j < Hp; j += blockDim.x) {
    float h = 0.f;
    if (active) {
      float c;
      lstm_cell(g[j], g[Hp + j], g[2 * Hp + j], g[3 * Hp + j], k == 0 ? 0.f : c_state[static_cast<size_t>(b) * Hp + j], h, c);
      c_state[static_cast<size_t>(b) * Hp + j] = c;
    }
    __nv_bfloat16 hi, mid, lo;
    split3(h, hi, mid, lo);
    hrow[j] = hi; hrow[Hp + j] = mid; hrow[2 * Hp + j] = lo;
    if (!next) hi = mid = lo = __float2bfloat16_rn(0.f);
    irow[Hp + j] = hi; irow[3 * Hp + j] = mid; irow[5 * Hp + j] = lo;    // [embed | h] in each 2Hp-wide plane
    split3(next ? e[j] : 0.f, hi, mid, lo);
    irow[j] = hi; irow[2 * Hp + j] = mid; irow[4 * Hp + j] = lo;
  }
}

// ---------------------------------------------------------------------------------------------- lattice rows
// grid (n_rows), block 128.  (The lattice kernel's TMA zero-fills the rows of its last tile past n_rows.)
__global__ void __launch_bounds__(128)
align_rows_kernel(const float* __restrict__ enc_proj, const float* __restrict__ pred_proj, const int64_t* __restrict__ offs,
                  const int64_t* __restrict__ row_base, const int32_t* __restrict__ tgt_len, const int32_t* __restrict__ targets,
                  int B, int U1, int U_max, int Hj, int64_t r0, __nv_bfloat16* __restrict__ planes, int32_t* __restrict__ tcol) {
  const int r = blockIdx.x;
  __nv_bfloat16* row = planes + static_cast<size_t>(r) * 3 * Hj;
  const int64_t n = r0 + r;
  int lo = 0, hi = B - 1;                                  // the utterance whose node range holds n
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (offs[mid] <= n) lo = mid; else hi = mid - 1;
  }
  const int b = lo, U = tgt_len[b];
  const int64_t local = n - offs[b];
  const int t = static_cast<int>(local / (U + 1)), u = static_cast<int>(local % (U + 1));
  if (threadIdx.x == 0) tcol[r] = u < U ? targets[static_cast<size_t>(b) * U_max + u] : -1;
  const float4* ep = reinterpret_cast<const float4*>(enc_proj + static_cast<size_t>(row_base[b] + t) * Hj);
  const float4* pp = reinterpret_cast<const float4*>(pred_proj + (static_cast<size_t>(b) * U1 + u) * Hj);
  for (int j4 = threadIdx.x; j4 < Hj / 4; j4 += blockDim.x) {
    const float4 a = ep[j4], g = pp[j4];
    const float x[4] = {fmaxf(a.x + g.x, 0.f), fmaxf(a.y + g.y, 0.f), fmaxf(a.z + g.z, 0.f), fmaxf(a.w + g.w, 0.f)};
    __nv_bfloat16 h[4], m[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) split3(x[i], h[i], m[i], l[i]);
    const auto pack = [](const __nv_bfloat16 (&v)[4]) {
      return make_uint2(static_cast<uint32_t>(__bfloat16_as_ushort(v[0])) | (static_cast<uint32_t>(__bfloat16_as_ushort(v[1])) << 16),
                        static_cast<uint32_t>(__bfloat16_as_ushort(v[2])) | (static_cast<uint32_t>(__bfloat16_as_ushort(v[3])) << 16));
    };
    reinterpret_cast<uint2*>(row)[j4] = pack(h);
    reinterpret_cast<uint2*>(row + Hj)[j4] = pack(m);
    reinterpret_cast<uint2*>(row + 2 * Hj)[j4] = pack(l);
  }
}

// ---------------------------------------------------------------------------------------------- fused joint + log-softmax
//   warp 0      TMA producer   A (128 rows x 64 K) and W (256 rows x 64 K) tiles, 128B swizzle -> 4-stage smem ring
//   warp 1      MMA issuer     tcgen05.mma 128 x 256 x 16, fp32 accumulators in TMEM, two stages (512 columns)
//   warps 2..9  epilogue       one thread per row and column half (128 columns of the 256-wide N block): running
//                              (max, sum exp) over the row's N blocks, the blank and target logits; the halves merge in
//                              shared memory after the last N block.  Overlaps the MMAs of the next N block.
constexpr int kLatBM = 128, kLatBN = 256, kLatBK = 64, kLatStages = 4, kLatEpiWarps = 8;
constexpr int kLatThreads = 32 * (2 + kLatEpiWarps);
constexpr int kLatABytes = kLatBM * kLatBK * 2, kLatBBytes = kLatBN * kLatBK * 2, kLatStageBytes = kLatABytes + kLatBBytes;
constexpr int kLatTmemCols = 2 * kLatBN;
constexpr int kLatSmemBytes = kLatStages * kLatStageBytes + 1024 /*align slack*/ + 256 /*barriers*/ + kLatBM * 4 * 4 /*half merge*/;
static_assert(kLatSmemBytes <= 227 * 1024, "shared memory layout");

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kLatEpiWarps) : "memory"); }

__global__ void __launch_bounds__(kLatThreads, 1)
align_lattice_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const float* __restrict__ bias,
                     const int32_t* __restrict__ tcol, float2* __restrict__ out, int M, int N, int K, int V) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + kLatStages * kLatStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kLatStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kLatStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kLatStages + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * kLatStages + 4);
  float4* merge = reinterpret_cast<float4*>(smem_raw + ((bar_base + 256u) - smem_u32(smem_raw)));   // [128 rows] of the upper half
  auto smem_a = [&](int s) { return smem_base + s * kLatStageBytes; };
  auto smem_b = [&](int s) { return smem_base + s * kLatStageBytes + kLatABytes; };

  const int warp = warp_id_uniform();
  const int lane = lane_id();
  const int num_m = (M + kLatBM - 1) / kLatBM;
  const int num_n = (N + kLatBN - 1) / kLatBN;
  const int num_k = K / kLatBK;
  const int NC = V + 1;                                    // classes; columns >= NC are padding (zero logits, not -inf)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    for (int s = 0; s < kLatStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), kLatEpiWarps); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<kLatTmemCols>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int mb = blockIdx.x; mb < num_m; mb += gridDim.x)
        for (int nb = 0; nb < num_n; ++nb)
          for (int kb = 0; kb < num_k; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            mbar_arrive_expect_tx(full_bar(stage), kLatStageBytes);        // out-of-range rows are zero-filled and counted
            tma_load_2d(smem_a(stage), &tm_a, kb * kLatBK, mb * kLatBM, full_bar(stage));
            tma_load_2d(smem_b(stage), &tm_b, kb * kLatBK, nb * kLatBN, full_bar(stage));
            if (++stage == kLatStages) { stage = 0; phase ^= 1u; }
          }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(kLatBM, kLatBN);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int mb = blockIdx.x; mb < num_m; mb += gridDim.x)
        for (int nb = 0; nb < num_n; ++nb, ++it) {
          const int acc = it & 1;
          mbar_wait(tempty_bar(acc), ((it >> 1) & 1u) ^ 1u);
          tcgen05_fence_after();
          const uint32_t d_tmem = tmem_base + acc * kLatBN;
          for (int kb = 0; kb < num_k; ++kb) {
            mbar_wait(full_bar(stage), phase);
            tcgen05_fence_after();
            const uint64_t da = umma_desc_k_sw128(smem_a(stage));
            const uint64_t db = umma_desc_k_sw128(smem_b(stage));
#pragma unroll
            for (int k = 0; k < kLatBK / 16; ++k) umma_bf16_ss(d_tmem, da + 2u * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit(empty_bar(stage));
            if (++stage == kLatStages) { stage = 0; phase ^= 1u; }
          }
          umma_commit(tfull_bar(acc));
        }
    }
  } else {
    const int q = warp & 3;                                // TMEM lane quarter = the warp's 32 rows
    const int half = (warp - 2) >> 2;                      // which 128 columns of the N block
    int it = 0;
    for (int mb = blockIdx.x; mb < num_m; mb += gridDim.x) {
      const int rl = q * 32 + lane, row = mb * kLatBM + rl;
      const int tc = row < M ? tcol[row] : -1;
      float mx = -INFINITY, se = 0.f, lb = -INFINITY, ly = -INFINITY;
      for (int nb = 0; nb < num_n; ++nb, ++it) {
        const int acc = it & 1;
        mbar_wait(tfull_bar(acc), (it >> 1) & 1u);
        tcgen05_fence_after();
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          const int col0 = nb * kLatBN + half * 128 + c * 32;
          if (col0 >= NC) break;                           // warp-uniform: only padding beyond
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kLatBN + half * 128 + c * 32, r);
          tmem_ld_wait();
          float v[32];
          const float4* b4 = reinterpret_cast<const float4*>(bias + col0);   // col0 + 32 <= n_pad: col0 < NC, both multiples of 32
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 bb = __ldg(b4 + j);
            v[4 * j] = __uint_as_float(r[4 * j]) + bb.x; v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + bb.y;
            v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + bb.z; v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + bb.w;
          }
          if (col0 + 32 > NC) {                            // the chunk holding the last class: padding columns leave the sum
#pragma unroll
            for (int j = 0; j < 32; ++j) if (col0 + j >= NC) v[j] = -INFINITY;
          }
          if (static_cast<unsigned>(V - col0) < 32u) {     // blank column
#pragma unroll
            for (int j = 0; j < 32; ++j) if (col0 + j == V) lb = v[j];
          }
          if (static_cast<unsigned>(tc - col0) < 32u) {    // this row's target column
#pragma unroll
            for (int j = 0; j < 32; ++j) if (col0 + j == tc) ly = v[j];
          }
          float cm = v[0];
#pragma unroll
          for (int j = 1; j < 32; ++j) cm = fmaxf(cm, v[j]);
          if (cm > mx) { se *= __expf(mx - cm); mx = cm; }
          float s = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) s += __expf(v[j] - mx);
          se += s;
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
      }
      // merge the two column halves of the row
      if (half == 1) merge[rl] = make_float4(mx, se, lb, ly);
      epi_bar_sync();
      if (half == 0 && row < M) {
        const float4 o = merge[rl];
        const float m2 = fmaxf(mx, o.x);
        const float lse = m2 + logf(se * expf(mx - m2) + o.y * expf(o.x - m2));
        const float blank = fmaxf(lb, o.z), tgt = fmaxf(ly, o.w);
        out[row] = make_float2(blank - lse, tc >= 0 ? tgt - lse : 0.f);
      }
      epi_bar_sync();                                      // merge slots free for the next row block
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<kLatTmemCols>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------- Viterbi + forward
__device__ __forceinline__ double logaddexp(double a, double b) {
  const double hi = a > b ? a : b, lo = a > b ? b : a;
  return hi + log1p(exp(lo - hi));
}

// grid (B), block 256.  Anti-diagonal d = t + u; two diagonals of (Viterbi, forward) in shared memory indexed by u.
// Back-pointer per node: 1 = reached by emitting y_u from (t, u - 1), 0 = by a blank from (t - 1, u), which wins exact ties:
// the backtrace runs from the last node, so preferring the blank edge moves every token to its earliest frame.
//
// kSpan (rs_rnnt_align_spans): item b is the frame window [lo, hi) of span[b], T = hi - lo (enc_len holds T, T_max the row
// pitch F_max of path_logp and lattice).  The path may start at any node (t, 0) at no cost -- back-pointer 2, which wins an
// exact tie with the blank edge -- and ends with the closing blank of any frame t_e at u = U.  The end terms are folded in
// ascending t by whichever thread owns the diagonal's node (t, U): a strict running max (the earliest t_e wins a tie) and a
// running logaddexp, in shared memory after the four diagonals.  The backtrace runs from (t_e, U) to the first start state;
// frames are reported as lo + t, and path_logp[b, t] of every frame of the span is lb(t, u_t) plus the ly of the tokens the
// path emits at t, summed in fp32 in that order (the blank, then the tokens from the last to the first); 0 elsewhere.
template <bool kSpan>
__global__ void __launch_bounds__(256)
align_dp_kernel(const float2* __restrict__ lp, const int64_t* __restrict__ offs, const int32_t* __restrict__ enc_len,
                const int32_t* __restrict__ tgt_len, int T_max, int U_max, int U1, uint8_t* __restrict__ bp_all,
                int32_t* __restrict__ frames, float* __restrict__ tok_logp, double* __restrict__ viterbi, double* __restrict__ loglik,
                float* __restrict__ lattice, const int32_t* __restrict__ span, float* __restrict__ path_logp) {
  extern __shared__ double dp_smem[];
  const int b = blockIdx.x;
  const int T = enc_len[b], U = tgt_len[b], W = U + 1;
  const float2* L = lp + offs[b];
  uint8_t* P = bp_all + offs[b];
  auto av = [&](int i) { return dp_smem + i * U1; };             // [Viterbi even | Viterbi odd | forward even | forward odd]
  auto af = [&](int i) { return dp_smem + (2 + i) * U1; };
  double* end_acc = dp_smem + 4 * U1;                            // kSpan: [Viterbi end max, forward end sum], then t_e
  int* end_t = reinterpret_cast<int*>(end_acc + 2);
  if (lattice != nullptr) {
    for (int i = threadIdx.x; i < T * W; i += blockDim.x) {
      const int t = i / W, u = i % W;
      const float2 x = L[i];
      float* dst = lattice + ((static_cast<size_t>(b) * T_max + t) * (U_max + 1) + u) * 2;
      dst[0] = x.x; dst[1] = x.y;
    }
  }
  for (int u = U + threadIdx.x; u < U_max; u += blockDim.x) {
    frames[static_cast<size_t>(b) * U_max + u] = -1;
    tok_logp[static_cast<size_t>(b) * U_max + u] = 0.f;
  }
  if constexpr (kSpan) {
    for (int t = threadIdx.x; t < T_max; t += blockDim.x) path_logp[static_cast<size_t>(b) * T_max + t] = 0.f;
  }
  for (int d = 0; d < T + U; ++d) {
    const double* pv = av((d & 1) ^ 1); const double* pf = af((d & 1) ^ 1);
    double* cv = av(d & 1); double* cf = af(d & 1);
    const int u_lo = d - (T - 1) > 0 ? d - (T - 1) : 0, u_hi = d < U ? d : U;
    for (int u = u_lo + threadIdx.x; u <= u_hi; u += blockDim.x) {
      const int t = d - u;
      double v = 0.0, f = 0.0;
      uint8_t e = 0;
      if (t > 0 && u > 0) {
        const double lb = static_cast<double>(L[(t - 1) * W + u].x), ly = static_cast<double>(L[t * W + u - 1].y);
        const double vb = pv[u] + lb, ve = pv[u - 1] + ly;
        e = ve > vb;
        v = e ? ve : vb;
        f = logaddexp(pf[u] + lb, pf[u - 1] + ly);
      } else if (u > 0) {
        const double ly = static_cast<double>(L[t * W + u - 1].y);
        v = pv[u - 1] + ly; f = pf[u - 1] + ly; e = 1;
      } else if (t > 0) {
        const double lb = static_cast<double>(L[(t - 1) * W + u].x);
        v = pv[u] + lb; f = pf[u] + lb;
        if constexpr (kSpan) {                                   // fresh start at (t, 0): 0, wins an exact tie
          e = v > 0.0 ? 0 : 2;
          v = e ? 0.0 : v;
          f = logaddexp(0.0, f);
        }
      } else if constexpr (kSpan) {
        e = 2;
      }
      cv[u] = v; cf[u] = f;
      P[t * W + u] = e;
      if constexpr (kSpan) {
        if (u == U) {                                            // one node per diagonal, diagonals in ascending t
          const double lb_end = static_cast<double>(L[t * W + U].x);
          const double ve = v + lb_end, fe = f + lb_end;
          if (t == 0) {
            end_acc[0] = ve; end_acc[1] = fe; *end_t = 0;
          } else {
            if (ve > end_acc[0]) { end_acc[0] = ve; *end_t = t; }
            end_acc[1] = logaddexp(end_acc[1], fe);
          }
        }
      }
    }
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  if constexpr (kSpan) {
    viterbi[b] = end_acc[0];
    loglik[b] = end_acc[1];
    const int lo = span[3 * b + 1];
    int t = *end_t, u = U;
    float acc = L[t * W + U].x;
    for (;;) {
      const uint8_t p = P[t * W + u];
      if (p == 1) {
        --u;
        const float y = L[t * W + u].y;
        frames[static_cast<size_t>(b) * U_max + u] = lo + t;
        tok_logp[static_cast<size_t>(b) * U_max + u] = y;
        acc += y;
      } else {
        path_logp[static_cast<size_t>(b) * T_max + t] = acc;
        if (p == 2) break;
        --t;
        acc = L[t * W + u].x;
      }
    }
  } else {
    const int dl = T - 1 + U;
    const double lb_end = static_cast<double>(L[(T - 1) * W + U].x);
    viterbi[b] = av(dl & 1)[U] + lb_end;
    loglik[b] = af(dl & 1)[U] + lb_end;
    int t = T - 1, u = U;
    while (u > 0) {
      if (P[t * W + u]) {
        --u;
        frames[static_cast<size_t>(b) * U_max + u] = t;
        tok_logp[static_cast<size_t>(b) * U_max + u] = L[t * W + u].y;
      } else {
        --t;
      }
    }
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------ host side
cudaError_t align_check(const int32_t* targets, const int32_t* tgt_len, int B, int U_max, int V, int* bad, cudaStream_t s) {
  const int64_t n = static_cast<int64_t>(B) * U_max;
  const int grid = static_cast<int>(n / 256 + 1 < 1024 ? n / 256 + 1 : 1024);
  align_check_kernel<<<grid, 256, 0, s>>>(targets, tgt_len, B, U_max, V, bad);
  return cudaGetLastError();
}

cudaError_t align_pred(const float* gates, float* c_state, const int32_t* targets, const int32_t* tgt_len, int B, int U_max, int U1,
                       int k, const float* embed, int Hp, void* in_planes, void* h_planes, cudaStream_t s) {
  align_pred_kernel<<<B, 128, 0, s>>>(gates, c_state, targets, tgt_len, U_max, U1, k, embed, Hp, static_cast<__nv_bfloat16*>(in_planes),
                                      static_cast<__nv_bfloat16*>(h_planes));
  return cudaGetLastError();
}

cudaError_t align_rows(const float* enc_proj, const float* pred_proj, const int64_t* offs, const int64_t* row_base,
                       const int32_t* tgt_len, const int32_t* targets, int B, int U1, int U_max, int Hj, int64_t r0, int n_rows,
                       void* planes, int32_t* tcol, cudaStream_t s) {
  align_rows_kernel<<<n_rows, 128, 0, s>>>(enc_proj, pred_proj, offs, row_base, tgt_len, targets, B, U1, U_max, Hj, r0,
                                           static_cast<__nv_bfloat16*>(planes), tcol);
  return cudaGetLastError();
}

cudaError_t align_lattice(const void* planes, const void* w3, const float* bias, const int32_t* tcol, float2* out, int n_rows,
                          int n_pad, int Hj, int V, int num_sms, cudaStream_t s, char* err) {
  const int K = 3 * Hj;
  if (K % kLatBK != 0 || n_pad % 64 != 0 || V + 1 > n_pad) {
    snprintf(err, 256, "align_lattice: unsupported shape (3*Hj=%d must be a multiple of 64, n_pad=%d of 64, V+1 <= n_pad)", K, n_pad);
    return cudaErrorInvalidValue;
  }
  static DeviceOnce attr_once;
  if (attr_once.pending()) {
    cudaError_t e = cudaFuncSetAttribute(align_lattice_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLatSmemBytes);
    if (e != cudaSuccess) { snprintf(err, 256, "cudaFuncSetAttribute(smem=%d): %s", kLatSmemBytes, cudaGetErrorString(e)); return e; }
    attr_once.set();
  }
  CUtensorMap tm_a, tm_b;
  if (!make_tmap_bf16(&tm_a, planes, n_rows, K, K, kLatBM, err)) return cudaErrorInvalidValue;
  if (!make_tmap_bf16(&tm_b, w3, n_pad, K, K, kLatBN, err)) return cudaErrorInvalidValue;
  const int blocks = (n_rows + kLatBM - 1) / kLatBM;
  const int grid = blocks < num_sms ? blocks : num_sms;
  align_lattice_kernel<<<grid, kLatThreads, kLatSmemBytes, s>>>(tm_a, tm_b, bias, tcol, out, n_rows, n_pad, K, V);
  return cudaGetLastError();
}

size_t align_dp_smem_bytes(int U1, bool span) { return static_cast<size_t>(4) * U1 * sizeof(double) + (span ? 32 : 0); }

namespace {
template <bool kSpan>
cudaError_t launch_dp(const float2* lp, const int64_t* offs, const int32_t* enc_len, const int32_t* tgt_len, int B, int T_max,
                      int U_max, int U1, uint8_t* bp, int32_t* frames, float* tok_logp, double* viterbi, double* loglik, float* lattice,
                      const int32_t* span, float* path_logp, cudaStream_t s) {
  const size_t smem = align_dp_smem_bytes(U1, kSpan);
  if (smem > 48 * 1024) {
    static DeviceOnce attr_once;
    if (attr_once.pending()) {
      cudaError_t e = cudaFuncSetAttribute(align_dp_kernel<kSpan>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      if (e != cudaSuccess) return e;
      attr_once.set();
    }
  }
  align_dp_kernel<kSpan><<<B, 256, smem, s>>>(lp, offs, enc_len, tgt_len, T_max, U_max, U1, bp, frames, tok_logp, viterbi, loglik,
                                              lattice, span, path_logp);
  return cudaGetLastError();
}
}  // namespace

cudaError_t align_dp(const float2* lp, const int64_t* offs, const int32_t* enc_len, const int32_t* tgt_len, int B, int T_max,
                     int U_max, int U1, uint8_t* bp, int32_t* frames, float* tok_logp, double* viterbi, double* loglik, float* lattice,
                     const int32_t* span, float* path_logp, cudaStream_t s) {
  return span != nullptr
             ? launch_dp<true>(lp, offs, enc_len, tgt_len, B, T_max, U_max, U1, bp, frames, tok_logp, viterbi, loglik, lattice, span,
                               path_logp, s)
             : launch_dp<false>(lp, offs, enc_len, tgt_len, B, T_max, U_max, U1, bp, frames, tok_logp, viterbi, loglik, lattice,
                                nullptr, nullptr, s);
}

}  // namespace rs
