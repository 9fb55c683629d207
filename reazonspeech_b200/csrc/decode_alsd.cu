// ALSD beam search (alignment-length synchronous decoding) for the RNN-T head, batched over utterances: NeMo's
// BeamRNNTInfer.align_length_sync_decoding, the strategy the shipped reazonspeech-nemo-v2 checkpoint decodes with by default
// -- the reference's own post-processing is written for its hypotheses (pkg/nemo-asr/src/decode.py:29 "Decode ALSD beam search
// info", :38-40 the leading blank of y_sequence, :48 step - idx - 1).  Semantics restated in oracle/alsd_restated.py.
//
// One step = one anti-diagonal i = t + u of the (frame, token) lattice for every utterance at once.  The three matrix products
// of a step (joint logits of the live hypotheses, LSTM gates and joint.pred of the newly extended ones) go through the tcgen05
// GEMM of gemm_tcgen05.cu with their fp32 activations split into three bf16 terms (24 mantissa bits against bf16-exact
// weights: fp32-accurate log-probabilities, so that beam decisions move only with the encoder's rounding, not the decoder's);
// this file holds the kernels in between:
//
//   alsd_rows_kernel     live (utterance, hypothesis) rows: relu(enc_proj[b, t] + pred_proj[b, k]) -> three bf16 planes
//   [GEMM]               logits[rows, V + 1] = planes . [W_out | W_out | W_out]^T + b_out
//   alsd_reduce_kernel   per row: log-sum-exp, log p(blank), the `beam` best non-blank classes (ties: lower index)
//   alsd_select_kernel   per utterance: A = [stay, extensions ...] per live hypothesis in beam order, the `beam` best by score
//                        (stable: ties keep A's order, as Python's sorted does), NeMo's recombine_hypotheses, the finished
//                        list (hypotheses that took the blank at the last frame), back-pointer nodes of the extensions
//   alsd_lstm_in_kernel  extended hypotheses: [embed[token] | h_parent] -> three bf16 planes
//   [GEMM]               gates = planes . [W_lstm x3]^T + b
//   alsd_cell_kernel     LSTM cell, new (h, c); h -> three bf16 planes         (kept hypotheses: state copied from the parent)
//   [GEMM]               pred_proj = planes . [W_pred x3]^T + b_pred
//   alsd_commit_kernel   the new beam's state / pred_proj become current
//
// Scores are doubles (Python floats in NeMo), log-probabilities fp32 (torch.log_softmax of fp32 logits).
#include <cfloat>

#include "alsd.h"
#include "common.cuh"
#include "kernels.h"
#include "rnnt_cell.cuh"

namespace rs {

namespace {

constexpr int kMaxBeam = 8;

// ---------------------------------------------------------------------------------------------- joint rows
// grid (B * beam), block 128.  Row r = b * beam + k.  Dead rows (hypothesis absent, or past the last frame) are zero-filled:
// their logits are never read.
__global__ void __launch_bounds__(128)
alsd_rows_kernel(const AlsdState st, const float* __restrict__ enc_proj, const int32_t* __restrict__ enc_len, int T_max, int Hj,
                 int step, __nv_bfloat16* __restrict__ planes) {
  const int r = blockIdx.x, b = r / st.beam, k = r % st.beam;
  const int n_h = st.n_hyp[b];
  const int T = enc_len[b];
  int t = -1;
  if (!st.done[b] && k < n_h) {
    t = step - st.u[r];
    if (t > T - 1) t = -1;
  }
  if (threadIdx.x == 0) st.row_t[r] = t;
  __nv_bfloat16* row = planes + static_cast<size_t>(r) * 3 * Hj;
  const float* ep = enc_proj + (static_cast<size_t>(b) * T_max + (t >= 0 ? t : 0)) * Hj;
  const float* pp = st.pp + static_cast<size_t>(r) * Hj;
  for (int j = threadIdx.x; j < Hj; j += blockDim.x) {
    const float x = t >= 0 ? fmaxf(ep[j] + pp[j], 0.f) : 0.f;
    __nv_bfloat16 h, m, l;
    split3(x, h, m, l);
    row[j] = h; row[Hj + j] = m; row[2 * Hj + j] = l;
  }
}

// ---------------------------------------------------------------------------------------------- per-row reductions
// grid (B * beam), block 256: log-sum-exp over the V + 1 classes, log p(blank), the `beam` largest non-blank log-probabilities
// (ties -> lower class index).
__global__ void __launch_bounds__(256)
alsd_reduce_kernel(const AlsdState st, const float* __restrict__ logits, int ld, int V) {
  const int r = blockIdx.x;
  if (st.row_t[r] < 0) return;
  __shared__ float s_red[8];
  __shared__ float s_val[8];
  __shared__ int s_idx[8];
  const float* x = logits + static_cast<size_t>(r) * ld;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int NC = V + 1;
  float mx = -FLT_MAX;
  for (int j = tid; j < NC; j += 256) mx = fmaxf(mx, x[j]);
  mx = warp_max(mx);
  if (lane == 0) s_red[warp] = mx;
  __syncthreads();
  mx = s_red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, s_red[w]);
  __syncthreads();
  float se = 0.f;
  for (int j = tid; j < NC; j += 256) se += expf(x[j] - mx);
  se = warp_sum(se);
  if (lane == 0) s_red[warp] = se;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) tot += s_red[w];
  const float lse = mx + logf(tot);
  if (tid == 0) st.cand_logp[r * (kMaxBeam + 1)] = x[V] - lse;            // blank
  // top-`beam` non-blank classes: `beam` rounds of (max, lowest index), each round excluding what was taken before
  float prev_v = FLT_MAX;
  int prev_i = -1;
  for (int round = 0; round < st.beam; ++round) {
    float bv = -FLT_MAX;
    int bi = 0x7fffffff;
    for (int j = tid; j < V; j += 256) {
      const float v = x[j];
      const bool after = v < prev_v || (v == prev_v && j > prev_i);        // strictly after the previous pick in (value desc, index asc) order
      if (after && (v > bv || (v == bv && j < bi))) { bv = v; bi = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    __syncthreads();
    if (lane == 0) { s_val[warp] = bv; s_idx[warp] = bi; }
    __syncthreads();
    bv = s_val[0]; bi = s_idx[0];
#pragma unroll
    for (int w = 1; w < 8; ++w)
      if (s_val[w] > bv || (s_val[w] == bv && s_idx[w] < bi)) { bv = s_val[w]; bi = s_idx[w]; }
    if (tid == 0) {
      st.cand_logp[r * (kMaxBeam + 1) + 1 + round] = bv - lse;
      st.cand_tok[r * kMaxBeam + round] = bi;
    }
    prev_v = bv; prev_i = bi;
  }
}

// ---------------------------------------------------------------------------------------------- beam update
__device__ __forceinline__ double logaddexp(double a, double b) {
  const double hi = a > b ? a : b, lo = a > b ? b : a;
  return hi + log1p(exp(lo - hi));
}

// grid (B), block 32 (lane 0 does the serial work: at most beam * (beam + 1) <= 72 candidates).
__global__ void __launch_bounds__(32)
alsd_select_kernel(const AlsdState st, const int32_t* __restrict__ enc_len, int step, int blank, float u_max_ratio, int recombine_returns_input) {
  const int b = blockIdx.x;
  if (threadIdx.x != 0 || st.done[b]) return;
  const int K = st.beam;
  const int T = enc_len[b];
  const int u_max = static_cast<int>(u_max_ratio * static_cast<float>(T));
  if (step >= T + u_max) {                             // the loop of the reference ends here whether or not hypotheses remain
    st.done[b] = 1;
    atomicAdd(st.n_done, 1);
    return;
  }
  // A in the reference's order: for every live hypothesis of B: [stay, extension 0 .. K-1]
  double a_score[kMaxBeam * (kMaxBeam + 1)];
  int a_par[kMaxBeam * (kMaxBeam + 1)], a_tok[kMaxBeam * (kMaxBeam + 1)];
  int n_a = 0;
  const int n_h = st.n_hyp[b];
  for (int k = 0; k < n_h; ++k) {
    const int r = b * K + k;
    const int t = st.row_t[r];
    if (t < 0) continue;                               // past the last frame: dropped (it entered `final` when it got there)
    const double s0 = st.score[r];
    const double stay = s0 + static_cast<double>(st.cand_logp[r * (kMaxBeam + 1)]);
    a_score[n_a] = stay; a_par[n_a] = k; a_tok[n_a] = -1; ++n_a;
    if (t == T - 1) {                                  // finished hypothesis: keep the best by score / len(y) (score_norm), first one on ties
      const double key = st.score_norm ? stay / static_cast<double>(st.u[r] + 1) : stay;
      if (!st.has_final[b] || key > st.final_key[b]) {
        st.has_final[b] = 1; st.final_key[b] = key; st.final_score[b] = stay; st.final_node[b] = st.node[r]; st.final_u[b] = st.u[r];
      }
    }
    for (int c = 0; c < K; ++c) {
      a_score[n_a] = s0 + static_cast<double>(st.cand_logp[r * (kMaxBeam + 1) + 1 + c]);
      a_par[n_a] = k; a_tok[n_a] = st.cand_tok[r * kMaxBeam + c]; ++n_a;
    }
  }
  if (n_a == 0) {                                      // every hypothesis has left the lattice: the reference breaks out of its loop
    st.done[b] = 1;
    atomicAdd(st.n_done, 1);
    return;
  }
  // the K best of A by score, stable
  int pick[kMaxBeam];
  bool used[kMaxBeam * (kMaxBeam + 1)];
  for (int i = 0; i < n_a; ++i) used[i] = false;
  const int n_new = n_a < K ? n_a : K;
  for (int j = 0; j < n_new; ++j) {
    int best = -1;
    for (int i = 0; i < n_a; ++i)
      if (!used[i] && (best < 0 || a_score[i] > a_score[best])) best = i;
    used[best] = true;
    pick[j] = best;
  }
  // new beam (written to the `next` half; the commit kernel swaps)
  double n_score[kMaxBeam];
  unsigned long long n_hash[kMaxBeam];
  int n_len[kMaxBeam];
  for (int j = 0; j < n_new; ++j) {
    const int a = pick[j], pk = a_par[a], pr = b * K + pk;
    n_score[j] = a_score[a];
    n_hash[j] = a_tok[a] >= 0 ? st.hash[pr] * 1000003ull + static_cast<unsigned long long>(a_tok[a] + 1) : st.hash[pr];
    n_len[j] = st.u[pr] + (a_tok[a] >= 0 ? 1 : 0);
  }
  // NeMo's recombine_hypotheses: the score of a later duplicate is added (logaddexp) into the first occurrence; as recalled, the
  // reference then returns its INPUT list, duplicates included (oracle/alsd_restated.py `recombine_returns_input`)
  bool dropped[kMaxBeam];
  for (int j = 0; j < n_new; ++j) dropped[j] = false;
  for (int j = 1; j < n_new; ++j)
    for (int f = 0; f < j; ++f)
      if (!dropped[f] && n_hash[f] == n_hash[j] && n_len[f] == n_len[j]) {        // equal token sequences (64-bit sequence hash + length)
        n_score[f] = logaddexp(n_score[f], n_score[j]);
        if (!recombine_returns_input) dropped[j] = true;
        break;
      }
  int w = 0;
  for (int j = 0; j < n_new; ++j) {
    if (dropped[j]) continue;
    const int a = pick[j], pk = a_par[a], pr = b * K + pk, nr = b * K + w;
    st.nx_score[nr] = n_score[j];
    st.nx_hash[nr] = n_hash[j];
    st.nx_parent[nr] = pk;
    st.nx_tok[nr] = a_tok[a];
    if (a_tok[a] >= 0) {                               // extension: one more token, emitted at alignment step `step`
      st.nx_u[nr] = st.u[pr] + 1;
      const int node = st.n_nodes[b]++;
      st.node_parent[static_cast<size_t>(b) * st.max_nodes + node] = st.node[pr];
      st.node_tok[static_cast<size_t>(b) * st.max_nodes + node] = a_tok[a];
      st.node_step[static_cast<size_t>(b) * st.max_nodes + node] = step;
      st.nx_node[nr] = node;
    } else {
      st.nx_u[nr] = st.u[pr];
      st.nx_node[nr] = st.node[pr];
    }
    ++w;
  }
  st.nx_n_hyp[b] = w;
  (void)blank;
}

// ---------------------------------------------------------------------------------------------- predictor of the extensions
// grid (B * beam), block 128: rows of the NEXT beam.  Extended hypotheses get [embed[token] | h_parent] as three bf16 planes
// (K = 2 * Hp per plane); kept ones (and absent rows) get zeros and are skipped by the cell kernel.
__global__ void __launch_bounds__(128)
alsd_lstm_in_kernel(const AlsdState st, const float* __restrict__ embed, int Hp, __nv_bfloat16* __restrict__ planes) {
  const int r = blockIdx.x, b = r / st.beam, k = r % st.beam;
  const bool ext = !st.done[b] && k < st.nx_n_hyp[b] && st.nx_tok[r] >= 0;
  __nv_bfloat16* row = planes + static_cast<size_t>(r) * 6 * Hp;
  const float* e = embed + static_cast<size_t>(ext ? st.nx_tok[r] : 0) * Hp;
  const float* h = st.h + (static_cast<size_t>(b) * st.beam + (ext ? st.nx_parent[r] : 0)) * Hp;
  for (int j = threadIdx.x; j < 2 * Hp; j += blockDim.x) {
    const float x = ext ? (j < Hp ? e[j] : h[j - Hp]) : 0.f;
    __nv_bfloat16 hi, mid, lo;
    split3(x, hi, mid, lo);
    row[j] = hi; row[2 * Hp + j] = mid; row[4 * Hp + j] = lo;
  }
}

// grid (B * beam), block 128: LSTM cell (gate order i, f, g, o; biases already in `gates`), new state into the `next` half;
// h as three bf16 planes for joint.pred.  Kept hypotheses copy (h, c) from their parent; their pred_proj is copied at commit.
__global__ void __launch_bounds__(128)
alsd_cell_kernel(const AlsdState st, const float* __restrict__ gates, int Hp, __nv_bfloat16* __restrict__ planes) {
  const int r = blockIdx.x, b = r / st.beam, k = r % st.beam;
  const bool live = !st.done[b] && k < st.nx_n_hyp[b];
  const bool ext = live && st.nx_tok[r] >= 0;
  const size_t pr = static_cast<size_t>(b) * st.beam + (live ? st.nx_parent[r] : 0);
  const float* g = gates + static_cast<size_t>(r) * 4 * Hp;
  __nv_bfloat16* row = planes + static_cast<size_t>(r) * 3 * Hp;
  for (int j = threadIdx.x; j < Hp; j += blockDim.x) {
    float h2 = 0.f, c2 = 0.f;
    if (ext) {
      lstm_cell(g[j], g[Hp + j], g[2 * Hp + j], g[3 * Hp + j], st.c[pr * Hp + j], h2, c2);
    } else if (live) {
      h2 = st.h[pr * Hp + j]; c2 = st.c[pr * Hp + j];
    }
    st.nx_h[static_cast<size_t>(r) * Hp + j] = h2;
    st.nx_c[static_cast<size_t>(r) * Hp + j] = c2;
    __nv_bfloat16 hi, mid, lo;
    split3(ext ? h2 : 0.f, hi, mid, lo);
    row[j] = hi; row[Hp + j] = mid; row[2 * Hp + j] = lo;
  }
}

// grid (B * beam), block 128: the next beam becomes current.  pred_proj: the GEMM's row for extended hypotheses, the parent's for
// kept ones (read from the current half before it is overwritten: every CTA reads its parent row first, then all write after a
// grid-wide ordering provided by running this in two launches: phase 0 stages into nx_pp, phase 1 copies nx_* over the current).
__global__ void __launch_bounds__(128)
alsd_commit_kernel(const AlsdState st, const float* __restrict__ pp_new, int Hp, int Hj, int phase) {
  const int r = blockIdx.x, b = r / st.beam, k = r % st.beam;
  if (st.done[b]) return;
  const bool live = k < st.nx_n_hyp[b];
  if (phase == 0) {
    if (!live) return;
    const bool ext = st.nx_tok[r] >= 0;
    const float* src = ext ? pp_new + static_cast<size_t>(r) * Hj : st.pp + (static_cast<size_t>(b) * st.beam + st.nx_parent[r]) * Hj;
    for (int j = threadIdx.x; j < Hj; j += blockDim.x) st.nx_pp[static_cast<size_t>(r) * Hj + j] = src[j];
    return;
  }
  if (live) {
    for (int j = threadIdx.x; j < Hj; j += blockDim.x) st.pp[static_cast<size_t>(r) * Hj + j] = st.nx_pp[static_cast<size_t>(r) * Hj + j];
    for (int j = threadIdx.x; j < Hp; j += blockDim.x) {
      st.h[static_cast<size_t>(r) * Hp + j] = st.nx_h[static_cast<size_t>(r) * Hp + j];
      st.c[static_cast<size_t>(r) * Hp + j] = st.nx_c[static_cast<size_t>(r) * Hp + j];
    }
  }
  if (threadIdx.x == 0) {
    if (live) {
      st.score[r] = st.nx_score[r]; st.hash[r] = st.nx_hash[r]; st.u[r] = st.nx_u[r]; st.node[r] = st.nx_node[r];
    }
    if (k == 0) st.n_hyp[b] = st.nx_n_hyp[b];
  }
}

// grid (B), block 32: initial beam = one hypothesis [blank] with score 0 (its predictor state is computed by one pass of the
// lstm_in / cell / commit kernels with nx_tok = blank -> the zero embedding)
__global__ void alsd_init_kernel(const AlsdState st, int blank) {
  const int b = blockIdx.x;
  if (threadIdx.x != 0) return;
  const int K = st.beam;
  st.done[b] = 0; st.has_final[b] = 0; st.n_hyp[b] = 0; st.nx_n_hyp[b] = 1; st.n_nodes[b] = 1;
  st.node_parent[static_cast<size_t>(b) * st.max_nodes] = -1;
  st.node_tok[static_cast<size_t>(b) * st.max_nodes] = blank;
  st.node_step[static_cast<size_t>(b) * st.max_nodes] = -1;
  for (int k = 0; k < K; ++k) { st.u[b * K + k] = 0; st.nx_tok[b * K + k] = -1; st.nx_parent[b * K + k] = 0; }
  const int r = b * K;
  st.nx_score[r] = 0.0; st.nx_hash[r] = 1469598103934665603ull; st.nx_u[r] = 0; st.nx_node[r] = 0; st.nx_tok[r] = blank; st.nx_parent[r] = 0;
  if (b == 0) *st.n_done = 0;
}

// grid (B), block 32: walk the back-pointers of the winning hypothesis (best finished one; with none, the best of the last
// beam by the same key) and write y_sequence (leading blank) and the alignment steps of its tokens.
__global__ void alsd_output_kernel(const AlsdState st, int blank, int32_t* __restrict__ y_out, int32_t* __restrict__ step_out,
                                   int32_t* __restrict__ n_out, double* __restrict__ score_out, int U_cap) {
  const int b = blockIdx.x;
  if (threadIdx.x != 0) return;
  int node, u;
  double score;
  if (st.has_final[b]) { node = st.final_node[b]; u = st.final_u[b]; score = st.final_score[b]; }
  else {
    int best = 0;
    double bk = -DBL_MAX;
    for (int k = 0; k < st.n_hyp[b]; ++k) {
      const int r = b * st.beam + k;
      const double key = st.score_norm ? st.score[r] / static_cast<double>(st.u[r] + 1) : st.score[r];
      if (key > bk) { bk = key; best = k; }
    }
    const int r = b * st.beam + best;
    node = st.node[r]; u = st.u[r]; score = st.score[r];
  }
  n_out[b] = u;
  score_out[b] = score;
  y_out[static_cast<size_t>(b) * (U_cap + 1)] = blank;
  int pos = u;
  while (node > 0 && pos > 0) {
    if (pos <= U_cap) {
      y_out[static_cast<size_t>(b) * (U_cap + 1) + pos] = st.node_tok[static_cast<size_t>(b) * st.max_nodes + node];
      step_out[static_cast<size_t>(b) * U_cap + pos - 1] = st.node_step[static_cast<size_t>(b) * st.max_nodes + node];
    }
    node = st.node_parent[static_cast<size_t>(b) * st.max_nodes + node];
    --pos;
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------ host side
size_t alsd_state_bytes(int B, int beam, int Hp, int Hj, int max_nodes) {
  const size_t R = static_cast<size_t>(B) * beam;
  size_t n = 0;
  auto add = [&](size_t bytes) { n = (n + 255) & ~static_cast<size_t>(255); n += bytes; };
  for (int i = 0; i < 2; ++i) { add(R * 8); add(R * 8); add(R * 4); add(R * 4); }          // score, hash, u, node (cur + next)
  add(R * 4); add(R * 4); add(R * 4);                                                       // nx_parent, nx_tok, row_t
  for (int i = 0; i < 2; ++i) { add(R * Hp * 4); add(R * Hp * 4); add(R * Hj * 4); }        // h, c, pp (cur + next)
  add(R * (kMaxBeam + 1) * 4); add(R * kMaxBeam * 4);                                       // candidates
  add(static_cast<size_t>(B) * 4 * 8);                                                      // n_hyp, nx_n_hyp, done, has_final, n_nodes, final_node, final_u (+pad)
  add(static_cast<size_t>(B) * 8 * 2);                                                      // final_key, final_score
  add(static_cast<size_t>(B) * max_nodes * 4 * 3);                                          // node tree
  add(256);                                                                                 // n_done
  return n + 256;
}

void alsd_bind_state(AlsdState& st, void* base, int B, int beam, int Hp, int Hj, int max_nodes, bool score_norm) {
  const size_t R = static_cast<size_t>(B) * beam;
  char* p = static_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) { off = (off + 255) & ~static_cast<size_t>(255); char* q = p + off; off += bytes; return q; };
  st.beam = beam; st.max_nodes = max_nodes; st.score_norm = score_norm ? 1 : 0;
  st.score = reinterpret_cast<double*>(take(R * 8)); st.hash = reinterpret_cast<unsigned long long*>(take(R * 8));
  st.u = reinterpret_cast<int*>(take(R * 4)); st.node = reinterpret_cast<int*>(take(R * 4));
  st.nx_score = reinterpret_cast<double*>(take(R * 8)); st.nx_hash = reinterpret_cast<unsigned long long*>(take(R * 8));
  st.nx_u = reinterpret_cast<int*>(take(R * 4)); st.nx_node = reinterpret_cast<int*>(take(R * 4));
  st.nx_parent = reinterpret_cast<int*>(take(R * 4)); st.nx_tok = reinterpret_cast<int*>(take(R * 4)); st.row_t = reinterpret_cast<int*>(take(R * 4));
  st.h = reinterpret_cast<float*>(take(R * Hp * 4)); st.c = reinterpret_cast<float*>(take(R * Hp * 4)); st.pp = reinterpret_cast<float*>(take(R * Hj * 4));
  st.nx_h = reinterpret_cast<float*>(take(R * Hp * 4)); st.nx_c = reinterpret_cast<float*>(take(R * Hp * 4)); st.nx_pp = reinterpret_cast<float*>(take(R * Hj * 4));
  st.cand_logp = reinterpret_cast<float*>(take(R * (kMaxBeam + 1) * 4)); st.cand_tok = reinterpret_cast<int*>(take(R * kMaxBeam * 4));
  int* ints = reinterpret_cast<int*>(take(static_cast<size_t>(B) * 4 * 8));
  st.n_hyp = ints; st.nx_n_hyp = ints + B; st.done = ints + 2 * B; st.has_final = ints + 3 * B; st.n_nodes = ints + 4 * B;
  st.final_node = ints + 5 * B; st.final_u = ints + 6 * B;
  double* dbl = reinterpret_cast<double*>(take(static_cast<size_t>(B) * 8 * 2));
  st.final_key = dbl; st.final_score = dbl + B;
  int* tree = reinterpret_cast<int*>(take(static_cast<size_t>(B) * max_nodes * 4 * 3));
  st.node_parent = tree; st.node_tok = tree + static_cast<size_t>(B) * max_nodes; st.node_step = tree + 2 * static_cast<size_t>(B) * max_nodes;
  st.n_done = reinterpret_cast<int*>(take(256));
}

cudaError_t alsd_launch_init(const AlsdState& st, int B, int blank, cudaStream_t s) {
  alsd_init_kernel<<<B, 32, 0, s>>>(st, blank);
  return cudaGetLastError();
}
cudaError_t alsd_launch_rows(const AlsdState& st, int B, const float* enc_proj, const int32_t* enc_len, int T_max, int Hj, int step, void* planes, cudaStream_t s) {
  alsd_rows_kernel<<<B * st.beam, 128, 0, s>>>(st, enc_proj, enc_len, T_max, Hj, step, static_cast<__nv_bfloat16*>(planes));
  return cudaGetLastError();
}
cudaError_t alsd_launch_reduce(const AlsdState& st, int B, const float* logits, int ld, int V, cudaStream_t s) {
  alsd_reduce_kernel<<<B * st.beam, 256, 0, s>>>(st, logits, ld, V);
  return cudaGetLastError();
}
cudaError_t alsd_launch_select(const AlsdState& st, int B, const int32_t* enc_len, int step, int blank, float u_max_ratio, bool recombine_returns_input, cudaStream_t s) {
  alsd_select_kernel<<<B, 32, 0, s>>>(st, enc_len, step, blank, u_max_ratio, recombine_returns_input ? 1 : 0);
  return cudaGetLastError();
}
cudaError_t alsd_launch_lstm_in(const AlsdState& st, int B, const float* embed, int Hp, void* planes, cudaStream_t s) {
  alsd_lstm_in_kernel<<<B * st.beam, 128, 0, s>>>(st, embed, Hp, static_cast<__nv_bfloat16*>(planes));
  return cudaGetLastError();
}
cudaError_t alsd_launch_cell(const AlsdState& st, int B, const float* gates, int Hp, void* planes, cudaStream_t s) {
  alsd_cell_kernel<<<B * st.beam, 128, 0, s>>>(st, gates, Hp, static_cast<__nv_bfloat16*>(planes));
  return cudaGetLastError();
}
cudaError_t alsd_launch_commit(const AlsdState& st, int B, const float* pp_new, int Hp, int Hj, cudaStream_t s) {
  alsd_commit_kernel<<<B * st.beam, 128, 0, s>>>(st, pp_new, Hp, Hj, 0);
  alsd_commit_kernel<<<B * st.beam, 128, 0, s>>>(st, pp_new, Hp, Hj, 1);
  return cudaGetLastError();
}
cudaError_t alsd_launch_output(const AlsdState& st, int B, int blank, int32_t* y, int32_t* steps, int32_t* n, double* score, int U_cap, cudaStream_t s) {
  alsd_output_kernel<<<B, 32, 0, s>>>(st, blank, y, steps, n, score, U_cap);
  return cudaGetLastError();
}

}  // namespace rs
