// Host-side interface of the RNN-T forced-alignment kernels (align.cu); internal to librs_engine.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rs {

// Rows of one lattice chunk (a multiple of the 128-row tile): bounds the A planes at kAlignChunkRows * 3 * Hj bf16.
constexpr int kAlignChunkRows = 128 * 1024;

// bad |= 1 when a target of u < tgt_len[b] lies outside [0, V)
cudaError_t align_check(const int32_t* targets, const int32_t* tgt_len, int B, int U_max, int V, int* bad, cudaStream_t s);
// Teacher-forced predictor step k (0: the SOS step): LSTM cell on gates [B, 4Hp] -> h_k as three bf16 planes into row b * U1 + k
// of h_planes [B * U1, 3Hp]; the next step's input [embed[y_{k+1}] | h_k] as three planes into in_planes [B, 6Hp].
cudaError_t align_pred(const float* gates, float* c_state, const int32_t* targets, const int32_t* tgt_len, int B, int U_max, int U1,
                       int k, const float* embed, int Hp, void* in_planes, void* h_planes, cudaStream_t s);
// Rows [r0, r0 + n_rows) of the compact node list (item b owns [offs[b], offs[b + 1]), node t * (U_b + 1) + u):
// relu(enc_proj[row_base[b] + t] + pred_proj[b, u]) as three bf16 planes [n_rows, 3Hj], and the row's target column (-1 at
// u = U_b).  row_base[b] is b * T_max for a whole utterance, src * T_max + lo for the frame window [lo, hi) of row src.
cudaError_t align_rows(const float* enc_proj, const float* pred_proj, const int64_t* offs, const int64_t* row_base,
                       const int32_t* tgt_len, const int32_t* targets, int B, int U1, int U_max, int Hj, int64_t r0, int n_rows,
                       void* planes, int32_t* tcol, cudaStream_t s);
// Fused joint output layer + log-softmax over the rows of one chunk: out[r] = (log p(blank), log p(target column)).
cudaError_t align_lattice(const void* planes, const void* w3, const float* bias, const int32_t* tcol, float2* out, int n_rows,
                          int n_pad, int Hj, int V, int num_sms, cudaStream_t s, char* err);
// Viterbi + forward sweep of every item's lattice (one CTA each), backtrace, optional scatter of the lattice.  With span
// [B, 3] (src, lo, hi) non-null the path may start and end at any frame of the window: enc_len then holds hi - lo, T_max is
// the row pitch F_max of lattice and path_logp [B, F_max], and frames are lo + the window frame.
cudaError_t align_dp(const float2* lp, const int64_t* offs, const int32_t* enc_len, const int32_t* tgt_len, int B, int T_max,
                     int U_max, int U1, uint8_t* bp, int32_t* frames, float* tok_logp, double* viterbi, double* loglik, float* lattice,
                     const int32_t* span, float* path_logp, cudaStream_t s);
size_t align_dp_smem_bytes(int U1, bool span = false);

}  // namespace rs
