// Host-side launch interface of the sm_100a kernels (internal to librs_engine.so).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct CUtensorMap_st;

namespace rs {

struct GemmArgs {
  const void* a;       // bf16 [M,K] row-major
  const void* w;       // bf16 [N,K] row-major (nn.Linear layout)
  const float* bias;   // f32 [N] or nullptr
  const float* resid;  // f32 [M,N] for RS_EPI_RESID_F32
  void* out;
  int M, N, K;
  int epilogue;        // rs_epilogue
  float alpha;
  // RS_EPI_QKV_VT: columns >= split go, transposed, to out2 (bf16 [N - split, ld2]; ld2 >= M rounded up to 256)
  void* out2 = nullptr; int split = 0, ld2 = 0;
};

// Returns cudaSuccess or the failing CUDA error; err (>=256 B) receives a description.
cudaError_t launch_gemm(const GemmArgs& g, int num_sms, cudaStream_t stream, char* err);
// TMA descriptor of a bf16 row-major [rows, cols] operand (row pitch ld elements): (box_rows x 64) boxes, 128B swizzle,
// out-of-range rows zero-filled.  (CUtensorMap_st is cuda.h's CUtensorMap, named here without the driver API include.)
bool make_tmap_bf16(::CUtensorMap_st* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, char* err);
cudaError_t gemm_debug_cycles(long long* out64);   // timeline of the last 2-CTA launch (see g_gemm_prof)

cudaError_t launch_layernorm(const float* x, const float* gamma, const float* beta, float* out_f32,
                             void* out_bf16, const float* gamma2, const float* beta2, int rows, int d,
                             float eps, cudaStream_t stream);

struct SubsampleArgs {
  const float* mel; const int32_t* mel_len;   // un-normalised log-mel [B, F_max, n_mels] and valid frames
  const float* mel_stats;                     // [B, n_mels, 2] (mean, 1 / (std + eps)) from the log-mel kernel
  int B, F_max, n_mels, C;
  const float* w0; const float* b0;      // conv.0  [C,9], [C]
  const float* wd1; const float* bd1;    // conv.2  [C,9], [C]
  void* out1;                            // bf16 [B,T2,F2,C]
  int T1, F1, T2, F2;
};
cudaError_t launch_sub_conv0_dw1(const SubsampleArgs& a, cudaStream_t stream);
// depthwise 3x3 s2 on channels-last bf16 [B,Tin,Fin,C] (rows t >= len_in(b) read as zero)
cudaError_t launch_sub_dw(const void* in, void* out, const float* w, const float* b, const int32_t* mel_len,
                          int len_shift, int B, int Tin, int Fin, int Tout, int Fout, int C, cudaStream_t stream);

// GLU output u bf16 [B*T_max, d] -> depthwise conv (k taps, BN folded) -> swish -> bf16
cudaError_t launch_conv_dw(const void* u, void* out, const float* w /*[k,d]*/, const float* shift /*[d]*/,
                           const int32_t* enc_len, int B, int T_max, int d, int k, cudaStream_t stream);

struct AttnArgs {
  const void* qkv;       // bf16 [B*T_max, 3*d]: q + pos_bias_u | k | (unused; V goes to vt)
  const void* pos;       // bf16 [H, n_rel_pad, dk]: linear_pos(pos_emb) per head, rows beyond the 2w+1 offsets zero (packed at load)
  const float* bd_bias;  // f32 [H, n_rel_pad]: (pos_bias_v - pos_bias_u) . pos[h][c]
  int n_rel_pad;
  const float* bias_u;   // f32 [H, dk]
  void* out;             // bf16 [B*T_max, d]
  const int32_t* enc_len;
  int B, T_max, H, dk, w_left, w_right, n_global;
  const void* vt = nullptr; int ld_vt = 0;   // V^T bf16 [H*dk, ld_vt] written by the QKV GEMM (RS_EPI_QKV_VT)
};
bool attention_tc_supported(const AttnArgs& a);
cudaError_t launch_attention_tc(const AttnArgs& a, cudaStream_t stream);
cudaError_t attention_tc_debug_cycles(long long* out16);   // clock64 stamps of CTA (1,0,0) of the last launch

struct DecodeArgs {
  const float* enc_proj;      // f32 [B*T_max, Hj]  (joint.enc applied to every frame)
  const int32_t* enc_len;
  const void* w_out;          // bf16 [V+1, Hj]
  const float* b_out;         // f32 [V+1]
  const float* embed;         // f32 [V+1, Hp]
  const void* w_lstm;         // bf16 [4*Hp, 2*Hp]  (W_ih | W_hh, gate order i,f,g,o)
  const float* b_lstm;        // f32 [4*Hp]  (b_ih + b_hh)
  const float* gate_tab;      // f32 [V+1, 4*Hp]: W_ih . embed[k] + b_ih + b_hh (the input half of the gates, per token)
  const void* w_pred;         // bf16 [Hj, Hp]
  const float* b_pred;        // f32 [Hj]
  int32_t* tokens; int32_t* frames; int32_t* n_tok;
  int B, T_max, Hj, Hp, V, U_max, max_symbols;
};
// windowed (kFrames per iteration) persistent decode, joint on tcgen05 (decode_spec.cu); workspace from rnnt_spec_workspace_bytes()
size_t rnnt_spec_workspace_bytes(int B, int Hj, int Hp, int num_sms);
size_t rnnt_spec_prof_offset(int B, int Hj, int Hp);        // where the kernel's 12 cycle counters sit inside that workspace
cudaError_t launch_rnnt_greedy_spec(const DecodeArgs& a, void* workspace, int num_sms, cudaStream_t stream);

// norm_audio on the device: polyphase resampling to 16 kHz + channel average + transcribe()'s zero padding (resample.cu)
struct ResampleArgs {
  const void* in; bool in_i16;          // [B, C, L_in_max] f32, or int16 PCM (scaled by 2^-15)
  const int32_t* len_in;                // [B] valid samples per utterance (per channel)
  int B, C, L_in_max;
  const float* taps; int taps_per_phase, up, down, n_pre_remove;   // polyphase FIR from engine.py::resample_taps: taps[up][taps_per_phase]
  int pad;                              // zero samples in front of and behind every resampled utterance
  float* out; int L_out_row;            // [B, L_out_row] f32, fully written (zeros outside the utterance)
  int32_t* len_out;                     // [B] resampled length + 2 * pad
};
cudaError_t launch_resample_mono(const ResampleArgs& a, cudaStream_t stream);

// small utility kernels
cudaError_t launch_f32_to_bf16(const float* in, void* out, int64_t n, cudaStream_t stream);
cudaError_t launch_zero_pad_rows(float* x, const int32_t* len, int B, int T_max, int d, cudaStream_t stream);

}  // namespace rs
