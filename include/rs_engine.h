/*
 * rs_engine.h -- C ABI of the B200-native FastConformer-RNNT engine.
 *
 * The reference (reazon-research/ReazonSpeech) has no native layer: its hot path is one
 * opaque Python call into NeMo,
 *     model.transcribe([waveform], batch_size=1, return_hypotheses=True, verbose=...)
 *                                              pkg/nemo-asr/src/transcribe.py:48-53
 * whose result is consumed as hyp.y_sequence / hyp.timestamp (pkg/nemo-asr/src/decode.py:40,44).
 * This header is the boundary a binding for that call site would target (INTEGRATION.md shows
 * the ctypes stub).  Each entry point names the NeMo stage it replaces (SURVEY.md section 8a).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - every function returns RS_OK (0) or a negative rs_status; rs_last_error() gives the text.
 *   - "dev" pointers are CUDA device pointers on the engine's device, caller-allocated unless
 *     stated; "host" pointers are host memory (pinned for best throughput).
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden synchronisation
 *     except where stated (rs_transcribe_batch synchronises before returning).
 *   - an engine is bound to one device and is not re-entrant; distinct engines are independent.
 *   - batched activations are padded row-major [B, T_max, ...] with a per-utterance length
 *     vector; rows at or beyond an utterance's length never influence valid rows.
 */
#ifndef RS_ENGINE_H_
#define RS_ENGINE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum rs_status {
  RS_OK = 0,
  RS_ERR_INVALID_ARG = -1,
  RS_ERR_CUDA = -2,
  RS_ERR_MISSING_WEIGHT = -3,
  RS_ERR_WORKSPACE = -4,
  RS_ERR_UNSUPPORTED = -5
} rs_status;

/* Mirrors the fields of the .nemo model_config.yaml the path consumes (SURVEY.md App. A.1). */
typedef struct rs_model_config {
  int32_t sample_rate, n_window_size, n_window_stride, n_fft, n_mels;
  float preemph, log_zero_guard, norm_eps;
  int32_t n_layers, d_model, n_heads, d_ff, conv_kernel, sub_channels;
  int32_t att_left, att_right, global_tokens;
  float xscale, ln_eps;
  int32_t vocab_size;   /* blank id == vocab_size; classes == vocab_size + 1 */
  int32_t pred_hidden, joint_hidden, max_symbols;
} rs_model_config;

/* One packed weight tensor, resident on the device (packing: reazonspeech_b200/engine.py::pack_weights is the definition of
 * the names, shapes and value transforms -- e.g. "pred.gate_tab" f32 [V+1, 4*pred_hidden] = W_ih . embed[k] + b_ih + b_hh,
 * the per-token input half of the LSTM gates; rs_engine_create names the first tensor it misses in rs_last_error). */
typedef enum rs_dtype { RS_F32 = 0, RS_BF16 = 1, RS_I32 = 2 } rs_dtype;
typedef struct rs_tensor {
  const char* name;
  const void* dev_ptr;
  int32_t dtype;     /* rs_dtype */
  int64_t numel;
} rs_tensor;

typedef struct rs_engine rs_engine;

/* Epilogues of the tcgen05 GEMM  out = epi(A[M,K] * W[N,K]^T)  (SURVEY.md App. A.3). */
typedef enum rs_epilogue {
  RS_EPI_BIAS_BF16 = 0,       /* out_bf16[M,N]   = acc + bias                                  */
  RS_EPI_BIAS_RELU_BF16 = 1,  /* out_bf16[M,N]   = relu(acc + bias)                            */
  RS_EPI_BIAS_SWISH_BF16 = 2, /* out_bf16[M,N]   = swish(acc + bias)                           */
  RS_EPI_BIAS_GLU_BF16 = 3,   /* out_bf16[M,N/2] = a * sigmoid(g); W rows interleaved 16/16    */
  RS_EPI_RESID_F32 = 4,       /* out_f32[M,N]    = resid + alpha * (acc + bias)  (may alias: with out == resid and
                                 N % 256 == 0 the add is a TMA reduce-add performed by the memory system -- the residual is never
                                 read into the SM; same fp32 sum, bit-identical to the two-buffer form)   */
  RS_EPI_BIAS_F32 = 5,        /* out_f32[M,N]    = alpha * (acc + bias)                        */
  RS_EPI_BIAS_F16 = 6,        /* out_f16[M,N]    = acc + bias  (IEEE half)                          */
  RS_EPI_QKV_VT = 7           /* fused QKV projection: columns [0, split) -> out_bf16[M, ldo] as RS_EPI_BIAS_BF16,
                                 columns [split, N) -> TRANSPOSED into out2_bf16[N - split, ld2] (V^T, keys contiguous:
                                 the K-major B operand of the attention kernel's P.V product)               */
} rs_epilogue;

/* ---- lifetime -------------------------------------------------------------------------- */
/* Replaces EncDecRNNTBPEModel.from_pretrained (transcribe.py:26-28) below the Python loader. */
int rs_engine_create(const rs_model_config* cfg, const rs_tensor* weights, int n_weights,
                     int device, rs_engine** out);
void rs_engine_destroy(rs_engine* e);
/* Text of the last failure on `e` (or of the last failed rs_engine_create when e == NULL). */
const char* rs_last_error(const rs_engine* e);

/* Scratch the engine needs for a batch of B utterances of at most L_max samples. */
int rs_workspace_bytes(const rs_engine* e, int B, int L_max, size_t* bytes);
int rs_set_workspace(rs_engine* e, void* dev_ptr, size_t bytes);

/* ---- shape arithmetic --------------------------------------------------------------------
 * rs_mel_frames / rs_enc_frames: TENSOR time sizes for a buffer of n_samples (frames of the centred
 * STFT = n/hop + 1; ConvSubsampling.calc_length applied to it three times, rounded up to a multiple of 8):
 * what callers allocate.
 * rs_mel_valid / rs_enc_valid: the VALID lengths of an utterance of n_samples
 * (FilterbankFeatures.get_seq_len = n/hop, then calc_length x3): what mel_len / enc_len will hold. */
int rs_mel_frames(const rs_engine* e, int n_samples);
int rs_enc_frames(const rs_engine* e, int n_samples);
int rs_mel_valid(const rs_engine* e, int n_samples);
int rs_enc_valid(const rs_engine* e, int n_samples);

/* ---- stages (each is also a parity-test seam) --------------------------------------------- */
/* N1 AudioToMelSpectrogramPreprocessor: wav f32[B,L_max] + len -> mel f32[B,F_max,n_mels]
 * (time-major, per-feature normalised, rows >= mel_len zero) + mel_len i32[B].  Needs the workspace
 * (rs_set_workspace) for the per-feature statistics.  On the fused paths below the features stay
 * un-normalised in the workspace and the normalisation is applied by the first subsampling kernel's load. */
int rs_logmel(rs_engine* e, const float* wav_dev, const int32_t* len_dev, int B, int L_max,
              float* mel_dev, int32_t* mel_len_dev, void* stream);
/* N2-N7 ConformerEncoder: mel -> enc f32[B,T_max,d_model] + enc_len i32[B].
 * n_layers < 0 runs the configured depth (smaller values are for stage tests). */
int rs_encode(rs_engine* e, const float* mel_dev, const int32_t* mel_len_dev, int B, int F_max,
              float* enc_dev, int32_t* enc_len_dev, int n_layers, void* stream);
/* N8-N9 RNNTDecoder + RNNTJoint + greedy loop: enc -> tokens/frames i32[B,U_max], n_tok i32[B].
 * n_tok[b] is the true emission count (may exceed U_max; only U_max entries are stored). */
int rs_rnnt_greedy(rs_engine* e, const float* enc_dev, const int32_t* enc_len_dev, int B,
                   int T_max, int32_t* tokens_dev, int32_t* frames_dev, int32_t* n_tok_dev,
                   int U_max, void* stream);
/* Device-resident whole path (what bench.py's `value` times). */
int rs_transcribe_device(rs_engine* e, const float* wav_dev, const int32_t* len_dev, int B,
                         int L_max, int32_t* tokens_dev, int32_t* frames_dev, int32_t* n_tok_dev,
                         int U_max, void* stream);
/* The model.transcribe seam with HOST buffers: H2D + whole path + D2H; synchronises. */
int rs_transcribe_batch(rs_engine* e, const float* wav_host, const int32_t* len_host, int B,
                        int L_max, int32_t* tokens_host, int32_t* frames_host,
                        int32_t* n_tok_host, int U_max, void* stream);
/* The same two entry points for 16-bit PCM (what audio files hold): samples are scaled by 2^-15 inside the
 * log-mel kernel's staging load -- the value decoding a 16-bit WAV to float32 gives (the reference loads files
 * through librosa.load, pkg/nemo-asr/src/audio.py:32-42) -- so the results equal the float entry points' on
 * the converted samples, for half the host-to-device and HBM bytes.  L_max must be a multiple of 4 for the
 * vectorised load (any value works, unaligned rows fall back to scalar loads). */
int rs_transcribe_device_pcm16(rs_engine* e, const int16_t* wav_dev, const int32_t* len_dev, int B,
                               int L_max, int32_t* tokens_dev, int32_t* frames_dev,
                               int32_t* n_tok_dev, int U_max, void* stream);
int rs_transcribe_batch_pcm16(rs_engine* e, const int16_t* wav_host, const int32_t* len_host, int B,
                              int L_max, int32_t* tokens_host, int32_t* frames_host,
                              int32_t* n_tok_host, int U_max, void* stream);

/* ALSD beam search (NeMo BeamRNNTInfer.align_length_sync_decoding, the shipped checkpoint's default strategy; the reference's
 * decode.py is written for its hypotheses, pkg/nemo-asr/src/decode.py:29,38-40,48): enc f32[B,T_max,d_model] + enc_len ->
 * y i32[B, U_cap + 1] (leading blank, then the tokens), step i32[B, U_cap] (alignment step t + u of every token =
 * Hypothesis.timestamp after NeMo's pack_hypotheses), n i32[B] tokens, score f64[B] (log-probability of the winner).
 * beam 1..8; u_max_ratio = alsd_max_target_len (NeMo: 2.0); score_norm: rank finished hypotheses by score / len(y);
 * recombine_returns_input: NeMo's recombine_hypotheses as recalled (adds duplicate scores, keeps the duplicates).
 * Needs the "alsd.*" weight tensors at rs_engine_create.  Synchronises before returning. */
int rs_rnnt_alsd(rs_engine* e, const float* enc_dev, const int32_t* enc_len_dev, int B, int T_max, int beam,
                 float u_max_ratio, int score_norm, int recombine_returns_input, int32_t* y_dev, int32_t* step_dev,
                 int32_t* n_dev, double* score_dev, int U_cap, void* stream);

/* RNN-T forced alignment of given token sequences: enc f32[B,T_max,d_model] + enc_len, targets i32[B,U_max] (ids in
 * [0, vocab_size)) + tgt_len i32[B] -> frames i32[B,U_max] (emitting encoder frame of each token on the Viterbi path),
 * tok_logp f32[B,U_max], viterbi f64[B], loglik f64[B] (forward sum over all alignments = -RNN-T loss),
 * lattice f32[B,T_max,U_max+1,2] (nullable: log p(blank), log p(next target) per node; other entries unspecified).
 * Entries of frames / tok_logp at or beyond tgt_len[b] are -1 / 0.  enc_len[b] in [1, T_max], tgt_len[b] in [0, U_max],
 * U_max >= 1; a violated range, or a target outside [0, vocab_size), returns RS_ERR_INVALID_ARG before any computation.
 * Needs the "alsd.*" weight tensors (RS_ERR_UNSUPPORTED without them).  Synchronises before returning. */
int rs_rnnt_align(rs_engine* e, const float* enc_dev, const int32_t* enc_len_dev, int B, int T_max,
                  const int32_t* targets_dev, const int32_t* tgt_len_dev, int U_max,
                  int32_t* frames_dev, float* tok_logp_dev, double* viterbi_dev, double* loglik_dev,
                  float* lattice_dev, void* stream);

/* Free-span RNN-T alignment: find each of K known token sequences (captions) inside a frame window of one encoder row, as
 * when a broadcast caption is searched for in the audio around its display time.  enc f32[B,T_max,d_model] + enc_len i32[B];
 * span i32[K,3] = (src row, lo, hi): caption k lives somewhere in frames [lo, hi) of row src; targets i32[K,U_max] +
 * tgt_len i32[K].  The lattice of caption k is rs_rnnt_align's lattice of enc[src, lo:hi] (W = hi - lo frames).  The path may
 * start at any node (t, 0) at no cost and ends with the closing blank of any frame t_e at u = U:
 *   alpha(t, 0) = max(0, alpha(t-1, 0) + lb(t-1, 0)),   viterbi = max_t alpha(t, U) + lb(t, U),
 * and loglik is the same recursion with logaddexp (logsumexp over every (start, end) pair of rs_rnnt_align's loglik), all in
 * float64.  Ties: at u = 0 an exact tie goes to the fresh start, at the end to the earliest t_e, inside the lattice to the
 * blank edge (as rs_rnnt_align).  Every log p(blank) <= 0, so the best span is exactly [frames[0], frames[U-1]].
 * Outputs: frames i32[K,U_max] (ABSOLUTE encoder frame, lo + window frame, of each token on the best path; -1 past tgt_len),
 * tok_logp f32[K,U_max], path_logp f32[K,F_max] (indexed by window frame t - lo: lb(t, u_t) plus the log p of the tokens the
 * path emits at t, summed in fp32; 0 outside the span, and the span's entries sum to viterbi up to fp32 rounding),
 * viterbi f64[K], loglik f64[K], lattice f32[K,F_max,U_max+1,2] (nullable; other entries unspecified).
 * RS_ERR_INVALID_ARG before any computation when: enc_len[b] outside [0, T_max], src outside [0, B), lo < 0, lo >= hi,
 * hi > enc_len[src], tgt_len[k] outside [1, U_max], F_max < max(hi - lo), or a target outside [0, vocab_size).
 * joint.enc runs once over the B * T_max rows and the predictor once over the K captions.  Needs the "alsd.*" weight tensors
 * (RS_ERR_UNSUPPORTED without them).  Synchronises before returning. */
int rs_rnnt_align_spans(rs_engine* e, const float* enc_dev, const int32_t* enc_len_dev, int B, int T_max, int K,
                        const int32_t* span_dev, const int32_t* targets_dev, const int32_t* tgt_len_dev, int U_max,
                        int32_t* frames_dev, float* tok_logp_dev, float* path_logp_dev, int F_max, double* viterbi_dev,
                        double* loglik_dev, float* lattice_dev, void* stream);

/* norm_audio on the device (pkg/nemo-asr/src/audio.py:54-68: resample to 16 kHz, then average the channels) fused with
 * transcribe()'s padding (audio.py:70-83): in [B, channels, L_in_max] f32 or int16 PCM at the native rate ->
 * out f32 [B, L_out_row], row b = pad zeros | resampled mono utterance | zeros, len_out[b] = resampled length + 2 pad;
 * feed out / len_out to rs_transcribe_device.  The polyphase FIR (taps [up][taps_per_phase], n_pre_remove) is
 * scipy.signal.resample_poly's, designed by the host binding (reazonspeech_b200/engine.py::resample_taps). */
int rs_resample_mono(rs_engine* e, const void* in_dev, int in_is_pcm16, const int32_t* len_in_dev, int B,
                     int channels, int L_in_max, const float* taps_dev, int taps_per_phase, int up, int down,
                     int n_pre_remove, int pad, float* out_dev, int L_out_row, int32_t* len_out_dev, void* stream);

/* Host-side half of transcribe()'s padding (pkg/nemo-asr/src/audio.py:70-83) for a batch: row r of dst[B][L] (pinned host
 * memory the caller then hands to rs_transcribe_batch / _pcm16) = zeros(pad) | src[r][0 .. n[r]) | zeros to L.
 * dst_is_pcm16: rows are int16 and every source must be int16; otherwise rows are float32 and an int16 source
 * (src_is_pcm16[r] != 0; the array may be NULL = all float32) is scaled by 1/32768.  No engine, no CUDA call: plain
 * copies split over `threads` host threads, so a binding can stage a batch without holding its interpreter lock. */
int rs_stage_rows(void* dst, int64_t L, const void* const* src, const int64_t* n, const int32_t* src_is_pcm16,
                  int dst_is_pcm16, int B, int64_t pad, int threads);

/* ---- kernel-level seams (parity tests and roofline measurement) --------------------------- */
int rs_gemm_bf16(rs_engine* e, const void* a_bf16, const void* w_bf16, const float* bias,
                 const float* resid, void* out, int M, int N, int K, int epilogue, float alpha,
                 void* stream);
int rs_layernorm(rs_engine* e, const float* x, const float* gamma, const float* beta,
                 float* out_f32 /*nullable*/, void* out_bf16 /*nullable*/, int rows, int d,
                 void* stream);
/* Counters: kernels launched by this engine since creation (bench.py's gpu_launches). */
int64_t rs_launch_count(const rs_engine* e);
/* Per-stage device time of the last rs_transcribe_* call when timing was enabled: ms[0..4] = log-mel, subsampling,
 * conformer layers, f32->bf16 + joint.enc GEMM, greedy decode (ms[5..7] are zero).  Every entry point records the
 * stage marks.  The log-mel stage ends at the log-mel of the last utterance chunk, so for rs_transcribe_batch /
 * _pcm16 with chunked copies (B >= 16) it includes the host-to-device copies and the first subsampling conv of the
 * chunks before the last one, which overlap it. */
int rs_enable_stage_timing(rs_engine* e, int on);
int rs_stage_times_ms(const rs_engine* e, float* ms /*[8]*/);
int rs_debug_decode_cycles(rs_engine* e, int B, int L_max, int U_max, int64_t* out8);   /* profiling aid, see engine.cu */
int rs_debug_attention_cycles(rs_engine* e, int64_t* out16);   /* clock64 stamps of one CTA of the last attention launch */
int rs_debug_gemm_cycles(rs_engine* e, int64_t* out64);        /* clock64 timeline of the last 2-CTA GEMM launch: first / last cluster x 32 stamps (gemm_tcgen05.cu) */
/* Per-launch CUDA-event timing of the tcgen05 GEMM (the dominant kernel): while enabled every GEMM
 * launch is bracketed by two events on its stream.  rs_gemm_timing() synchronises, returns the summed
 * device time, the summed algorithmic FLOPs (2*M*N*K) and the launch count since it was enabled or
 * last read, and resets the accumulators. */
int rs_enable_gemm_timing(rs_engine* e, int on);
int rs_gemm_timing(rs_engine* e, double* ms, double* flops, int64_t* launches);
/* Per-kernel CUDA-event timing of EVERY launch inside the real pipeline (warm caches, back-to-back launches, unlike
 * the cold, serialised launches ncu reports).  rs_kernel_timing() synchronises the device and writes one line per
 * kernel name, "name<TAB>launches<TAB>total_ms", into buf; the log is reset. */
int rs_enable_kernel_timing(rs_engine* e, int on);
int rs_kernel_timing(rs_engine* e, char* buf, int buf_bytes);

#ifdef __cplusplus
}
#endif
#endif /* RS_ENGINE_H_ */
