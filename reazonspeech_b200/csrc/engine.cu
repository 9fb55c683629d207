// C ABI of the engine (include/rs_engine.h): weight table lookup, workspace planning and the
// launch sequence of the FastConformer-RNNT path.  Host-side orchestration only; every device
// operation is one of the sm_100a kernels declared in kernels.h.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/rs_engine.h"
#include "alsd.h"
#include "kernels.h"
#include "logmel.h"

namespace {

thread_local char g_create_error[512] = "";

// NVTX range around the ENQUEUE of a stage (SURVEY.md section 5: per-stage ranges for Nsight Systems / Compute).  Header-only
// NVTX v3: a no-op unless a tool has injected itself into the process.
struct Nvtx {
  explicit Nvtx(const char* name) { nvtxRangePushA(name); }
  ~Nvtx() { nvtxRangePop(); }
  Nvtx(const Nvtx&) = delete;
  Nvtx& operator=(const Nvtx&) = delete;
};

struct Tensor { const void* p = nullptr; int dtype = 0; int64_t numel = 0; };

struct LayerW {
  const float *ln_ff1_g, *ln_ff1_b, *ff1_b1, *ff1_b2;
  const void *ff1_w1, *ff1_w2;
  const float *ln_att_g, *ln_att_b, *bqkv, *att_u, *att_bdbias, *bo;
  const void *wqkv, *att_pos, *wo;
  const float *ln_conv_g, *ln_conv_b, *pw1_b, *dw_w, *dw_shift, *pw2_b;
  const void *pw1_w, *pw2_w;
  const float *ln_ff2_g, *ln_ff2_b, *ff2_b1, *ff2_b2;
  const void *ff2_w1, *ff2_w2;
  const float *ln_out_g, *ln_out_b;
};

struct Plan {           // workspace offsets (bytes) for one (B, L_max)
  int B, L_max, F_max, T1, F1, T2, F2, T3, F3, M;
  size_t wav, len, mel, mel_len, mel_part, mel_stats, enc_len, sub1, sub2, sub3, sub4, x, xn, hbuf, abuf, cbuf, vt, enc, encp;
  int n_rel_pad, ld_vt;
  size_t tokens, frames, ntok, dec_ws, total;
};

inline int conv_len(int n) { return n > 0 ? (n - 1) / 2 + 1 : 0; }   // floor division as in NeMo's calc_length: 0 stays 0
// Encoder-frame capacity of the padded activation tensors: the subsampled length rounded up to a multiple of 8, so that
// every utterance starts at a 16-byte-aligned column of the transposed V buffer (TMA wants the innermost coordinate
// 16-byte aligned: an odd T_max raised "illegal instruction" on the V^T tile loads of the attention kernel).
inline int enc_capacity(int mel_frames) { return (conv_len(conv_len(conv_len(mel_frames))) + 7) & ~7; }

// CUDA-event pairs around launches on their own streams, created on first use and reused after clear(); one
// (tag, flops) entry per completed pair.
struct EventLog {
  bool on = false;
  std::vector<cudaEvent_t> ev;
  std::vector<std::pair<std::string, double>> entries;
  void begin(cudaStream_t s) {
    const size_t i = 2 * entries.size();
    while (ev.size() < i + 2) { cudaEvent_t x; cudaEventCreate(&x); ev.push_back(x); }
    cudaEventRecord(ev[i], s);
  }
  void end(cudaStream_t s, const std::string& tag, double flops) {
    cudaEventRecord(ev[2 * entries.size() + 1], s);
    entries.emplace_back(tag, flops);
  }
  float ms(size_t i) const { float t = 0.f; cudaEventElapsedTime(&t, ev[2 * i], ev[2 * i + 1]); return t; }
  void clear() { entries.clear(); }
  ~EventLog() { for (cudaEvent_t x : ev) cudaEventDestroy(x); }
};

}  // namespace

struct rs_engine {
  rs_model_config cfg;
  int device = 0;
  int num_sms = 148;
  std::map<std::string, Tensor> w;
  rs::LmTables fe{};          // tables of the fused log-mel kernel (logmel_tables.py)
  // ALSD beam search (decode_alsd.cu): fp32-accurate tripled weights (optional: present when the engine was created with them),
  // an engine-owned workspace grown on demand, a pinned word for the periodic "all utterances finished" check
  struct { const void *out_w3 = nullptr, *lstm_w3 = nullptr, *pred_w3 = nullptr; const float* out_b = nullptr; int n_pad = 0; } alsd;
  void* alsd_ws = nullptr;
  size_t alsd_ws_bytes = 0;
  int* alsd_done_host = nullptr;
  unsigned int* lm_tickets = nullptr;   // per-utterance CTA tickets of the log-mel statistics (engine-owned, kept zero between launches)
  static constexpr int kMaxBatch = 1 << 16;
  struct { const float *c0w, *c0b, *d1w, *d1b, *p1b, *d2w, *d2b, *p2b, *ob; const void *p1w, *p2w, *ow; } sub;
  std::vector<LayerW> layers;
  struct { const void *enc_w, *out_w, *lstm_w, *pred_w; const float *enc_b, *out_b, *embed, *lstm_b, *pred_b, *gate_tab; } dec;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  mutable char err[512] = "";
  int64_t launches = 0;
  bool timing = false;
  cudaEvent_t ev[6] = {};               // stage marks of the whole path (rs_stage_times_ms)
  bool ev_ok = false;
  EventLog gemm_log;                    // every GEMM launch, with its 2*M*N*K
  // per-kernel timing inside the real pipeline (warm caches, back-to-back launches): event pair around every launch
  EventLog kernel_log;
  // rs_transcribe_batch: host->device copies run on their own stream in utterance chunks so the frontend of
  // chunk i overlaps the copy of chunk i+1
  static constexpr int kCopyChunks = 8;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_ev[kCopyChunks + 1] = {};
  bool copy_ok = false;
};

namespace {

int fail(const rs_engine* e, int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(e ? e->err : g_create_error, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define RS_CUDA(e, call)                                                                   \
  do {                                                                                     \
    cudaError_t _c = (call);                                                               \
    if (_c != cudaSuccess) return fail((e), RS_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(_c)); \
  } while (0)

// Bump allocator of workspace offsets: every region starts 256-byte aligned; `off` ends as the total size.
struct Arena {
  size_t off = 0;
  size_t take(size_t bytes) { const size_t o = off; off = (off + bytes + 255) & ~static_cast<size_t>(255); return o; }
};

inline size_t dec_ws_bytes(const rs_engine* e, int B) {
  return rs::rnnt_spec_workspace_bytes(B, e->cfg.joint_hidden, e->cfg.pred_hidden, e->num_sms);
}

Plan make_plan(const rs_engine* e, int B, int L_max, int U_max) {
  const rs_model_config& c = e->cfg;
  Plan p{};
  p.B = B; p.L_max = L_max;
  p.F_max = L_max / c.n_window_stride + 1;
  p.T1 = conv_len(p.F_max); p.F1 = conv_len(c.n_mels);
  p.T2 = conv_len(p.T1); p.F2 = conv_len(p.F1);
  p.T3 = enc_capacity(p.F_max); p.F3 = conv_len(p.F2);
  p.M = B * p.T3;
  const size_t C = c.sub_channels, d = c.d_model;
  const size_t wide = static_cast<size_t>(c.d_ff) > 3 * d ? c.d_ff : 3 * d;
  Arena a;
  p.wav = a.take(static_cast<size_t>(B) * L_max * 4);
  p.len = a.take(static_cast<size_t>(B) * 4);
  p.mel = a.take(static_cast<size_t>(B) * p.F_max * c.n_mels * 4);
  p.mel_len = a.take(static_cast<size_t>(B) * 4);
  p.mel_part = a.take(static_cast<size_t>(B) * rs::logmel_tiles(L_max, c.n_window_stride) * c.n_mels * 2 * 4);   // per-CTA (sum, sum of squares)
  p.mel_stats = a.take(static_cast<size_t>(B) * c.n_mels * 2 * 4);                                               // (mean, 1 / (std + eps))
  p.enc_len = a.take(static_cast<size_t>(B) * 4);
  p.sub1 = a.take(static_cast<size_t>(B) * p.T2 * p.F2 * C * 2);
  p.sub2 = a.take(static_cast<size_t>(B) * p.T2 * p.F2 * C * 2);
  p.sub3 = a.take(static_cast<size_t>(B) * p.T3 * p.F3 * C * 2);
  p.sub4 = a.take(static_cast<size_t>(B) * p.T3 * p.F3 * C * 2);
  p.x = a.take(static_cast<size_t>(p.M) * d * 4);
  p.xn = a.take(static_cast<size_t>(p.M) * d * 2);
  p.hbuf = a.take(static_cast<size_t>(p.M) * wide * 2);
  p.abuf = a.take(static_cast<size_t>(p.M) * d * 2);
  p.cbuf = a.take(static_cast<size_t>(p.M) * d * 2);
  p.n_rel_pad = ((c.att_left + c.att_right + 1 + 31) / 32) * 32;
  p.ld_vt = ((p.M + 255) / 256) * 256 + 64;                               // V^T row pitch: covers the GEMM's 256-row tile overhang
  p.vt = a.take(static_cast<size_t>(d) * p.ld_vt * 2);
  p.enc = a.take(static_cast<size_t>(p.M) * d * 4);
  p.encp = a.take(static_cast<size_t>(p.M) * c.joint_hidden * 4);
  p.tokens = a.take(static_cast<size_t>(B) * U_max * 4);
  p.frames = a.take(static_cast<size_t>(B) * U_max * 4);
  p.ntok = a.take(static_cast<size_t>(B) * 4);
  p.dec_ws = a.take(dec_ws_bytes(e, B));
  p.total = a.off;
  return p;
}

template <typename T>
T* at(const rs_engine* e, size_t off) { return reinterpret_cast<T*>(static_cast<char*>(e->ws) + off); }

int need(rs_engine* e, const char* name, int dtype, int64_t numel, const void** out) {
  auto it = e->w.find(name);
  if (it == e->w.end()) return fail(e, RS_ERR_MISSING_WEIGHT, "weight '%s' missing from the table", name);
  if (it->second.dtype != dtype || it->second.numel != numel)
    return fail(e, RS_ERR_MISSING_WEIGHT, "weight '%s': dtype/numel (%d, %lld) != expected (%d, %lld)", name,
                it->second.dtype, (long long)it->second.numel, dtype, (long long)numel);
  *out = it->second.p;
  return RS_OK;
}

#define NEED(field, name, dt, n)                                                   \
  do {                                                                             \
    const void* _p;                                                                \
    int _r = need(e, (name), (dt), (n), &_p);                                      \
    if (_r != RS_OK) return _r;                                                    \
    field = static_cast<decltype(field)>(_p);                                      \
  } while (0)

int bind_weights(rs_engine* e) {
  const rs_model_config& c = e->cfg;
  const int64_t d = c.d_model, ff = c.d_ff, C = c.sub_channels, H = c.n_heads, dk = d / H;
  const int64_t n_rel_pad = ((c.att_left + c.att_right + 1 + 31) / 32) * 32, k = c.conv_kernel;
  const int64_t F3 = conv_len(conv_len(conv_len(c.n_mels)));
  NEED(e->fe.window, "fe.window", RS_F32, c.n_fft);
  NEED(e->fe.tw_b, "fe.tw_b", RS_F32, 512);
  NEED(e->fe.tw_x, "fe.tw_x", RS_F32, 256);
  NEED(e->fe.mel_meta, "fe.mel_meta", RS_I32, rs::kLmMetaInts);
  {
    auto it = e->w.find("fe.mel_w");
    if (it == e->w.end() || it->second.dtype != RS_F32 || it->second.numel <= 0 || it->second.numel % 16)
      return fail(e, RS_ERR_MISSING_WEIGHT, "weight 'fe.mel_w' (f32 [taps, 16]) missing from the table or misshapen");
    e->fe.mel_w = static_cast<const float*>(it->second.p);
    e->fe.n_taps = static_cast<int>(it->second.numel / 16);
  }
  NEED(e->sub.c0w, "sub.conv0.w", RS_F32, C * 9); NEED(e->sub.c0b, "sub.conv0.b", RS_F32, C);
  NEED(e->sub.d1w, "sub.dw1.w", RS_F32, C * 9); NEED(e->sub.d1b, "sub.dw1.b", RS_F32, C);
  NEED(e->sub.p1w, "sub.pw1.w", RS_BF16, C * C); NEED(e->sub.p1b, "sub.pw1.b", RS_F32, C);
  NEED(e->sub.d2w, "sub.dw2.w", RS_F32, C * 9); NEED(e->sub.d2b, "sub.dw2.b", RS_F32, C);
  NEED(e->sub.p2w, "sub.pw2.w", RS_BF16, C * C); NEED(e->sub.p2b, "sub.pw2.b", RS_F32, C);
  NEED(e->sub.ow, "sub.out.w", RS_BF16, d * F3 * C); NEED(e->sub.ob, "sub.out.b", RS_F32, d);
  e->layers.resize(c.n_layers);
  for (int i = 0; i < c.n_layers; ++i) {
    LayerW& L = e->layers[i];
    char nm[64];
    auto N = [&](const char* s) { snprintf(nm, sizeof nm, "L%d.%s", i, s); return nm; };
    NEED(L.ln_ff1_g, N("ln_ff1.g"), RS_F32, d); NEED(L.ln_ff1_b, N("ln_ff1.b"), RS_F32, d);
    NEED(L.ff1_w1, N("ff1.w1"), RS_BF16, ff * d); NEED(L.ff1_b1, N("ff1.b1"), RS_F32, ff);
    NEED(L.ff1_w2, N("ff1.w2"), RS_BF16, d * ff); NEED(L.ff1_b2, N("ff1.b2"), RS_F32, d);
    NEED(L.ln_att_g, N("ln_att.g"), RS_F32, d); NEED(L.ln_att_b, N("ln_att.b"), RS_F32, d);
    NEED(L.wqkv, N("att.wqkv"), RS_BF16, 3 * d * d); NEED(L.bqkv, N("att.bqkv"), RS_F32, 3 * d);
    NEED(L.att_pos, N("att.pos"), RS_BF16, H * n_rel_pad * dk);
    NEED(L.att_u, N("att.u"), RS_F32, d); NEED(L.att_bdbias, N("att.bdbias"), RS_F32, H * n_rel_pad);
    NEED(L.wo, N("att.wo"), RS_BF16, d * d); NEED(L.bo, N("att.bo"), RS_F32, d);
    NEED(L.ln_conv_g, N("ln_conv.g"), RS_F32, d); NEED(L.ln_conv_b, N("ln_conv.b"), RS_F32, d);
    NEED(L.pw1_w, N("conv.pw1.w"), RS_BF16, 2 * d * d); NEED(L.pw1_b, N("conv.pw1.b"), RS_F32, 2 * d);
    NEED(L.dw_w, N("conv.dw.w"), RS_F32, k * d); NEED(L.dw_shift, N("conv.dw.shift"), RS_F32, d);
    NEED(L.pw2_w, N("conv.pw2.w"), RS_BF16, d * d); NEED(L.pw2_b, N("conv.pw2.b"), RS_F32, d);
    NEED(L.ln_ff2_g, N("ln_ff2.g"), RS_F32, d); NEED(L.ln_ff2_b, N("ln_ff2.b"), RS_F32, d);
    NEED(L.ff2_w1, N("ff2.w1"), RS_BF16, ff * d); NEED(L.ff2_b1, N("ff2.b1"), RS_F32, ff);
    NEED(L.ff2_w2, N("ff2.w2"), RS_BF16, d * ff); NEED(L.ff2_b2, N("ff2.b2"), RS_F32, d);
    NEED(L.ln_out_g, N("ln_out.g"), RS_F32, d); NEED(L.ln_out_b, N("ln_out.b"), RS_F32, d);
  }
  const int64_t Hj = c.joint_hidden, Hp = c.pred_hidden, NC = c.vocab_size + 1;
  if (e->w.count("alsd.out.w3") != 0) {                  // optional: only an engine that was asked for beam search carries these
    const int64_t n_pad = (NC + 63) / 64 * 64;
    NEED(e->alsd.out_w3, "alsd.out.w3", RS_BF16, n_pad * 3 * Hj); NEED(e->alsd.out_b, "alsd.out.b", RS_F32, n_pad);
    NEED(e->alsd.lstm_w3, "alsd.lstm.w3", RS_BF16, 4 * Hp * 6 * Hp); NEED(e->alsd.pred_w3, "alsd.pred.w3", RS_BF16, Hj * 3 * Hp);
    e->alsd.n_pad = static_cast<int>(n_pad);
  }
  NEED(e->dec.enc_w, "joint.enc.w", RS_BF16, Hj * d); NEED(e->dec.enc_b, "joint.enc.b", RS_F32, Hj);
  NEED(e->dec.out_w, "joint.out.w", RS_BF16, NC * Hj); NEED(e->dec.out_b, "joint.out.b", RS_F32, NC);
  NEED(e->dec.embed, "pred.embed", RS_F32, NC * Hp);
  NEED(e->dec.lstm_w, "pred.lstm.w", RS_BF16, 4 * Hp * 2 * Hp); NEED(e->dec.lstm_b, "pred.lstm.b", RS_F32, 4 * Hp);
  NEED(e->dec.gate_tab, "pred.gate_tab", RS_F32, NC * 4 * Hp);     // W_ih . embed[k] + b_ih + b_hh per token k (decode_spec.cu)
  NEED(e->dec.pred_w, "joint.pred.w", RS_BF16, Hj * Hp); NEED(e->dec.pred_b, "joint.pred.b", RS_F32, Hj);
  return RS_OK;
}

__global__ void enc_len_kernel(const int32_t* __restrict__ mel_len, int32_t* __restrict__ enc_len, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int n = mel_len[b];
  for (int i = 0; i < 3; ++i) n = n > 0 ? (n - 1) / 2 + 1 : 0;
  enc_len[b] = n;
}

#define RS_TRY(x) do { int _r = (x); if (_r != RS_OK) return _r; } while (0)

// Every launch of the engine goes through here.  `call(msg)` enqueues `n` kernels on `s` and returns the CUDA error (msg, 256
// bytes, may describe it better than the error's name).  Counts the launches, brackets the enqueue in the event logs that are
// on (the GEMM log takes the launches with flops > 0) and turns a failure into fail("<tag>: <description>").  In the kernel
// log the launch is named by `tag` without a leading "rs::" and without its argument list.
template <typename Call>
int launch(rs_engine* e, cudaStream_t s, const char* tag, int n, double flops, Call&& call) {
  const bool klog = e->kernel_log.on, glog = flops > 0 && e->gemm_log.on;
  if (glog) e->gemm_log.begin(s);
  if (klog) e->kernel_log.begin(s);
  char msg[256] = "";
  const cudaError_t c = call(msg);
  if (c != cudaSuccess) return fail(e, RS_ERR_CUDA, "%s: %s", tag, msg[0] ? msg : cudaGetErrorString(c));
  if (klog || glog) {
    std::string name(tag);
    if (name.rfind("rs::", 0) == 0) name = name.substr(4);
    name = name.substr(0, name.find('('));
    if (klog) e->kernel_log.end(s, name, 0.0);
    if (glog) e->gemm_log.end(s, name, flops);
  }
  e->launches += n;
  return RS_OK;
}

#define RS_K(e, s, call, n) RS_TRY(launch((e), (s), #call, (n), 0.0, [&](char*) { return (call); }))

int gemm(rs_engine* e, const rs::GemmArgs& g, cudaStream_t s) {
  char tag[64] = "gemm";
  if (e->kernel_log.on) snprintf(tag, sizeof tag, "gemm N=%d K=%d epi=%d", g.N, g.K, g.epilogue);
  return launch(e, s, tag, 1, 2.0 * g.M * static_cast<double>(g.N) * g.K,
                [&](char* msg) { return rs::launch_gemm(g, e->num_sms, s, msg); });
}

int gemm(rs_engine* e, const void* a, const void* w, const float* bias, const float* resid, void* out, int M, int N,
         int K, int epi, float alpha, cudaStream_t s) {
  return gemm(e, rs::GemmArgs{a, w, bias, resid, out, M, N, K, epi, alpha}, s);
}

int check_ws(rs_engine* e, const Plan& p) {
  if (e->ws == nullptr) return fail(e, RS_ERR_WORKSPACE, "no workspace set (rs_set_workspace)");
  if (p.total > e->ws_bytes)
    return fail(e, RS_ERR_WORKSPACE, "workspace too small: need %zu bytes for B=%d L_max=%d, have %zu", p.total, p.B, p.L_max, e->ws_bytes);
  return RS_OK;
}

void mark(rs_engine* e, int i, cudaStream_t s) {
  if (e->timing && e->ev_ok) cudaEventRecord(e->ev[i], s);
}

// Log-mel of utterances [b0, b0 + nb) of a batch whose statistics live at plan offsets (absolute utterance index).
// normalise = false leaves `mel` un-normalised for sub_conv0_dw1_kernel (the transcribe path); rs_logmel passes true.
int do_logmel(rs_engine* e, const void* wav, bool i16, const int32_t* len, int nb, int L_max, float* mel, int32_t* mel_len,
              float* partials, float* stats, int b0, bool normalise, cudaStream_t s) {
  Nvtx range("rs::logmel");
  const rs_model_config& c = e->cfg;
  if (b0 + nb > rs_engine::kMaxBatch) return fail(e, RS_ERR_INVALID_ARG, "batch of %d utterances exceeds the engine limit of %d", b0 + nb, rs_engine::kMaxBatch);
  rs::LogmelArgs a{};
  a.wav = wav; a.wav_i16 = i16; a.len = len; a.B = nb; a.L_max = L_max; a.mel = mel; a.mel_len = mel_len;
  a.partials = partials + static_cast<size_t>(b0) * rs::logmel_tiles(L_max, c.n_window_stride) * c.n_mels * 2;
  a.stats = stats + static_cast<size_t>(b0) * c.n_mels * 2;
  a.tickets = e->lm_tickets + b0;
  a.tb = e->fe; a.n_mels = c.n_mels; a.hop = c.n_window_stride; a.n_fft = c.n_fft; a.win = c.n_window_size;
  a.preemph = c.preemph; a.guard = c.log_zero_guard; a.eps = c.norm_eps; a.normalise_in_place = normalise;
  RS_K(e, s, rs::launch_logmel_fused(a, s), normalise ? 2 : 1);
  return RS_OK;
}

// mel_stats == nullptr: `mel` is already normalised (rs_encode takes rs_logmel's output)
int do_sub_conv0(rs_engine* e, const Plan& p, const float* mel, const int32_t* mel_len, const float* mel_stats, int b0, int nb, cudaStream_t s) {
  Nvtx range("rs::subsampling.conv0_dw1");
  const rs_model_config& c = e->cfg;
  const int C = c.sub_channels;
  rs::SubsampleArgs sa{mel + static_cast<size_t>(b0) * p.F_max * c.n_mels, mel_len + b0,
                       mel_stats ? mel_stats + static_cast<size_t>(b0) * c.n_mels * 2 : nullptr, nb, p.F_max, c.n_mels, C,
                       e->sub.c0w, e->sub.c0b, e->sub.d1w, e->sub.d1b,
                       at<uint16_t>(e, p.sub1) + static_cast<size_t>(b0) * p.T2 * p.F2 * C, p.T1, p.F1, p.T2, p.F2};
  RS_K(e, s, rs::launch_sub_conv0_dw1(sa, s), 1);
  return RS_OK;
}

// The encoder after the first (fused) subsampling conv, which the caller has run into p.sub1.
int do_encode(rs_engine* e, const Plan& p, const int32_t* mel_len, float* enc, int32_t* enc_len, int n_layers, cudaStream_t s) {
  const rs_model_config& c = e->cfg;
  const int d = c.d_model, C = c.sub_channels, M = p.M, B = p.B;
  if (n_layers < 0 || n_layers > c.n_layers) n_layers = c.n_layers;
  enc_len_kernel<<<(B + 127) / 128, 128, 0, s>>>(mel_len, enc_len, B);
  RS_K(e, s, cudaGetLastError(), 1);
  // ---- ConvSubsampling
  RS_TRY(gemm(e, at<void>(e, p.sub1), e->sub.p1w, e->sub.p1b, nullptr, at<void>(e, p.sub2), B * p.T2 * p.F2, C, C,
              RS_EPI_BIAS_RELU_BF16, 1.f, s));
  RS_K(e, s, rs::launch_sub_dw(at<void>(e, p.sub2), at<void>(e, p.sub3), e->sub.d2w, e->sub.d2b, mel_len, 2, B, p.T2, p.F2,
                            p.T3, p.F3, C, s), 1);
  RS_TRY(gemm(e, at<void>(e, p.sub3), e->sub.p2w, e->sub.p2b, nullptr, at<void>(e, p.sub4), B * p.T3 * p.F3, C, C,
              RS_EPI_BIAS_RELU_BF16, 1.f, s));
  float* x = at<float>(e, p.x);
  Nvtx layers_range("rs::conformer_layers");
  RS_TRY(gemm(e, at<void>(e, p.sub4), e->sub.ow, e->sub.ob, nullptr, x, M, d, p.F3 * C, RS_EPI_BIAS_F32, c.xscale, s));
  mark(e, 2, s);
  // ---- Conformer layers
  void* xn = at<void>(e, p.xn); void* hb = at<void>(e, p.hbuf); void* ab = at<void>(e, p.abuf); void* cb = at<void>(e, p.cbuf);
  if (n_layers > 0) {
    const LayerW& L0 = e->layers[0];
    RS_K(e, s, rs::launch_layernorm(x, L0.ln_ff1_g, L0.ln_ff1_b, nullptr, xn, nullptr, nullptr, M, d, c.ln_eps, s), 1);
  }
  auto resid_gemm = [&](const void* a, const void* w, const float* bias, int K, float alpha) -> int {
    return gemm(e, a, w, bias, x, x, M, d, K, RS_EPI_RESID_F32, alpha, s);
  };
  for (int i = 0; i < n_layers; ++i) {
    const LayerW& L = e->layers[i];
    char layer_name[32];
    snprintf(layer_name, sizeof layer_name, "rs::conformer_layer[%d]", i);
    Nvtx layer_range(layer_name);
    RS_TRY(gemm(e, xn, L.ff1_w1, L.ff1_b1, nullptr, hb, M, c.d_ff, d, RS_EPI_BIAS_SWISH_BF16, 1.f, s));
    RS_TRY(resid_gemm(hb, L.ff1_w2, L.ff1_b2, c.d_ff, 0.5f));
    RS_K(e, s, rs::launch_layernorm(x, L.ln_att_g, L.ln_att_b, nullptr, xn, nullptr, nullptr, M, d, c.ln_eps, s), 1);
    // the relative-position term (q + pos_bias_v) . p[c] is a UMMA inside the attention kernel (attention_tc.cu): no score tensor in HBM
    rs::AttnArgs aa{hb, L.att_pos, L.att_bdbias, p.n_rel_pad, L.att_u, ab, enc_len, B, p.T3, c.n_heads, d / c.n_heads, c.att_left, c.att_right, c.global_tokens};
    aa.vt = at<void>(e, p.vt); aa.ld_vt = p.ld_vt;
    {   // q | k row-major, V transposed (keys contiguous) for the attention's P.V product
      rs::GemmArgs g{xn, L.wqkv, L.bqkv, nullptr, hb, M, 3 * d, d, RS_EPI_QKV_VT, 1.f};
      g.out2 = at<void>(e, p.vt); g.split = 2 * d; g.ld2 = p.ld_vt;
      RS_TRY(gemm(e, g, s));
    }
    RS_K(e, s, rs::launch_attention_tc(aa, s), c.global_tokens > 0 ? 2 : 1);
    RS_TRY(resid_gemm(ab, L.wo, L.bo, d, 1.f));
    RS_K(e, s, rs::launch_layernorm(x, L.ln_conv_g, L.ln_conv_b, nullptr, xn, nullptr, nullptr, M, d, c.ln_eps, s), 1);
    RS_TRY(gemm(e, xn, L.pw1_w, L.pw1_b, nullptr, ab, M, 2 * d, d, RS_EPI_BIAS_GLU_BF16, 1.f, s));
    RS_K(e, s, rs::launch_conv_dw(ab, cb, L.dw_w, L.dw_shift, enc_len, B, p.T3, d, c.conv_kernel, s), 1);
    RS_TRY(resid_gemm(cb, L.pw2_w, L.pw2_b, d, 1.f));
    RS_K(e, s, rs::launch_layernorm(x, L.ln_ff2_g, L.ln_ff2_b, nullptr, xn, nullptr, nullptr, M, d, c.ln_eps, s), 1);
    RS_TRY(gemm(e, xn, L.ff2_w1, L.ff2_b1, nullptr, hb, M, c.d_ff, d, RS_EPI_BIAS_SWISH_BF16, 1.f, s));
    RS_TRY(resid_gemm(hb, L.ff2_w2, L.ff2_b2, c.d_ff, 0.5f));
    if (i + 1 < n_layers) {   // norm_out chained with the next layer's norm_feed_forward1
      const LayerW& Ln = e->layers[i + 1];
      RS_K(e, s, rs::launch_layernorm(x, L.ln_out_g, L.ln_out_b, x, xn, Ln.ln_ff1_g, Ln.ln_ff1_b, M, d, c.ln_eps, s), 1);
    } else {
      RS_K(e, s, rs::launch_layernorm(x, L.ln_out_g, L.ln_out_b, enc, nullptr, nullptr, nullptr, M, d, c.ln_eps, s), 1);
    }
  }
  if (n_layers == 0) RS_CUDA(e, cudaMemcpyAsync(enc, x, static_cast<size_t>(M) * d * 4, cudaMemcpyDeviceToDevice, s));
  RS_K(e, s, rs::launch_zero_pad_rows(enc, enc_len, B, p.T3, d, s), 1);
  return RS_OK;
}

int do_greedy(rs_engine* e, const Plan& p, const float* enc, const int32_t* enc_len, int T_max, int32_t* tokens,
              int32_t* frames, int32_t* ntok, int U_max, cudaStream_t s) {
  Nvtx range("rs::rnnt_greedy (joint.enc projection + persistent decode)");
  const rs_model_config& c = e->cfg;
  const int M = p.B * T_max;
  RS_K(e, s, rs::launch_f32_to_bf16(enc, at<void>(e, p.xn), static_cast<int64_t>(M) * c.d_model, s), 1);
  RS_TRY(gemm(e, at<void>(e, p.xn), e->dec.enc_w, e->dec.enc_b, nullptr, at<void>(e, p.encp), M, c.joint_hidden, c.d_model,
              RS_EPI_BIAS_F32, 1.f, s));
  mark(e, 4, s);
  rs::DecodeArgs da{at<float>(e, p.encp), enc_len, e->dec.out_w, e->dec.out_b, e->dec.embed, e->dec.lstm_w, e->dec.lstm_b, e->dec.gate_tab,
                    e->dec.pred_w, e->dec.pred_b, tokens, frames, ntok, p.B, T_max, c.joint_hidden, c.pred_hidden,
                    c.vocab_size, U_max, c.max_symbols};
  // One decode kernel for every batch size (windowed, weights-stationary, joint on tcgen05: decode_spec.cu): an utterance's
  // logits are accumulated in the same order whether it is decoded alone or inside a batch, so results do not depend on
  // batch composition.
  RS_K(e, s, rs::launch_rnnt_greedy_spec(da, at<void>(e, p.dec_ws), e->num_sms, s), 2);
  return RS_OK;
}

// The whole path.  chunks == 0: wav / len and the outputs are device pointers, nothing synchronises.  chunks >= 1: they are
// host buffers; wav / len are copied into the workspace in `chunks` utterance chunks -- on the copy stream when there are
// several, so that log-mel and the first (fused) subsampling conv of a chunk that has landed overlap the copy of the next --
// and the results are copied back before the call synchronises.  `wav` holds f32 samples, or int16 PCM (scaled by 2^-15
// inside the log-mel kernel) when i16.
int transcribe(rs_engine* e, const void* wav_in, bool i16, const int32_t* len_in, int B, int L_max, int32_t* tokens,
               int32_t* frames, int32_t* n_tok, int U_max, int chunks, cudaStream_t s) {
  Plan p = make_plan(e, B, L_max, U_max);
  RS_TRY(check_ws(e, p));
  const bool host = chunks > 0;
  const size_t esz = i16 ? 2 : 4;                       // the waveform region of the workspace is sized for f32
  const char* wav = host ? at<char>(e, p.wav) : static_cast<const char*>(wav_in);
  const int32_t* len = host ? at<int32_t>(e, p.len) : len_in;
  const int per = host ? (B + chunks - 1) / chunks : B;
  const cudaStream_t cs = chunks > 1 ? e->copy_stream : s;
  if (host) {
    if (cs != s) {   // the workspace may still be in use by work already queued on the caller's stream
      RS_CUDA(e, cudaEventRecord(e->copy_ev[rs_engine::kCopyChunks], s));
      RS_CUDA(e, cudaStreamWaitEvent(cs, e->copy_ev[rs_engine::kCopyChunks], 0));
    }
    RS_CUDA(e, cudaMemcpyAsync(at<int32_t>(e, p.len), len_in, static_cast<size_t>(B) * 4, cudaMemcpyHostToDevice, cs));
    for (int c = 0, b0 = 0; b0 < B; ++c, b0 += per) {
      const size_t off = static_cast<size_t>(b0) * L_max * esz, bytes = static_cast<size_t>(std::min(per, B - b0)) * L_max * esz;
      RS_CUDA(e, cudaMemcpyAsync(at<char>(e, p.wav) + off, static_cast<const char*>(wav_in) + off, bytes, cudaMemcpyHostToDevice, cs));
      if (cs != s) RS_CUDA(e, cudaEventRecord(e->copy_ev[c], cs));
    }
  }
  float* mel = at<float>(e, p.mel);
  int32_t* mel_len = at<int32_t>(e, p.mel_len);
  float* stats = at<float>(e, p.mel_stats);
  mark(e, 0, s);
  for (int c = 0, b0 = 0; b0 < B; ++c, b0 += per) {
    const int nb = std::min(per, B - b0);
    if (cs != s) RS_CUDA(e, cudaStreamWaitEvent(s, e->copy_ev[c], 0));
    RS_TRY(do_logmel(e, wav + static_cast<size_t>(b0) * L_max * esz, i16, len + b0, nb, L_max,
                     mel + static_cast<size_t>(b0) * p.F_max * e->cfg.n_mels, mel_len + b0, at<float>(e, p.mel_part), stats, b0, false, s));
    if (b0 + nb == B) mark(e, 1, s);
    RS_TRY(do_sub_conv0(e, p, mel, mel_len, stats, b0, nb, s));
  }
  RS_TRY(do_encode(e, p, mel_len, at<float>(e, p.enc), at<int32_t>(e, p.enc_len), -1, s));
  mark(e, 3, s);
  int32_t* tok = host ? at<int32_t>(e, p.tokens) : tokens;
  int32_t* frm = host ? at<int32_t>(e, p.frames) : frames;
  int32_t* cnt = host ? at<int32_t>(e, p.ntok) : n_tok;
  RS_TRY(do_greedy(e, p, at<float>(e, p.enc), at<int32_t>(e, p.enc_len), p.T3, tok, frm, cnt, U_max, s));
  mark(e, 5, s);
  if (host) {
    RS_CUDA(e, cudaMemcpyAsync(tokens, tok, static_cast<size_t>(B) * U_max * 4, cudaMemcpyDeviceToHost, s));
    RS_CUDA(e, cudaMemcpyAsync(frames, frm, static_cast<size_t>(B) * U_max * 4, cudaMemcpyDeviceToHost, s));
    RS_CUDA(e, cudaMemcpyAsync(n_tok, cnt, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost, s));
    RS_CUDA(e, cudaStreamSynchronize(s));
  }
  return RS_OK;
}

// The four rs_transcribe_* entry points: argument check, device, and the host entries' chunk rule (kCopyChunks chunks on
// the copy stream from 2 * kCopyChunks utterances on, else one on the caller's stream).
int transcribe_entry(const char* name, rs_engine* e, const void* wav, bool i16, const int32_t* len, int B, int L_max,
                     int32_t* tokens, int32_t* frames, int32_t* n_tok, int U_max, bool host, void* stream) {
  if (!e || !wav || !len || !tokens || !frames || !n_tok || B <= 0 || L_max <= 0 || U_max <= 0)
    return fail(e, RS_ERR_INVALID_ARG, "%s: bad arguments", name);
  RS_CUDA(e, cudaSetDevice(e->device));
  const int chunks = !host ? 0 : (e->copy_ok && B >= 2 * rs_engine::kCopyChunks) ? rs_engine::kCopyChunks : 1;
  return transcribe(e, wav, i16, len, B, L_max, tokens, frames, n_tok, U_max, chunks, static_cast<cudaStream_t>(stream));
}

}  // namespace

extern "C" {

int rs_engine_create(const rs_model_config* cfg, const rs_tensor* weights, int n_weights, int device, rs_engine** out) {
  if (cfg == nullptr || weights == nullptr || out == nullptr) return fail(nullptr, RS_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  if (cfg->n_fft != 512) return fail(nullptr, RS_ERR_UNSUPPORTED, "n_fft=%d unsupported (frontend kernel is built for 512)", cfg->n_fft);
  if (cfg->d_model % cfg->n_heads || cfg->d_model / cfg->n_heads != 128)
    return fail(nullptr, RS_ERR_UNSUPPORTED, "d_model/n_heads must be 128 (got %d/%d)", cfg->d_model, cfg->n_heads);
  if (cfg->d_model != 256 && cfg->d_model != 512 && cfg->d_model != 1024)
    return fail(nullptr, RS_ERR_UNSUPPORTED, "d_model=%d unsupported (256/512/1024)", cfg->d_model);
  if (cfg->conv_kernel != 9) return fail(nullptr, RS_ERR_UNSUPPORTED, "conv_kernel=%d unsupported (9)", cfg->conv_kernel);
  if (cfg->global_tokens < 0 || cfg->global_tokens > 1)
    return fail(nullptr, RS_ERR_UNSUPPORTED, "global_tokens=%d unsupported (the attention kernels implement 0 or 1)", cfg->global_tokens);
  if (cfg->att_left < 0 || cfg->att_right < 0 || cfg->att_left > 128 || cfg->att_right > 128 || (cfg->att_left & 7))
    return fail(nullptr, RS_ERR_UNSUPPORTED, "att context (%d, %d) unsupported: the attention kernel covers limited local context with 0 <= left, right <= 128 and left %% 8 == 0 (the shipped model is [128, 128])", cfg->att_left, cfg->att_right);
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0)
    return fail(nullptr, RS_ERR_CUDA, "no CUDA device available (%s); this engine has no CPU path", cudaGetErrorString(ce));
  if (device < 0 || device >= ndev) return fail(nullptr, RS_ERR_INVALID_ARG, "device %d out of range (%d devices)", device, ndev);
  ce = cudaSetDevice(device);
  if (ce != cudaSuccess) return fail(nullptr, RS_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(ce));
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) return fail(nullptr, RS_ERR_UNSUPPORTED, "device %d is sm_%d%d; kernels are built for sm_100a only", device, prop.major, prop.minor);
  rs_engine* e = new rs_engine();
  e->cfg = *cfg; e->device = device; e->num_sms = prop.multiProcessorCount;
  for (int i = 0; i < n_weights; ++i) e->w[weights[i].name] = Tensor{weights[i].dev_ptr, weights[i].dtype, weights[i].numel};
  int r = bind_weights(e);
  if (r != RS_OK) { snprintf(g_create_error, sizeof g_create_error, "%s", e->err); delete e; return r; }
  if (cudaMalloc(&e->lm_tickets, rs_engine::kMaxBatch * sizeof(unsigned int)) != cudaSuccess ||
      cudaMemset(e->lm_tickets, 0, rs_engine::kMaxBatch * sizeof(unsigned int)) != cudaSuccess) {
    snprintf(g_create_error, sizeof g_create_error, "cannot allocate the log-mel ticket array (%s)", cudaGetErrorString(cudaGetLastError()));
    cudaFree(e->lm_tickets);
    delete e;
    return RS_ERR_CUDA;
  }
  e->ev_ok = true;
  for (auto& ev : e->ev) if (cudaEventCreate(&ev) != cudaSuccess) e->ev_ok = false;
  e->copy_ok = cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
  for (auto& ev : e->copy_ev) if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) e->copy_ok = false;
  *out = e;
  return RS_OK;
}

void rs_engine_destroy(rs_engine* e) {
  if (e == nullptr) return;
  if (e->ev_ok) for (auto& ev : e->ev) cudaEventDestroy(ev);
  for (auto& ev : e->copy_ev) if (ev) cudaEventDestroy(ev);
  if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
  cudaFree(e->lm_tickets);
  cudaFree(e->alsd_ws);
  if (e->alsd_done_host) cudaFreeHost(e->alsd_done_host);
  delete e;
}

const char* rs_last_error(const rs_engine* e) { return e ? e->err : g_create_error; }

int rs_workspace_bytes(const rs_engine* e, int B, int L_max, size_t* bytes) {
  if (e == nullptr || bytes == nullptr || B <= 0 || L_max <= 0) return fail(e, RS_ERR_INVALID_ARG, "bad arguments");
  // token capacity: max_symbols per encoder frame is the hard upper bound of the greedy loop
  const int T = enc_capacity(L_max / e->cfg.n_window_stride + 1);
  *bytes = make_plan(e, B, L_max, T * e->cfg.max_symbols).total;
  return RS_OK;
}

int rs_set_workspace(rs_engine* e, void* dev_ptr, size_t bytes) {
  if (e == nullptr) return RS_ERR_INVALID_ARG;
  if (reinterpret_cast<uintptr_t>(dev_ptr) & 255) return fail(e, RS_ERR_INVALID_ARG, "workspace must be 256-byte aligned");
  e->ws = dev_ptr; e->ws_bytes = bytes;
  return RS_OK;
}

int rs_mel_frames(const rs_engine* e, int n) { return n / e->cfg.n_window_stride + 1; }
int rs_enc_frames(const rs_engine* e, int n) { return enc_capacity(rs_mel_frames(e, n)); }
int rs_mel_valid(const rs_engine* e, int n) { return (n + 2 * (e->cfg.n_fft / 2) - e->cfg.n_fft) / e->cfg.n_window_stride; }
int rs_enc_valid(const rs_engine* e, int n) { return conv_len(conv_len(conv_len(rs_mel_valid(e, n)))); }

int rs_logmel(rs_engine* e, const float* wav, const int32_t* len, int B, int L_max, float* mel, int32_t* mel_len, void* stream) {
  if (!e || !wav || !len || !mel || !mel_len || B <= 0 || L_max <= 0) return fail(e, RS_ERR_INVALID_ARG, "rs_logmel: bad arguments");
  RS_CUDA(e, cudaSetDevice(e->device));
  Plan p = make_plan(e, B, L_max, 1);               // the statistics scratch lives in the workspace
  RS_TRY(check_ws(e, p));
  return do_logmel(e, wav, false, len, B, L_max, mel, mel_len, at<float>(e, p.mel_part), at<float>(e, p.mel_stats), 0, true,
                   static_cast<cudaStream_t>(stream));
}

int rs_encode(rs_engine* e, const float* mel, const int32_t* mel_len, int B, int F_max, float* enc, int32_t* enc_len,
              int n_layers, void* stream) {
  if (!e || !mel || !mel_len || !enc || !enc_len || B <= 0 || F_max <= 0) return fail(e, RS_ERR_INVALID_ARG, "rs_encode: bad arguments");
  RS_CUDA(e, cudaSetDevice(e->device));
  const int L_max = (F_max - 1) * e->cfg.n_window_stride;
  Plan p = make_plan(e, B, L_max, 1);
  RS_TRY(check_ws(e, p));
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  RS_TRY(do_sub_conv0(e, p, mel, mel_len, nullptr, 0, B, s));
  return do_encode(e, p, mel_len, enc, enc_len, n_layers, s);
}

int rs_rnnt_greedy(rs_engine* e, const float* enc, const int32_t* enc_len, int B, int T_max, int32_t* tokens,
                   int32_t* frames, int32_t* n_tok, int U_max, void* stream) {
  if (!e || !enc || !enc_len || !tokens || !frames || !n_tok || B <= 0 || T_max <= 0 || U_max <= 0)
    return fail(e, RS_ERR_INVALID_ARG, "rs_rnnt_greedy: bad arguments");
  RS_CUDA(e, cudaSetDevice(e->device));
  Plan p{};
  // only xn / encp / dec_ws are touched: size them for M = B*T_max rows
  p.B = B; p.M = B * T_max;
  Arena a;
  p.xn = a.take(static_cast<size_t>(p.M) * e->cfg.d_model * 2);
  p.encp = a.take(static_cast<size_t>(p.M) * e->cfg.joint_hidden * 4);
  p.dec_ws = a.take(dec_ws_bytes(e, B));
  p.total = a.off;
  RS_TRY(check_ws(e, p));
  return do_greedy(e, p, enc, enc_len, T_max, tokens, frames, n_tok, U_max, static_cast<cudaStream_t>(stream));
}

int rs_transcribe_device(rs_engine* e, const float* wav, const int32_t* len, int B, int L_max, int32_t* tokens,
                         int32_t* frames, int32_t* n_tok, int U_max, void* stream) {
  return transcribe_entry("rs_transcribe_device", e, wav, false, len, B, L_max, tokens, frames, n_tok, U_max, false, stream);
}

int rs_transcribe_device_pcm16(rs_engine* e, const int16_t* wav, const int32_t* len, int B, int L_max, int32_t* tokens,
                               int32_t* frames, int32_t* n_tok, int U_max, void* stream) {
  return transcribe_entry("rs_transcribe_device_pcm16", e, wav, true, len, B, L_max, tokens, frames, n_tok, U_max, false, stream);
}

int rs_transcribe_batch(rs_engine* e, const float* wav_host, const int32_t* len_host, int B, int L_max,
                        int32_t* tokens_host, int32_t* frames_host, int32_t* n_tok_host, int U_max, void* stream) {
  return transcribe_entry("rs_transcribe_batch", e, wav_host, false, len_host, B, L_max, tokens_host, frames_host, n_tok_host,
                          U_max, true, stream);
}

int rs_transcribe_batch_pcm16(rs_engine* e, const int16_t* wav_host, const int32_t* len_host, int B, int L_max,
                              int32_t* tokens_host, int32_t* frames_host, int32_t* n_tok_host, int U_max, void* stream) {
  return transcribe_entry("rs_transcribe_batch_pcm16", e, wav_host, true, len_host, B, L_max, tokens_host, frames_host,
                          n_tok_host, U_max, true, stream);
}

// ALSD beam search over encoder outputs (decode_alsd.cu; semantics: oracle/alsd_restated.py).  Synchronises: the host checks every
// 32 steps whether every utterance's search has ended.
int rs_rnnt_alsd(rs_engine* e, const float* enc, const int32_t* enc_len, int B, int T_max, int beam, float u_max_ratio, int score_norm,
                 int recombine_returns_input, int32_t* y_dev, int32_t* step_dev, int32_t* n_dev, double* score_dev, int U_cap, void* stream) {
  if (!e || !enc || !enc_len || !y_dev || !step_dev || !n_dev || !score_dev || B <= 0 || T_max <= 0 || U_cap <= 0 || beam < 1 || beam > 8 || u_max_ratio < 0.f)
    return fail(e, RS_ERR_INVALID_ARG, "rs_rnnt_alsd: bad arguments (beam must be 1..8)");
  if (e->alsd.out_w3 == nullptr)
    return fail(e, RS_ERR_UNSUPPORTED, "rs_rnnt_alsd: the engine was created without the beam-search weight tensors (alsd.*)");
  RS_CUDA(e, cudaSetDevice(e->device));
  Nvtx range("rs::rnnt_alsd");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const rs_model_config& c = e->cfg;
  const int Hj = c.joint_hidden, Hp = c.pred_hidden, d = c.d_model, V = c.vocab_size, blank = c.vocab_size, n_pad = e->alsd.n_pad;
  const int M = B * T_max, R = B * beam;
  const int total_steps = T_max + static_cast<int>(u_max_ratio * static_cast<float>(T_max));
  const int max_nodes = 1 + beam * (total_steps + 1);
  // ---- workspace
  Arena a;
  const size_t o_xn = a.take(static_cast<size_t>(M) * d * 2), o_encp = a.take(static_cast<size_t>(M) * Hj * 4);
  const size_t plane_cols = static_cast<size_t>(3 * Hj > 6 * Hp ? 3 * Hj : 6 * Hp);
  const size_t o_planes = a.take(static_cast<size_t>(R) * plane_cols * 2), o_logits = a.take(static_cast<size_t>(R) * n_pad * 4);
  const size_t o_gates = a.take(static_cast<size_t>(R) * 4 * Hp * 4), o_pp = a.take(static_cast<size_t>(R) * Hj * 4);
  const size_t state_bytes = rs::alsd_state_bytes(B, beam, Hp, Hj, max_nodes);
  const size_t o_state = a.take(state_bytes);
  const size_t need_bytes = a.off;
  if (need_bytes > e->alsd_ws_bytes) {
    RS_CUDA(e, cudaStreamSynchronize(s));
    cudaFree(e->alsd_ws); e->alsd_ws = nullptr; e->alsd_ws_bytes = 0;
    RS_CUDA(e, cudaMalloc(&e->alsd_ws, need_bytes));
    e->alsd_ws_bytes = need_bytes;
  }
  if (e->alsd_done_host == nullptr) RS_CUDA(e, cudaMallocHost(reinterpret_cast<void**>(&e->alsd_done_host), sizeof(int)));
  char* ws = static_cast<char*>(e->alsd_ws);
  void* xn = ws + o_xn; float* encp = reinterpret_cast<float*>(ws + o_encp); void* planes = ws + o_planes;
  float* logits = reinterpret_cast<float*>(ws + o_logits); float* gates = reinterpret_cast<float*>(ws + o_gates); float* ppn = reinterpret_cast<float*>(ws + o_pp);
  RS_CUDA(e, cudaMemsetAsync(ws + o_state, 0, state_bytes, s));
  rs::AlsdState st{};
  rs::alsd_bind_state(st, ws + o_state, B, beam, Hp, Hj, max_nodes, score_norm != 0);
  // ---- joint.enc over every frame (as in the greedy path)
  RS_K(e, s, rs::launch_f32_to_bf16(enc, xn, static_cast<int64_t>(M) * d, s), 1);
  RS_TRY(gemm(e, xn, e->dec.enc_w, e->dec.enc_b, nullptr, encp, M, Hj, d, RS_EPI_BIAS_F32, 1.f, s));
  // predictor of the extended hypotheses of the beam being built (also the start: [blank] from the zero state)
  auto predictor = [&]() -> int {
    RS_K(e, s, rs::alsd_launch_lstm_in(st, B, e->dec.embed, Hp, planes, s), 1);
    RS_TRY(gemm(e, planes, e->alsd.lstm_w3, e->dec.lstm_b, nullptr, gates, R, 4 * Hp, 6 * Hp, RS_EPI_BIAS_F32, 1.f, s));
    RS_K(e, s, rs::alsd_launch_cell(st, B, gates, Hp, planes, s), 1);
    RS_TRY(gemm(e, planes, e->alsd.pred_w3, e->dec.pred_b, nullptr, ppn, R, Hj, 3 * Hp, RS_EPI_BIAS_F32, 1.f, s));
    RS_K(e, s, rs::alsd_launch_commit(st, B, ppn, Hp, Hj, s), 2);
    return RS_OK;
  };
  RS_K(e, s, rs::alsd_launch_init(st, B, blank, s), 1);
  RS_TRY(predictor());
  for (int step = 0; step <= total_steps; ++step) {
    RS_K(e, s, rs::alsd_launch_rows(st, B, encp, enc_len, T_max, Hj, step, planes, s), 1);
    RS_TRY(gemm(e, planes, e->alsd.out_w3, e->alsd.out_b, nullptr, logits, R, n_pad, 3 * Hj, RS_EPI_BIAS_F32, 1.f, s));
    RS_K(e, s, rs::alsd_launch_reduce(st, B, logits, n_pad, V, s), 1);
    RS_K(e, s, rs::alsd_launch_select(st, B, enc_len, step, blank, u_max_ratio, recombine_returns_input != 0, s), 1);
    RS_TRY(predictor());
    if ((step & 31) == 31) {
      RS_CUDA(e, cudaMemcpyAsync(e->alsd_done_host, st.n_done, sizeof(int), cudaMemcpyDeviceToHost, s));
      RS_CUDA(e, cudaStreamSynchronize(s));
      if (*e->alsd_done_host >= B) break;
    }
  }
  RS_K(e, s, rs::alsd_launch_output(st, B, blank, y_dev, step_dev, n_dev, score_dev, U_cap, s), 1);
  RS_CUDA(e, cudaStreamSynchronize(s));
  return RS_OK;
}

int rs_resample_mono(rs_engine* e, const void* in_dev, int in_is_pcm16, const int32_t* len_in_dev, int B, int channels, int L_in_max,
                     const float* taps_dev, int taps_per_phase, int up, int down, int n_pre_remove, int pad, float* out_dev,
                     int L_out_row, int32_t* len_out_dev, void* stream) {
  if (!e || !in_dev || !len_in_dev || !taps_dev || !out_dev || !len_out_dev) return fail(e, RS_ERR_INVALID_ARG, "rs_resample_mono: bad arguments");
  RS_CUDA(e, cudaSetDevice(e->device));
  Nvtx range("rs::resample_mono");
  rs::ResampleArgs a{in_dev, in_is_pcm16 != 0, len_in_dev, B, channels, L_in_max, taps_dev, taps_per_phase, up, down, n_pre_remove, pad,
                     out_dev, L_out_row, len_out_dev};
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  RS_K(e, s, rs::launch_resample_mono(a, s), 1);
  return RS_OK;
}

int rs_gemm_bf16(rs_engine* e, const void* a, const void* w, const float* bias, const float* resid, void* out, int M,
                 int N, int K, int epilogue, float alpha, void* stream) {
  if (!e || !a || !w || !out) return fail(e, RS_ERR_INVALID_ARG, "rs_gemm_bf16: bad arguments");
  RS_CUDA(e, cudaSetDevice(e->device));
  return gemm(e, a, w, bias, resid, out, M, N, K, epilogue, alpha, static_cast<cudaStream_t>(stream));
}

int rs_layernorm(rs_engine* e, const float* x, const float* gamma, const float* beta, float* out_f32, void* out_bf16,
                 int rows, int d, void* stream) {
  if (!e || !x || !gamma || !beta) return fail(e, RS_ERR_INVALID_ARG, "rs_layernorm: bad arguments");
  RS_CUDA(e, cudaSetDevice(e->device));
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  RS_K(e, s, rs::launch_layernorm(x, gamma, beta, out_f32, out_bf16, nullptr, nullptr, rows, d, e->cfg.ln_eps, s), 1);
  return RS_OK;
}

int64_t rs_launch_count(const rs_engine* e) { return e ? e->launches : 0; }

int rs_enable_stage_timing(rs_engine* e, int on) {
  if (!e) return RS_ERR_INVALID_ARG;
  e->timing = on != 0;
  return RS_OK;
}

// Stages: [0] log-mel, [1] subsampling, [2] conformer layers, [3] f32->bf16 + joint.enc GEMM, [4] greedy decode.
int rs_stage_times_ms(const rs_engine* e, float* ms) {
  if (!e || !ms || !e->ev_ok) return RS_ERR_INVALID_ARG;
  for (int i = 0; i < 8; ++i) ms[i] = 0.f;
  if (cudaEventSynchronize(e->ev[5]) != cudaSuccess) return RS_ERR_CUDA;
  for (int i = 0; i < 5; ++i) cudaEventElapsedTime(&ms[i], e->ev[i], e->ev[i + 1]);
  return RS_OK;
}

// Debug: cycle counters of the batched decode kernel's CTA 0 from the last rs_transcribe_* call for (B, L_max):
// phase J, barrier, token reduce, phase L, barrier, phase P, barrier, iterations.  Synchronises the device.
int rs_debug_decode_cycles(rs_engine* e, int B, int L_max, int U_max, int64_t* out8) {
  if (!e || !out8) return RS_ERR_INVALID_ARG;
  Plan p = make_plan(e, B, L_max, U_max);
  RS_CUDA(e, cudaDeviceSynchronize());
  const size_t off = p.dec_ws + rs::rnnt_spec_prof_offset(B, e->cfg.joint_hidden, e->cfg.pred_hidden);
  RS_CUDA(e, cudaMemcpy(out8, static_cast<char*>(e->ws) + off, 96, cudaMemcpyDeviceToHost));
  return RS_OK;
}

int rs_enable_kernel_timing(rs_engine* e, int on) {
  if (!e) return RS_ERR_INVALID_ARG;
  e->kernel_log.on = on != 0;
  e->kernel_log.clear();
  return RS_OK;
}

// Text summary "name\tcount\ttotal_ms\n..." of every launch since rs_enable_kernel_timing(e, 1); resets the log.
int rs_kernel_timing(rs_engine* e, char* buf, int buf_bytes) {
  if (!e || !buf || buf_bytes <= 0) return RS_ERR_INVALID_ARG;
  RS_CUDA(e, cudaDeviceSynchronize());
  std::map<std::string, std::pair<int, double>> agg;
  const EventLog& log = e->kernel_log;
  for (size_t i = 0; i < log.entries.size(); ++i) {
    auto& a = agg[log.entries[i].first];
    a.first += 1; a.second += log.ms(i);
  }
  std::string out;
  char line[160];
  for (const auto& kv : agg) {
    snprintf(line, sizeof line, "%s\t%d\t%.4f\n", kv.first.c_str(), kv.second.first, kv.second.second);
    out += line;
  }
  snprintf(buf, static_cast<size_t>(buf_bytes), "%s", out.c_str());
  e->kernel_log.clear();
  return RS_OK;
}

int rs_debug_attention_cycles(rs_engine* e, int64_t* out16) {
  if (!e || !out16) return RS_ERR_INVALID_ARG;
  RS_CUDA(e, cudaDeviceSynchronize());
  RS_CUDA(e, rs::attention_tc_debug_cycles(reinterpret_cast<long long*>(out16)));
  return RS_OK;
}

int rs_debug_gemm_cycles(rs_engine* e, int64_t* out64) {
  if (!e || !out64) return RS_ERR_INVALID_ARG;
  RS_CUDA(e, cudaDeviceSynchronize());
  RS_CUDA(e, rs::gemm_debug_cycles(reinterpret_cast<long long*>(out64)));
  return RS_OK;
}

int rs_enable_gemm_timing(rs_engine* e, int on) {
  if (!e) return RS_ERR_INVALID_ARG;
  e->gemm_log.on = on != 0;
  e->gemm_log.clear();
  return RS_OK;
}

int rs_gemm_timing(rs_engine* e, double* ms, double* flops, int64_t* launches) {
  if (!e || !ms || !flops || !launches) return RS_ERR_INVALID_ARG;
  EventLog& log = e->gemm_log;
  const size_t n = log.entries.size();
  if (n > 0) RS_CUDA(e, cudaEventSynchronize(log.ev[2 * n - 1]));
  double total = 0.0, total_flops = 0.0;
  for (size_t i = 0; i < n; ++i) { total += log.ms(i); total_flops += log.entries[i].second; }
  *ms = total; *flops = total_flops; *launches = static_cast<int64_t>(n);
  log.clear();
  return RS_OK;
}

}  // extern "C"
