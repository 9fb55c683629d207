"""ctypes binding of librs_engine.so (include/rs_engine.h) + weight packing.

PyTorch is used for device memory, streams and the one-time weight repack only; every
operation on the inference path is a hand-written sm_100a kernel behind the C ABI.  There
is deliberately no CPU or eager-PyTorch fallback: if the library or a B200 is missing the
constructors raise.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .config import ModelConfig, conv_out_len, xscale
from .logmel_tables import logmel_tables
from .weights import StateDict, rel_pos_table

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "librs_engine.so")

EPI_BIAS_BF16, EPI_BIAS_RELU_BF16, EPI_BIAS_SWISH_BF16, EPI_BIAS_GLU_BF16, EPI_RESID_F32, EPI_BIAS_F32, EPI_BIAS_F16 = range(7)


class RsModelConfig(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_int32), ("n_window_size", C.c_int32), ("n_window_stride", C.c_int32),
        ("n_fft", C.c_int32), ("n_mels", C.c_int32),
        ("preemph", C.c_float), ("log_zero_guard", C.c_float), ("norm_eps", C.c_float),
        ("n_layers", C.c_int32), ("d_model", C.c_int32), ("n_heads", C.c_int32), ("d_ff", C.c_int32),
        ("conv_kernel", C.c_int32), ("sub_channels", C.c_int32),
        ("att_left", C.c_int32), ("att_right", C.c_int32), ("global_tokens", C.c_int32),
        ("xscale", C.c_float), ("ln_eps", C.c_float),
        ("vocab_size", C.c_int32), ("pred_hidden", C.c_int32), ("joint_hidden", C.c_int32), ("max_symbols", C.c_int32),
    ]


class RsTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("dev_ptr", C.c_void_p), ("dtype", C.c_int32), ("numel", C.c_int64)]


_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.int32: 2}
_lib = None

_vp, _ip, _i64, _f32, _f64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
_P = C.POINTER
_XCRIBE = [_vp, _vp, _vp, _ip, _ip, _vp, _vp, _vp, _ip, _vp]       # the four rs_transcribe_* entry points
# ctypes signature of every C-ABI entry point (include/rs_engine.h): name -> (restype, argtypes)
SIGNATURES = {
    "rs_engine_create": (_ip, [_P(RsModelConfig), _P(RsTensor), _ip, _ip, _P(_vp)]),
    "rs_engine_destroy": (None, [_vp]),
    "rs_last_error": (C.c_char_p, [_vp]),
    "rs_workspace_bytes": (_ip, [_vp, _ip, _ip, _P(C.c_size_t)]),
    "rs_set_workspace": (_ip, [_vp, _vp, C.c_size_t]),
    "rs_mel_frames": (_ip, [_vp, _ip]),
    "rs_enc_frames": (_ip, [_vp, _ip]),
    "rs_mel_valid": (_ip, [_vp, _ip]),
    "rs_enc_valid": (_ip, [_vp, _ip]),
    "rs_logmel": (_ip, [_vp, _vp, _vp, _ip, _ip, _vp, _vp, _vp]),
    "rs_encode": (_ip, [_vp, _vp, _vp, _ip, _ip, _vp, _vp, _ip, _vp]),
    "rs_rnnt_greedy": (_ip, [_vp, _vp, _vp, _ip, _ip, _vp, _vp, _vp, _ip, _vp]),
    "rs_transcribe_device": (_ip, _XCRIBE),
    "rs_transcribe_batch": (_ip, _XCRIBE),
    "rs_transcribe_device_pcm16": (_ip, _XCRIBE),
    "rs_transcribe_batch_pcm16": (_ip, _XCRIBE),
    "rs_resample_mono": (_ip, [_vp, _vp, _ip, _vp, _ip, _ip, _ip, _vp, _ip, _ip, _ip, _ip, _ip, _vp, _ip, _vp, _vp]),
    "rs_rnnt_alsd": (_ip, [_vp, _vp, _vp, _ip, _ip, _ip, _f32, _ip, _ip, _vp, _vp, _vp, _vp, _ip, _vp]),
    "rs_rnnt_align": (_ip, [_vp, _vp, _vp, _ip, _ip, _vp, _vp, _ip, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rs_rnnt_align_spans": (_ip, [_vp, _vp, _vp, _ip, _ip, _ip, _vp, _vp, _vp, _ip, _vp, _vp, _vp, _ip, _vp, _vp, _vp, _vp]),
    "rs_gemm_bf16": (_ip, [_vp, _vp, _vp, _vp, _vp, _vp, _ip, _ip, _ip, _ip, _f32, _vp]),
    "rs_layernorm": (_ip, [_vp, _vp, _vp, _vp, _vp, _vp, _ip, _ip, _vp]),
    "rs_launch_count": (_i64, [_vp]),
    "rs_enable_stage_timing": (_ip, [_vp, _ip]),
    "rs_stage_times_ms": (_ip, [_vp, _P(_f32)]),
    "rs_enable_gemm_timing": (_ip, [_vp, _ip]),
    "rs_gemm_timing": (_ip, [_vp, _P(_f64), _P(_f64), _P(_i64)]),
    "rs_debug_decode_cycles": (_ip, [_vp, _ip, _ip, _ip, _P(_i64)]),
    "rs_enable_kernel_timing": (_ip, [_vp, _ip]),
    "rs_kernel_timing": (_ip, [_vp, C.c_char_p, _ip]),
    "rs_debug_attention_cycles": (_ip, [_vp, _P(_i64)]),
    "rs_debug_gemm_cycles": (_ip, [_vp, _P(_i64)]),
    "rs_stage_rows": (_ip, [_vp, _i64, _P(_vp), _P(_i64), _P(C.c_int32), _ip, _ip, _i64, _ip]),
}
EXPORTS = list(SIGNATURES)


def load_library(build_if_missing: bool = True) -> C.CDLL:
    """dlopen librs_engine.so (building it with nvcc first if it is absent and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        if not build_if_missing:
            raise FileNotFoundError(_LIB_PATH)
        from .build import build
        build()
    lib = C.CDLL(_LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib


# --------------------------------------------------------------------------------------
# Weight packing (NeMo state dict -> the engine's named device tensors)
# --------------------------------------------------------------------------------------
def glu_interleave_index(d: int) -> torch.Tensor:
    """Row permutation of pointwise_conv1 so that each 32-column GEMM chunk holds 16 value rows
    followed by their 16 gate rows (RS_EPI_BIAS_GLU_BF16)."""
    blk = torch.arange(d // 16).repeat_interleave(32)
    within = torch.arange(32).repeat(d // 16)
    return torch.where(within < 16, blk * 16 + within, d + blk * 16 + within - 16)


def pack_weights(sd: StateDict, cfg: ModelConfig) -> Dict[str, torch.Tensor]:
    """NeMo-named fp32 state dict -> packed host tensors (bf16 GEMM weights, folded BN, ...)."""
    bf = lambda t: t.to(torch.bfloat16).contiguous()
    f32 = lambda t: t.to(torch.float32).contiguous()
    out: Dict[str, torch.Tensor] = dict(logmel_tables(cfg))
    d, H, dk, Cc = cfg.d_model, cfg.n_heads, cfg.d_head, cfg.sub_channels
    pe = "encoder.pre_encode."
    out["sub.conv0.w"] = f32(sd[pe + "conv.0.weight"].reshape(Cc, 9)); out["sub.conv0.b"] = f32(sd[pe + "conv.0.bias"])
    out["sub.dw1.w"] = f32(sd[pe + "conv.2.weight"].reshape(Cc, 9)); out["sub.dw1.b"] = f32(sd[pe + "conv.2.bias"])
    out["sub.pw1.w"] = bf(sd[pe + "conv.3.weight"].reshape(Cc, Cc)); out["sub.pw1.b"] = f32(sd[pe + "conv.3.bias"])
    out["sub.dw2.w"] = f32(sd[pe + "conv.5.weight"].reshape(Cc, 9)); out["sub.dw2.b"] = f32(sd[pe + "conv.5.bias"])
    out["sub.pw2.w"] = bf(sd[pe + "conv.6.weight"].reshape(Cc, Cc)); out["sub.pw2.b"] = f32(sd[pe + "conv.6.bias"])
    F3 = cfg.sub_freq
    # NeMo flattens [C, F3] channel-major (index c*F3+f); the engine's activations are [F3, C]
    out["sub.out.w"] = bf(sd[pe + "out.weight"].view(d, Cc, F3).permute(0, 2, 1).reshape(d, F3 * Cc))
    out["sub.out.b"] = f32(sd[pe + "out.bias"])
    table = rel_pos_table(cfg)
    glu_idx = glu_interleave_index(d)
    for i in range(cfg.n_layers):
        p, o = f"encoder.layers.{i}.", f"L{i}."
        for src, dst in (("norm_feed_forward1", "ln_ff1"), ("norm_self_att", "ln_att"), ("norm_conv", "ln_conv"),
                         ("norm_feed_forward2", "ln_ff2"), ("norm_out", "ln_out")):
            out[o + dst + ".g"] = f32(sd[p + src + ".weight"]); out[o + dst + ".b"] = f32(sd[p + src + ".bias"])
        for src, dst in (("feed_forward1", "ff1"), ("feed_forward2", "ff2")):
            out[o + dst + ".w1"] = bf(sd[p + src + ".linear1.weight"]); out[o + dst + ".b1"] = f32(sd[p + src + ".linear1.bias"])
            out[o + dst + ".w2"] = bf(sd[p + src + ".linear2.weight"]); out[o + dst + ".b2"] = f32(sd[p + src + ".linear2.bias"])
        a = p + "self_attn."
        out[o + "att.wqkv"] = bf(torch.cat([sd[a + "linear_q.weight"], sd[a + "linear_k.weight"], sd[a + "linear_v.weight"]], 0))
        # the q columns of the projection carry q + pos_bias_u (the content term (q+u).k is then a plain Q'K^T for the
        # tensor cores); the positional term and the global token, which want q + pos_bias_v resp. q, get u taken out again
        # through their own bias / in their own kernel
        u_flat = sd[a + "pos_bias_u"].reshape(-1)
        out[o + "att.bqkv"] = f32(torch.cat([sd[a + "linear_q.bias"] + u_flat, sd[a + "linear_k.bias"], sd[a + "linear_v.bias"]], 0))
        pos = torch.nn.functional.linear(table, sd[a + "linear_pos.weight"])          # input independent: once at load
        n_rel_pad = (cfg.n_rel + 31) // 32 * 32
        pos_h = torch.zeros(H, n_rel_pad, dk)
        pos_h[:, : cfg.n_rel] = pos.view(cfg.n_rel, H, dk).permute(1, 0, 2)
        out[o + "att.pos"] = bf(pos_h)                                                 # operand of the attention kernel's positional UMMA
        # (q + v).p = (q + u).p + (v - u).p: the second term is input independent -> the GEMM's bias
        out[o + "att.bdbias"] = f32((out[o + "att.pos"].float() * (sd[a + "pos_bias_v"] - sd[a + "pos_bias_u"])[:, None, :]).sum(-1).reshape(-1))
        out[o + "att.u"] = f32(sd[a + "pos_bias_u"].reshape(-1))
        out[o + "att.wo"] = bf(sd[a + "linear_out.weight"]); out[o + "att.bo"] = f32(sd[a + "linear_out.bias"])
        c = p + "conv."
        out[o + "conv.pw1.w"] = bf(sd[c + "pointwise_conv1.weight"][:, :, 0][glu_idx])
        out[o + "conv.pw1.b"] = f32(sd[c + "pointwise_conv1.bias"][glu_idx])
        s = sd[c + "batch_norm.weight"] / torch.sqrt(sd[c + "batch_norm.running_var"] + cfg.bn_eps)
        out[o + "conv.dw.w"] = f32((sd[c + "depthwise_conv.weight"][:, 0, :] * s[:, None]).T)
        out[o + "conv.dw.shift"] = f32((sd[c + "depthwise_conv.bias"] - sd[c + "batch_norm.running_mean"]) * s + sd[c + "batch_norm.bias"])
        out[o + "conv.pw2.w"] = bf(sd[c + "pointwise_conv2.weight"][:, :, 0]); out[o + "conv.pw2.b"] = f32(sd[c + "pointwise_conv2.bias"])
    l = "decoder.prediction.dec_rnn.lstm."
    out["joint.enc.w"] = bf(sd["joint.enc.weight"]); out["joint.enc.b"] = f32(sd["joint.enc.bias"])
    out["joint.out.w"] = bf(sd["joint.joint_net.2.weight"]); out["joint.out.b"] = f32(sd["joint.joint_net.2.bias"])
    out["pred.embed"] = f32(sd["decoder.prediction.embed.weight"])
    out["pred.lstm.w"] = bf(torch.cat([sd[l + "weight_ih_l0"], sd[l + "weight_hh_l0"]], 1))
    out["pred.lstm.b"] = f32(sd[l + "bias_ih_l0"] + sd[l + "bias_hh_l0"])
    # the input half of the LSTM gates is a function of the token alone: one row per token (decode_spec.cu), from the same
    # bf16-rounded W_ih the kernels multiply with, accumulated in fp32
    w_ih = sd[l + "weight_ih_l0"].to(torch.bfloat16).to(torch.float32)
    out["pred.gate_tab"] = f32(out["pred.embed"] @ w_ih.T + out["pred.lstm.b"])
    out["joint.pred.w"] = bf(sd["joint.pred.weight"]); out["joint.pred.b"] = f32(sd["joint.pred.bias"])
    return out


def alsd_tensors(packed: Dict[str, torch.Tensor], cfg: ModelConfig) -> Dict[str, torch.Tensor]:
    """Weights of the ALSD beam search (csrc/decode_alsd.cu): the predictor / joint matrices repeated three times along K, so
    that activations split into three bf16 terms (24 mantissa bits) meet bf16-exact weights -- fp32-accurate log-probabilities
    out of the bf16 tensor-core GEMM.  The output layer is padded to a multiple of 64 rows (zero rows, never read)."""
    nc, hj = cfg.vocab_size + 1, cfg.joint_hidden
    n_pad = (nc + 63) // 64 * 64
    w = torch.zeros(n_pad, hj, dtype=torch.bfloat16)
    w[:nc] = packed["joint.out.w"]
    b = torch.zeros(n_pad, dtype=torch.float32)
    b[:nc] = packed["joint.out.b"]
    return {"alsd.out.w3": torch.cat([w] * 3, dim=1).contiguous(), "alsd.out.b": b,
            "alsd.lstm.w3": torch.cat([packed["pred.lstm.w"]] * 3, dim=1).contiguous(),
            "alsd.pred.w3": torch.cat([packed["joint.pred.w"]] * 3, dim=1).contiguous()}


def resample_taps(orig_sr: int, target_sr: int):
    """The polyphase FIR of ``scipy.signal.resample_poly(x, up, down)`` (its default Kaiser-5 window design, restated here
    step by step) in the layout rs_resample_mono wants: (taps float32 [up, taps_per_phase], up, down, n_pre_remove).
    out[m] = sum_j taps[phase][j] * x[n_hi - j] with t = (m + n_pre_remove) * down, n_hi = t // up, phase = t % up."""
    from math import gcd
    from scipy.signal import firwin
    g = gcd(int(orig_sr), int(target_sr))
    up, down = int(target_sr) // g, int(orig_sr) // g
    if up == down == 1:                                  # already at the target rate: the identity filter (down-mix / padding only)
        return torch.ones(1, 1, dtype=torch.float32), 1, 1, 0
    max_rate = max(up, down)
    half_len = 10 * max_rate
    h = (firwin(2 * half_len + 1, 1.0 / max_rate, window=("kaiser", 5.0)) * up).astype(np.float32)
    n_pre_pad = down - half_len % down
    n_pre_remove = (half_len + n_pre_pad) // down
    hp = np.concatenate((np.zeros(n_pre_pad, np.float32), h))
    per = (len(hp) + up - 1) // up
    taps = np.zeros((up, per), np.float32)
    for p in range(up):
        col = hp[p::up]
        taps[p, : len(col)] = col
    return torch.from_numpy(taps), up, down, n_pre_remove


def to_rs_config(cfg: ModelConfig) -> RsModelConfig:
    return RsModelConfig(
        cfg.sample_rate, cfg.n_window_size, cfg.n_window_stride, cfg.n_fft, cfg.n_mels,
        cfg.preemph, cfg.log_zero_guard, cfg.norm_eps,
        cfg.n_layers, cfg.d_model, cfg.n_heads, cfg.d_ff, cfg.conv_kernel, cfg.sub_channels,
        cfg.att_left, cfg.att_right, cfg.global_tokens, xscale(cfg), cfg.ln_eps,
        cfg.vocab_size, cfg.pred_hidden, cfg.joint_hidden, cfg.max_symbols)


# --------------------------------------------------------------------------------------
# Engine
# --------------------------------------------------------------------------------------
class Engine:
    """One engine per device: packed weights + workspace + the C-ABI handle."""

    def __init__(self, cfg: ModelConfig, state_dict: Optional[StateDict], device: str = "cuda", packed: Optional[Dict[str, torch.Tensor]] = None,
                 alsd: bool = False):
        """``packed``: the result of ``pack_weights(state_dict, cfg)`` when several engines share one checkpoint (one replica
        per device): the repack is done once, every engine uploads its own copy."""
        if not torch.cuda.is_available():
            raise RuntimeError("reazonspeech_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = load_library()
        self.cfg = cfg
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError(f"device {device!r}: the B200 engine has no CPU path")
        self.dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self.dev_index)
        if packed is None:
            packed = pack_weights(state_dict, cfg)
        if alsd and "alsd.out.w3" not in packed:             # beam search wanted: +34 MB of tripled predictor / joint weights
            packed = dict(packed, **alsd_tensors(packed, cfg))
        self.weights = {k: v.to(self.device) for k, v in packed.items()}
        self._names = [k.encode() for k in self.weights]
        arr = (RsTensor * len(self.weights))()
        for i, (k, v) in enumerate(self.weights.items()):
            arr[i] = RsTensor(self._names[i], v.data_ptr(), _DTYPES[v.dtype], v.numel())
        self._rs_cfg = to_rs_config(cfg)
        h = C.c_void_p()
        rc = self.lib.rs_engine_create(C.byref(self._rs_cfg), arr, len(self.weights), self.dev_index, C.byref(h))
        if rc != 0:
            raise RuntimeError(f"rs_engine_create failed ({rc}): {self.lib.rs_last_error(None).decode()}")
        self.h = h
        self._ws: Optional[torch.Tensor] = None
        self._ws_key: Tuple[int, int] = (0, 0)

    def __del__(self):
        h = getattr(self, "h", None)
        if h:
            self.lib.rs_engine_destroy(h)
            self.h = None

    # -- helpers
    def _check(self, rc: int, what: str):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {self.lib.rs_last_error(self.h).decode()}")

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def ensure_workspace(self, B: int, L_max: int):
        if self._ws is not None and B <= self._ws_key[0] and L_max <= self._ws_key[1]:
            return
        B2, L2 = max(B, self._ws_key[0]), max(L_max, self._ws_key[1])
        n = C.c_size_t()
        self._check(self.lib.rs_workspace_bytes(self.h, B2, L2, C.byref(n)), "rs_workspace_bytes")
        self._ws = None
        self._ws = torch.empty(n.value + 256, dtype=torch.uint8, device=self.device)
        ptr = (self._ws.data_ptr() + 255) // 256 * 256
        self._check(self.lib.rs_set_workspace(self.h, ptr, n.value), "rs_set_workspace")
        self._ws_key = (B2, L2)

    def mel_frames(self, n: int) -> int:
        return self.lib.rs_mel_frames(self.h, n)

    def enc_frames(self, n: int) -> int:
        return self.lib.rs_enc_frames(self.h, n)

    def u_max(self, L_max: int) -> int:
        return self.enc_frames(L_max) * self.cfg.max_symbols

    @property
    def launch_count(self) -> int:
        return int(self.lib.rs_launch_count(self.h))

    # -- stages (device tensors in, device tensors out)
    def log_mel(self, wav: torch.Tensor, lens: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        B, L = wav.shape
        assert wav.dtype == torch.float32 and wav.is_contiguous() and lens.dtype == torch.int32
        self.ensure_workspace(B, L)                  # the per-feature statistics are reduced in the workspace
        F = self.mel_frames(L)
        mel = torch.empty(B, F, self.cfg.n_mels, dtype=torch.float32, device=self.device)
        mel_len = torch.empty(B, dtype=torch.int32, device=self.device)
        self._check(self.lib.rs_logmel(self.h, wav.data_ptr(), lens.data_ptr(), B, L, mel.data_ptr(), mel_len.data_ptr(),
                                       self._stream()), "rs_logmel")
        return mel, mel_len

    def encode(self, mel: torch.Tensor, mel_len: torch.Tensor, n_layers: int = -1) -> Tuple[torch.Tensor, torch.Tensor]:
        B, F, _ = mel.shape
        L = (F - 1) * self.cfg.n_window_stride
        self.ensure_workspace(B, L)
        T = self.enc_frames(L)                       # capacity of the padded encoder tensors (a multiple of 8)
        enc = torch.empty(B, T, self.cfg.d_model, dtype=torch.float32, device=self.device)
        enc_len = torch.empty(B, dtype=torch.int32, device=self.device)
        self._check(self.lib.rs_encode(self.h, mel.data_ptr(), mel_len.data_ptr(), B, F, enc.data_ptr(), enc_len.data_ptr(),
                                       n_layers, self._stream()), "rs_encode")
        return enc, enc_len

    def greedy(self, enc: torch.Tensor, enc_len: torch.Tensor, U_max: Optional[int] = None):
        B, T, _ = enc.shape
        assert enc.dtype == torch.float32 and enc.is_contiguous()
        self.ensure_workspace(B, (T * 8 + 8) * self.cfg.n_window_stride)
        U = U_max or T * self.cfg.max_symbols
        tokens = torch.zeros(B, U, dtype=torch.int32, device=self.device)
        frames = torch.zeros(B, U, dtype=torch.int32, device=self.device)
        ntok = torch.zeros(B, dtype=torch.int32, device=self.device)
        self._check(self.lib.rs_rnnt_greedy(self.h, enc.data_ptr(), enc_len.data_ptr(), B, T, tokens.data_ptr(),
                                            frames.data_ptr(), ntok.data_ptr(), U, self._stream()), "rs_rnnt_greedy")
        return tokens, frames, ntok

    def transcribe_device(self, wav: torch.Tensor, lens: torch.Tensor, U_max: Optional[int] = None, out=None):
        B, L = wav.shape
        self.ensure_workspace(B, L)
        U = U_max or self.u_max(L)
        if out is None:
            out = (torch.zeros(B, U, dtype=torch.int32, device=self.device),
                   torch.zeros(B, U, dtype=torch.int32, device=self.device),
                   torch.zeros(B, dtype=torch.int32, device=self.device))
        tokens, frames, ntok = out
        assert wav.dtype in (torch.float32, torch.int16) and wav.is_contiguous()
        fn, name = ((self.lib.rs_transcribe_device_pcm16, "rs_transcribe_device_pcm16") if wav.dtype == torch.int16
                    else (self.lib.rs_transcribe_device, "rs_transcribe_device"))        # int16: PCM, scaled by 2^-15 on the device
        self._check(fn(self.h, wav.data_ptr(), lens.data_ptr(), B, L, tokens.data_ptr(), frames.data_ptr(), ntok.data_ptr(), U, self._stream()), name)
        return tokens, frames, ntok

    def transcribe_host(self, wav: torch.Tensor, lens: torch.Tensor, U_max: Optional[int] = None, out=None):
        """wav: host float32 or int16 (PCM) [B, L] (pinned for speed), lens: host int32 [B] -> host tokens/frames/n_tok."""
        B, L = wav.shape
        assert wav.device.type == "cpu" and wav.dtype in (torch.float32, torch.int16) and wav.is_contiguous()
        self.ensure_workspace(B, L)
        U = U_max or self.u_max(L)
        if out is None:
            out = (torch.zeros(B, U, dtype=torch.int32).pin_memory(), torch.zeros(B, U, dtype=torch.int32).pin_memory(),
                   torch.zeros(B, dtype=torch.int32).pin_memory())
        tokens, frames, ntok = out
        fn, name = ((self.lib.rs_transcribe_batch_pcm16, "rs_transcribe_batch_pcm16") if wav.dtype == torch.int16
                    else (self.lib.rs_transcribe_batch, "rs_transcribe_batch"))
        self._check(fn(self.h, wav.data_ptr(), lens.data_ptr(), B, L, tokens.data_ptr(), frames.data_ptr(), ntok.data_ptr(), U, self._stream()), name)
        return tokens, frames, ntok

    def alsd(self, enc: torch.Tensor, enc_len: torch.Tensor, beam: int = 4, u_max_ratio: float = 2.0, score_norm: bool = True,
             recombine_returns_input: bool = True, U_cap: Optional[int] = None):
        """ALSD beam search over encoder outputs -> (y [B, U_cap + 1] with the leading blank, steps [B, U_cap], n [B], score [B])."""
        B, T, _ = enc.shape
        assert enc.dtype == torch.float32 and enc.is_contiguous() and enc_len.dtype == torch.int32
        U = U_cap or (T + int(u_max_ratio * T) + 1)
        y = torch.zeros(B, U + 1, dtype=torch.int32, device=self.device)
        steps = torch.zeros(B, U, dtype=torch.int32, device=self.device)
        n = torch.zeros(B, dtype=torch.int32, device=self.device)
        score = torch.zeros(B, dtype=torch.float64, device=self.device)
        self._check(self.lib.rs_rnnt_alsd(self.h, enc.data_ptr(), enc_len.data_ptr(), B, T, int(beam), float(u_max_ratio), int(score_norm),
                                          int(recombine_returns_input), y.data_ptr(), steps.data_ptr(), n.data_ptr(), score.data_ptr(), U,
                                          self._stream()), "rs_rnnt_alsd")
        return y, steps, n, score

    def align(self, enc: torch.Tensor, enc_len: torch.Tensor, targets: torch.Tensor, tgt_len: torch.Tensor, lattice: bool = False):
        """RNN-T forced alignment of the given token sequences (needs the ``alsd.*`` tensors: ``Engine(..., alsd=True)``).
        enc f32 [B, T, d_model], enc_len i32 [B], targets i32 [B, U_max] (ids in [0, vocab_size)), tgt_len i32 [B] ->
        (frames i32 [B, U_max]: encoder frame of every token on the Viterbi path, tok_logp f32 [B, U_max]: its log p,
        viterbi f64 [B], loglik f64 [B]: the log-likelihood summed over all alignments = -RNN-T loss
        [, lattice f32 [B, T, U_max + 1, 2]: (log p(blank), log p(next target)) of every node]).  Synchronises."""
        B, T, _ = enc.shape
        assert enc.dtype == torch.float32 and enc.is_contiguous() and enc_len.dtype == torch.int32
        assert targets.dtype == torch.int32 and targets.is_contiguous() and targets.dim() == 2 and tgt_len.dtype == torch.int32
        U = targets.shape[1]
        frames = torch.empty(B, U, dtype=torch.int32, device=self.device)
        tok_logp = torch.empty(B, U, dtype=torch.float32, device=self.device)
        viterbi = torch.empty(B, dtype=torch.float64, device=self.device)
        loglik = torch.empty(B, dtype=torch.float64, device=self.device)
        lat = torch.empty(B, T, U + 1, 2, dtype=torch.float32, device=self.device) if lattice else None
        self._check(self.lib.rs_rnnt_align(self.h, enc.data_ptr(), enc_len.data_ptr(), B, T, targets.data_ptr(), tgt_len.data_ptr(), U,
                                           frames.data_ptr(), tok_logp.data_ptr(), viterbi.data_ptr(), loglik.data_ptr(),
                                           lat.data_ptr() if lattice else None, self._stream()), "rs_rnnt_align")
        return (frames, tok_logp, viterbi, loglik, lat) if lattice else (frames, tok_logp, viterbi, loglik)

    def align_spans(self, enc: torch.Tensor, enc_len: torch.Tensor, spans: torch.Tensor, targets: torch.Tensor, tgt_len: torch.Tensor,
                    lattice: bool = False):
        """Free-span RNN-T alignment (rs_rnnt_align_spans): find each of K token sequences somewhere inside a frame window of
        one encoder row (needs ``Engine(..., alsd=True)``).  enc f32 [B, T, d_model], enc_len i32 [B], spans i32 [K, 3]
        (src row, lo, hi), targets i32 [K, U_max] (ids in [0, vocab_size)), tgt_len i32 [K] (>= 1) -> (frames i32 [K, U_max]:
        absolute encoder frame of every token on the best path, tok_logp f32 [K, U_max], path_logp f32 [K, F_max]: per window
        frame t - lo, the path's log p at that frame (0 outside the span), viterbi f64 [K], loglik f64 [K]
        [, lattice f32 [K, F_max, U_max + 1, 2]]), F_max = max(hi - lo).  Synchronises."""
        B, T, _ = enc.shape
        assert enc.dtype == torch.float32 and enc.is_contiguous() and enc_len.dtype == torch.int32
        assert targets.dtype == torch.int32 and targets.is_contiguous() and targets.dim() == 2 and tgt_len.dtype == torch.int32
        assert spans.dtype == torch.int32 and spans.dim() == 2 and spans.shape[1] == 3 and spans.shape[0] == targets.shape[0]
        K, U = targets.shape
        F = max(1, int((spans[:, 2] - spans[:, 1]).max())) if K else 1
        spans = spans.to(self.device).contiguous()
        frames = torch.empty(K, U, dtype=torch.int32, device=self.device)
        tok_logp = torch.empty(K, U, dtype=torch.float32, device=self.device)
        path_logp = torch.empty(K, F, dtype=torch.float32, device=self.device)
        viterbi = torch.empty(K, dtype=torch.float64, device=self.device)
        loglik = torch.empty(K, dtype=torch.float64, device=self.device)
        lat = torch.empty(K, F, U + 1, 2, dtype=torch.float32, device=self.device) if lattice else None
        self._check(self.lib.rs_rnnt_align_spans(self.h, enc.data_ptr(), enc_len.data_ptr(), B, T, K, spans.data_ptr(), targets.data_ptr(),
                                                 tgt_len.data_ptr(), U, frames.data_ptr(), tok_logp.data_ptr(), path_logp.data_ptr(), F,
                                                 viterbi.data_ptr(), loglik.data_ptr(), lat.data_ptr() if lattice else None,
                                                 self._stream()), "rs_rnnt_align_spans")
        out = (frames, tok_logp, path_logp, viterbi, loglik)
        return out + (lat,) if lattice else out

    def resample_mono(self, raw: torch.Tensor, lens: torch.Tensor, samplerate: int, pad: int = 0):
        """norm_audio on the device (pkg/nemo-asr/src/audio.py:54-68) + transcribe()'s padding: ``raw`` [B, C, L] float32 or
        int16 (PCM) on this device at ``samplerate``, ``lens`` int32 [B] valid samples -> (wav float32 [B, L16] at 16 kHz mono
        with ``pad`` zeros on both sides of every utterance, lens int32 [B]); feed both to ``transcribe_device``."""
        assert raw.dim() == 3 and raw.is_contiguous() and raw.dtype in (torch.float32, torch.int16) and lens.dtype == torch.int32
        key = int(samplerate)
        if not hasattr(self, "_rs_taps"):
            self._rs_taps = {}
        if key not in self._rs_taps:
            taps, up, down, pre = resample_taps(key, self.cfg.sample_rate)
            self._rs_taps[key] = (taps.to(self.device), up, down, pre)
        taps, up, down, pre = self._rs_taps[key]
        B, Cn, L = raw.shape
        n_out = (L * up + down - 1) // down
        L16 = (n_out + 2 * pad + 3) & ~3
        out = torch.empty(B, L16, dtype=torch.float32, device=self.device)
        out_len = torch.empty(B, dtype=torch.int32, device=self.device)
        self._check(self.lib.rs_resample_mono(self.h, raw.data_ptr(), int(raw.dtype == torch.int16), lens.data_ptr(), B, Cn, L,
                                              taps.data_ptr(), taps.shape[1], up, down, pre, pad, out.data_ptr(), L16, out_len.data_ptr(),
                                              self._stream()), "rs_resample_mono")
        return out, out_len

    # -- kernel seams
    def gemm(self, a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], epilogue: int,
             resid: Optional[torch.Tensor] = None, alpha: float = 1.0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        M, K = a.shape
        N = w.shape[0]
        assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and a.is_contiguous() and w.is_contiguous()
        if out is None:
            if epilogue in (EPI_RESID_F32, EPI_BIAS_F32):
                out = torch.empty(M, N, dtype=torch.float32, device=self.device)
            elif epilogue == EPI_BIAS_F16:
                out = torch.empty(M, N, dtype=torch.float16, device=self.device)
            elif epilogue == EPI_BIAS_GLU_BF16:
                out = torch.empty(M, N // 2, dtype=torch.bfloat16, device=self.device)
            else:
                out = torch.empty(M, N, dtype=torch.bfloat16, device=self.device)
        self._check(self.lib.rs_gemm_bf16(self.h, a.data_ptr(), w.data_ptr(), bias.data_ptr() if bias is not None else None,
                                          resid.data_ptr() if resid is not None else None, out.data_ptr(), M, N, K,
                                          epilogue, alpha, self._stream()), "rs_gemm_bf16")
        return out

    def layernorm(self, x: torch.Tensor, g: torch.Tensor, b: torch.Tensor, bf16_out: bool = True) -> torch.Tensor:
        rows, d = x.shape
        out = torch.empty(rows, d, dtype=torch.bfloat16 if bf16_out else torch.float32, device=self.device)
        self._check(self.lib.rs_layernorm(self.h, x.data_ptr(), g.data_ptr(), b.data_ptr(),
                                          None if bf16_out else out.data_ptr(), out.data_ptr() if bf16_out else None,
                                          rows, d, self._stream()), "rs_layernorm")
        return out

    def enable_stage_timing(self, on: bool = True):
        self._check(self.lib.rs_enable_stage_timing(self.h, int(on)), "rs_enable_stage_timing")

    def kernel_timing(self, enable: Optional[bool] = None):
        """enable=True/False switches per-launch event timing; with None returns {name: (launches, total_ms)} and resets."""
        if enable is not None:
            self._check(self.lib.rs_enable_kernel_timing(self.h, int(enable)), "rs_enable_kernel_timing")
            return None
        buf = C.create_string_buffer(1 << 16)
        self._check(self.lib.rs_kernel_timing(self.h, buf, len(buf)), "rs_kernel_timing")
        out = {}
        for line in buf.value.decode().splitlines():
            name, n, ms = line.split("\t")
            out[name] = (int(n), float(ms))
        return out

    def attention_cycles(self):
        """clock64 stamps of CTA (1,0,0) of the last tensor-core attention launch, relative to its first stamp."""
        out = (C.c_int64 * 16)()
        self._check(self.lib.rs_debug_attention_cycles(self.h, out), "rs_debug_attention_cycles")
        v = list(out)
        names = ["start", "tma_issue", "qk_landed", "s_issued", "pv_wait", "pv_issued", "dealloc", "_",
                 "sm_start", "sm_gscore_done", "sm_s_ready", "sm_pass1", "sm_pass2", "sm_o_wait", "sm_o_ready", "sm_end"]
        return {n: int(x - v[0]) for n, x in zip(names, v) if n != "_"}

    def gemm_cycles(self):
        """Timeline (SM clocks relative to kernel entry) of the last 2-CTA GEMM launch, for its first and its last cluster.
        Only a library built with RS_BUILD_FLAGS=-DRS_PROF writes the stamps (scripts/diag_gemm_timeline.py); the shipped one
        returns whatever the buffer held (zeros)."""
        out = (C.c_int64 * 64)()
        self._check(self.lib.rs_debug_gemm_cycles(self.h, out), "rs_debug_gemm_cycles")
        res = {}
        for c, tag in enumerate(("first_cluster", "last_cluster")):
            v = list(out)[32 * c: 32 * c + 32]
            d = {"roles_start": v[0] - v[30], "end": v[31] - v[30]}
            for i in range(3):
                if v[3 + 4 * i] > v[30]:
                    d[f"tile{i}"] = {"acc_free": v[1 + 4 * i] - v[30], "operands": v[2 + 4 * i] - v[30], "mma_issued": v[3 + 4 * i] - v[30],
                                     "acc_full": v[4 + 4 * i] - v[30], "epilogue_done": v[16 + 2 * i] - v[30]}
            res[tag] = d
        return res

    def decode_cycles(self, B: int, L_max: int, U_max: int):
        out = (C.c_int64 * 12)()
        self._check(self.lib.rs_debug_decode_cycles(self.h, B, L_max, U_max, out), "rs_debug_decode_cycles")
        return dict(zip(("phase_j", "barrier_a", "reduce", "phase_l", "barrier_b", "phase_p", "barrier_c", "iterations", "j_loads", "j_rows", "j_misc", "_"), [int(v) for v in out]))

    def enable_gemm_timing(self, on: bool = True):
        self._check(self.lib.rs_enable_gemm_timing(self.h, int(on)), "rs_enable_gemm_timing")

    def gemm_timing(self):
        """(summed device ms, summed algorithmic FLOPs, launches) of the tcgen05 GEMM since enabled / last read."""
        ms, fl, n = C.c_double(), C.c_double(), C.c_int64()
        self._check(self.lib.rs_gemm_timing(self.h, C.byref(ms), C.byref(fl), C.byref(n)), "rs_gemm_timing")
        return ms.value, fl.value, n.value

    def stage_times_ms(self) -> Dict[str, float]:
        ms = (C.c_float * 8)()
        self._check(self.lib.rs_stage_times_ms(self.h, ms), "rs_stage_times_ms")
        return dict(zip(("logmel", "subsample", "layers", "enc_proj", "decode"), [float(v) for v in ms[:5]]))
