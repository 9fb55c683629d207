"""The engine's measurement seams: GEMM timing, per-kernel timing and the launch counter.

bench.py reports GEMM launches and FLOPs, the per-kernel time map and `gpu_launches` through these calls, so their
counts are pinned here for one tiny-config call of the device-resident path, and the host-buffer entry point's launch
count is tied to the device entry's (its chunked copies add one log-mel and one subsampling launch per extra chunk).
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from reazonspeech_b200.config import conv_out_len
from reazonspeech_b200.synth import synth_clip


def _batch(B):
    waves = [np.pad(synth_clip(300 + i, 0.6 + 0.29 * (i % 5)), 8000) for i in range(B)]
    L = max(len(w) for w in waves)
    x = torch.zeros(B, L, dtype=torch.float32)
    for i, w in enumerate(waves):
        x[i, : len(w)] = torch.from_numpy(w)
    return x, torch.tensor([len(w) for w in waves], dtype=torch.int32)


def _gemm_shapes(cfg, B, L):
    """(M, N, K) of every GEMM of one transcribe call, in launch order."""
    F_max = L // cfg.n_window_stride + 1
    T2 = conv_out_len(conv_out_len(F_max))
    T3 = (conv_out_len(T2) + 7) & ~7                  # frame capacity: a multiple of 8
    F2, F3 = conv_out_len(conv_out_len(cfg.n_mels)), cfg.sub_freq
    C, d, ff, M = cfg.sub_channels, cfg.d_model, cfg.d_ff, B * T3
    shapes = [(B * T2 * F2, C, C), (B * T3 * F3, C, C), (M, d, F3 * C)]
    for _ in range(cfg.n_layers):
        shapes += [(M, ff, d), (M, d, ff), (M, 3 * d, d), (M, d, d), (M, 2 * d, d), (M, d, d), (M, ff, d), (M, d, ff)]
    return shapes + [(M, cfg.joint_hidden, d)]


# Per-kernel launch map of one tiny-config transcribe_device call (n_layers = 2, one global token).  The names are the
# keys bench.py's kernel_ms reports and looks up.
KERNEL_LAUNCHES = {
    "launch_logmel_fused": 1, "cudaGetLastError": 1, "launch_sub_conv0_dw1": 1, "launch_sub_dw": 1,
    "gemm N=64 K=64 epi=1": 2, "gemm N=256 K=640 epi=5": 1,
    "launch_layernorm": 9, "gemm N=1024 K=256 epi=2": 4, "gemm N=256 K=1024 epi=4": 4, "gemm N=768 K=256 epi=7": 2,
    "launch_attention_tc": 2, "gemm N=256 K=256 epi=4": 4, "gemm N=512 K=256 epi=3": 2, "launch_conv_dw": 2,
    "launch_zero_pad_rows": 1, "launch_f32_to_bf16": 1, "gemm N=128 K=256 epi=5": 1, "launch_rnnt_greedy_spec": 1,
}


def test_gemm_timing_counts_every_encoder_and_joint_gemm(tiny_engine, tiny_cfg):
    eng = tiny_engine
    x, lens = _batch(4)
    B, L = x.shape
    x, lens = x.cuda(), lens.cuda()
    eng.transcribe_device(x, lens)                     # warm-up, untimed
    torch.cuda.synchronize()
    eng.enable_gemm_timing(True)
    try:
        eng.transcribe_device(x, lens)
        torch.cuda.synchronize()
        ms, flops, n = eng.gemm_timing()
    finally:
        eng.enable_gemm_timing(False)
    shapes = _gemm_shapes(tiny_cfg, B, L)
    assert n == len(shapes) == 3 + 8 * tiny_cfg.n_layers + 1
    assert flops == sum(2.0 * M * N * K for M, N, K in shapes)
    assert ms > 0
    assert eng.gemm_timing() == (0.0, 0.0, 0)           # reading resets the accumulators


def test_kernel_timing_names_and_launches(tiny_engine):
    eng = tiny_engine
    x, lens = _batch(4)
    x, lens = x.cuda(), lens.cuda()
    eng.transcribe_device(x, lens)
    torch.cuda.synchronize()
    eng.kernel_timing(True)
    try:
        eng.transcribe_device(x, lens)
        got = eng.kernel_timing()
    finally:
        eng.kernel_timing(False)
    assert {k: n for k, (n, _) in got.items()} == KERNEL_LAUNCHES
    assert all(math.isfinite(ms) and ms >= 0 for _, ms in got.values())
    assert eng.kernel_timing() == {}                   # reading resets the log


def test_kernel_timing_of_a_stage_call_on_a_side_stream(tiny_engine, tiny_cfg):
    eng = tiny_engine
    d = tiny_cfg.d_model
    xr = torch.randn(300, d, device="cuda")
    g, b = torch.ones(d, device="cuda"), torch.zeros(d, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    eng.kernel_timing(True)
    try:
        with torch.cuda.stream(side):
            eng.layernorm(xr, g, b)
        got = eng.kernel_timing()
    finally:
        eng.kernel_timing(False)
    torch.cuda.synchronize()
    assert set(got) == {"launch_layernorm"}
    n, ms = got["launch_layernorm"]
    assert n == 1 and math.isfinite(ms) and ms >= 0


@pytest.mark.parametrize("B,chunks", [(8, 1), (16, 8), (19, 7)])
def test_host_entry_launches_match_device_entry(tiny_engine, B, chunks):
    """transcribe_host copies in ceil(B / 8)-utterance chunks once B >= 16; every extra chunk adds one log-mel and one
    subsampling-conv launch, nothing else."""
    eng = tiny_engine
    x, lens = _batch(B)
    xd, ld = x.cuda(), lens.cuda()
    xh = x.pin_memory()
    eng.transcribe_device(xd, ld)
    eng.transcribe_host(xh, lens)
    n0 = eng.launch_count
    eng.transcribe_device(xd, ld)
    n1 = eng.launch_count
    eng.transcribe_host(xh, lens)
    n2 = eng.launch_count
    torch.cuda.synchronize()
    assert (n2 - n1) == (n1 - n0) + 2 * (chunks - 1)
