"""Forced-alignment benchmark: rs_rnnt_align on the 619 M synthetic model over bench.py's clip set (the same seeded 30 s clips,
0.5 s of silence on both sides), each clip's targets being its own greedy transcript.  Prints one JSON line: the GPU and its
power limit (read in the same run), ms per rs_rnnt_align call (the encoder excluded; CUDA events, the call synchronises),
the predictor / rows / lattice / DP split from the engine's per-kernel timing, the lattice node count, the lattice kernel's
achieved TFLOP/s (2 * nodes * n_pad * 3 * joint_hidden) and the align RTFx including log-mel and the encoder.

    python scripts/bench_align.py [--clips 32] [--seconds 30] [--steps 10] [--warmup 2]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PAD = 8000                                         # 0.5 s at 16 kHz, as transcribe() pads


def power_limit_w() -> float:
    out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout
    return float(out.strip().splitlines()[0])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=32)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_align.py measures the GPU path: no CUDA device")
    from reazonspeech_b200.config import ModelConfig
    from reazonspeech_b200.engine import Engine
    from reazonspeech_b200.synth import synth_clip
    from reazonspeech_b200.weights import random_state_dict

    cfg = ModelConfig()
    eng = Engine(cfg, random_state_dict(cfg, seed=0), "cuda:0", alsd=True)
    B = args.clips
    L = int(args.seconds * 16000) + 2 * PAD
    wav = torch.zeros(B, L)
    for i in range(B):
        wav[i, PAD:L - PAD] = torch.from_numpy(synth_clip(i, args.seconds))     # bench.make_batch, rank 0
    wav_dev = wav.cuda()
    len_dev = torch.full((B,), L, dtype=torch.int32, device="cuda")
    eng.ensure_workspace(B, L)

    def encode():
        mel, mel_len = eng.log_mel(wav_dev, len_dev)
        return eng.encode(mel, mel_len)

    enc, enc_len = encode()
    tokens, _, ntok = eng.greedy(enc, enc_len)
    U = max(1, int(ntok.max()))
    targets = tokens[:, :U].contiguous()
    tgt_len = ntok.clamp(max=U).to(torch.int32).contiguous()
    nodes = int((enc_len.long() * (tgt_len.long() + 1)).sum())

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(args.steps):
            fn()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / args.steps

    ms_align = timed(lambda: eng.align(enc, enc_len, targets, tgt_len))
    ms_e2e = timed(lambda: eng.align(*encode(), targets, tgt_len))
    eng.kernel_timing(True)
    eng.align(enc, enc_len, targets, tgt_len)
    kt = eng.kernel_timing()
    eng.kernel_timing(False)
    Hj, Hp, n_pad = cfg.joint_hidden, cfg.pred_hidden, (cfg.n_classes + 63) // 64 * 64
    pred_gemms = (f"gemm N={4 * Hp} K={6 * Hp} ", f"gemm N={Hj} K={3 * Hp} ")
    split = {"predictor": sum(ms for k, (_, ms) in kt.items() if k == "align_pred" or k.startswith(pred_gemms)),
             "rows": kt.get("align_rows", (0, 0.0))[1], "lattice": kt.get("align_lattice", (0, 0.0))[1],
             "dp": kt.get("align_dp", (0, 0.0))[1], "enc_proj": sum(ms for k, (_, ms) in kt.items() if k.startswith(f"gemm N={Hj} K={cfg.d_model} "))}
    flops = 2.0 * nodes * n_pad * 3 * Hj
    print(json.dumps({
        "metric": "rnnt_align", "gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
        "clips": B, "seconds": args.seconds, "tokens_per_clip": float(tgt_len.float().mean()), "lattice_nodes": nodes,
        "ms_per_align_call": ms_align, "kernel_ms": split, "lattice_launches": kt.get("align_lattice", (0, 0.0))[0],
        "lattice_tflops": flops / (split["lattice"] * 1e-3) / 1e12 if split["lattice"] > 0 else None,
        "lattice_tflop_per_call": flops / 1e12, "a_plane_gb_per_call": nodes * 3 * Hj * 2 / 1e9,
        "align_rtfx_with_encoder": B * args.seconds / (ms_e2e * 1e-3), "ms_per_step_with_encoder": ms_e2e,
        "kernels": {k: v for k, v in kt.items()},
    }))


if __name__ == "__main__":
    main()
