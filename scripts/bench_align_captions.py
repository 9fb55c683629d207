"""Caption-placement benchmark: rs_rnnt_align_spans on the 619 M synthetic model (seed 0) over one seeded 1800 s recording
(synth_clip(0, 1800), 0.5 s of silence on both sides), encoded once.  The engine's own greedy transcript of it is cut into
captions of 24 tokens; each caption's display time is its spoken time shifted later by a seeded delay in [0, 20] s, like a
live caption, and it is searched for from 25 s before its display start to its display end, as align_captions does.  The
transcript is decoded per 30 s piece of the recording (bench.py's clip length), its frames moved onto the recording's axis:
decoded in one piece, this untrained checkpoint emits only ~100 tokens in the whole 1800 s (~3 per 30 s piece instead of
~104), which would leave a handful of captions spread over minutes each.

Prints one JSON line: the GPU and its power limit (read in the same run); T, captions, mean tokens and window frames per
caption, lattice nodes; ms for log-mel and the encoder; ms per rs_rnnt_align_spans call (CUDA events, the call
synchronises) and its predictor / rows / lattice / DP split from the engine's per-kernel timing; the lattice kernel's
TFLOP/s (2 * nodes * n_pad * 3 * joint_hidden), captions per second and the RTFx of the whole caption pass (log-mel, encoder
and the span call).  "placement_within_2_frames" is the share of captions whose first aligned frame lies within 2 frames of
the greedy frame of that token: a property of the untrained synthetic checkpoint, reported, not a target.

    python scripts/bench_align_captions.py [--seconds 1800] [--tokens 24] [--steps 10] [--warmup 2]
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


def greedy_by_piece(eng, x, piece_s: float = 30.0):
    """Greedy transcript of a 16 kHz recording decoded per piece of piece_s seconds (each with 0.5 s of silence on both sides,
    as transcribe() pads), frames moved onto the axis of the whole recording encoded with the same padding."""
    import torch
    n = int(piece_s * 16000)
    pieces = [x[i:i + n] for i in range(0, x.shape[0], n)]
    L = n + 2 * PAD
    wav = torch.zeros(len(pieces), L, device=x.device)
    for i, p in enumerate(pieces):
        wav[i, PAD:PAD + p.shape[0]] = p
    lens = torch.tensor([p.shape[0] + 2 * PAD for p in pieces], dtype=torch.int32, device=x.device)
    mel, mel_len = eng.log_mel(wav, lens)
    enc, enc_len = eng.encode(mel, mel_len)
    tk, fr, nt = [a.cpu() for a in eng.greedy(enc, enc_len)]
    step = round(piece_s / 0.08)
    toks, frs = [], []
    for i in range(len(pieces)):
        toks += tk[i, : int(nt[i])].tolist()
        frs += [f + i * step for f in fr[i, : int(nt[i])].tolist()]
    return toks, frs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1800.0)
    ap.add_argument("--tokens", type=int, default=24)
    ap.add_argument("--before", type=float, default=25.0)
    ap.add_argument("--max-delay", type=float, default=20.0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_align_captions.py measures the GPU path: no CUDA device")
    from reazonspeech_b200.config import ModelConfig
    from reazonspeech_b200.engine import Engine
    from reazonspeech_b200.nemo.asr.transcribe import window_frames
    from reazonspeech_b200.synth import synth_clip
    from reazonspeech_b200.weights import random_state_dict

    cfg = ModelConfig()
    eng = Engine(cfg, random_state_dict(cfg, seed=0), "cuda:0", alsd=True)
    wav = torch.from_numpy(np.pad(synth_clip(0, args.seconds), PAD).astype(np.float32))[None].cuda()
    lens = torch.tensor([wav.shape[1]], dtype=torch.int32, device="cuda")

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

    mel, mel_len = eng.log_mel(wav, lens)
    enc, enc_len = eng.encode(mel, mel_len)
    T = int(enc_len[0])
    toks, frs = greedy_by_piece(eng, wav[0, PAD:-PAD])
    rng = np.random.default_rng(0)
    items = []                                               # (lo, hi, tokens, greedy frame of the first token)
    for i in range(0, len(toks), args.tokens):
        t, f = toks[i:i + args.tokens], frs[i:i + args.tokens]
        start = 0.08 * f[0] - 0.5
        end = 0.08 * f[-1] - 0.5 + 0.08
        delay = float(rng.uniform(0.0, args.max_delay))
        lo, hi = window_frames(start + delay - args.before, end + delay, T)
        items.append((lo, hi, t, f[0]))
    K = len(items)
    U = max(len(it[2]) for it in items)
    spans = torch.tensor([[0, lo, hi] for lo, hi, _, _ in items], dtype=torch.int32, device="cuda")
    targets = torch.zeros(K, U, dtype=torch.int32)
    for k, it in enumerate(items):
        targets[k, : len(it[2])] = torch.tensor(it[2], dtype=torch.int32)
    targets = targets.cuda()
    tgt_len = torch.tensor([len(it[2]) for it in items], dtype=torch.int32, device="cuda")
    nodes = sum((hi - lo) * (len(t) + 1) for lo, hi, t, _ in items)

    ms_logmel = timed(lambda: eng.log_mel(wav, lens))
    ms_encoder = timed(lambda: eng.encode(mel, mel_len))
    ms_spans = timed(lambda: eng.align_spans(enc, enc_len, spans, targets, tgt_len))

    def whole():
        m, ml = eng.log_mel(wav, lens)
        e, el = eng.encode(m, ml)
        return eng.align_spans(e, el, spans, targets, tgt_len)

    ms_whole = timed(whole)
    frames = eng.align_spans(enc, enc_len, spans, targets, tgt_len)[0].cpu()
    placed = sum(abs(int(frames[k, 0]) - it[3]) <= 2 for k, it in enumerate(items))
    eng.kernel_timing(True)
    eng.align_spans(enc, enc_len, spans, targets, tgt_len)
    kt = eng.kernel_timing()
    eng.kernel_timing(False)
    Hj, Hp, n_pad = cfg.joint_hidden, cfg.pred_hidden, (cfg.n_classes + 63) // 64 * 64
    pred_gemms = (f"gemm N={4 * Hp} K={6 * Hp} ", f"gemm N={Hj} K={3 * Hp} ")
    split = {"predictor": sum(ms for k, (_, ms) in kt.items() if k == "align_pred" or k.startswith(pred_gemms)),
             "rows": kt.get("align_rows", (0, 0.0))[1], "lattice": kt.get("align_lattice", (0, 0.0))[1],
             "dp": kt.get("align_dp", (0, 0.0))[1],
             "enc_proj": sum(ms for k, (_, ms) in kt.items() if k.startswith(f"gemm N={Hj} K={cfg.d_model} "))}
    flops = 2.0 * nodes * n_pad * 3 * Hj
    print(json.dumps({
        "metric": "rnnt_align_spans", "gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
        "seconds": args.seconds, "T": T, "transcript_tokens": len(toks), "captions": K, "tokens_per_caption": float(np.mean([len(it[2]) for it in items])),
        "window_frames_per_caption": float(np.mean([hi - lo for lo, hi, _, _ in items])), "lattice_nodes": nodes,
        "ms_log_mel": ms_logmel, "ms_encoder": ms_encoder, "ms_per_align_spans_call": ms_spans, "kernel_ms": split,
        "lattice_tflops": flops / (split["lattice"] * 1e-3) / 1e12 if split["lattice"] > 0 else None,
        "lattice_tflop_per_call": flops / 1e12, "captions_per_second": K / (ms_spans * 1e-3),
        "ms_caption_pass": ms_whole, "rtfx_caption_pass": args.seconds / (ms_whole * 1e-3),
        "placement_within_2_frames": placed / K,
        "placement_note": "property of the untrained synthetic checkpoint, not a quality target",
        "kernels": {k: v for k, v in kt.items()},
    }))


if __name__ == "__main__":
    main()
