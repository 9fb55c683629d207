#!/usr/bin/env python
"""Benchmark of the hot path: RTFx (nominal audio seconds / wall second) of the batched
FastConformer-RNNT 619 M transcribe path, BASELINE.json configs[1] per GPU
(32 clips x 30 s of synthetic 16 kHz audio -> 32 x 496000 samples after the 0.5 s pads).

    python bench.py --gpus N --steps K --warmup W            # this framework (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU (oracle port)

One JSON line on stdout (rank 0).  `value` times rs_transcribe_device with the waveforms already
resident in HBM; `e2e` times rs_transcribe_batch (the model.transcribe seam of the C ABI) with
pinned HOST buffers, H2D and D2H inside the timed region.  Weights are seeded random weights of the
619 M architecture (no checkpoint is reachable offline), data is synthetic; both are stated.

    python bench.py --steps K --dump-outputs DIR    # also write the last timed step's outputs as DIR/*.npy

The inputs depend on the arguments only, so two builds run with the same arguments can be compared
output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NOMINAL_SECONDS = 30.0
PAD = 8000
METRIC = "RTFx (audio-s/wall-s) FastConformer-RNNT 619M"
UNIT = "audio-s/wall-s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1407.1), d.get("bf16_tflops", 1691.8), d.get("hbm_gbs", 6564.5), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def python_api_rtfx(eng, n_clips: int, seconds: float, rank: int, batches: int = 4):
    """RTFx of the call a user of the drop-in makes: ``transcribe_batch(model, audios)`` from numpy clips to
    TranscribeResult objects (norm_audio, in-place padding into reused pinned staging, rs_transcribe_batch on a
    worker thread, decode_hypothesis of batch k while batch k+1 runs) -- SURVEY.md section 8d item (ii)."""
    from reazonspeech_b200.nemo.asr import TranscribeConfig, audio_from_numpy, transcribe_batch
    from reazonspeech_b200.nemo.asr.transcribe import B200RnntModel
    from reazonspeech_b200.synth import synth_clip
    from reazonspeech_b200.tokenizer import PieceTableTokenizer, synthetic_pieces
    model = B200RnntModel(eng, PieceTableTokenizer(synthetic_pieces(eng.cfg.vocab_size)), max_batch=n_clips)
    audios = [audio_from_numpy(synth_clip(rank * n_clips + i, seconds), 16000) for i in range(n_clips)] * batches
    cfg = TranscribeConfig(verbose=False)
    transcribe_batch(model, audios[: 2 * n_clips], cfg)          # warm-up: sizes both staging sets
    t0 = time.perf_counter()
    res = transcribe_batch(model, audios, cfg)
    dt = time.perf_counter() - t0
    from reazonspeech_b200.nemo.asr import transcribe
    single = []
    for a in audios[:6]:                                          # the reference's own call shape: one clip per call
        t1 = time.perf_counter()
        transcribe(model, a, cfg)
        single.append(time.perf_counter() - t1)
    single_ms = 1e3 * float(np.median(single[1:]))
    return {"value": len(audios) * seconds / dt, "unit": UNIT, "clips": len(audios), "ms_per_batch": 1e3 * dt / batches,
            "single_clip_ms": single_ms, "single_clip_rtfx": seconds / (single_ms * 1e-3),
            "subwords_per_clip": sum(len(r.subwords) for r in res) / len(res),
            "what": "transcribe_batch(model, audios): numpy clips in, TranscribeResult out, one GPU"}


def alsd_rtfx(cfg, wav_dev, len_dev, seconds: float, beam: int = 4):
    """The same batch with the reference checkpoint's DEFAULT decoding (ALSD beam search, pkg/nemo-asr/src/decode.py:29) instead of
    greedy: log-mel + encoder + rs_rnnt_alsd, device-resident inputs, one warm-up + two timed passes (synchronous call)."""
    from reazonspeech_b200.engine import Engine
    from reazonspeech_b200.weights import random_state_dict
    eng = Engine(cfg, random_state_dict(cfg, seed=0), str(wav_dev.device), alsd=True)

    def one():
        mel, mel_len = eng.log_mel(wav_dev, len_dev)
        enc, enc_len = eng.encode(mel, mel_len)
        return eng.alsd(enc, enc_len, beam=beam)

    one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2):
        y, steps, n, score = one()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 2
    B = wav_dev.shape[0]
    return {"value": B * seconds / dt, "unit": UNIT, "ms_per_step": 1e3 * dt, "beam": beam, "tokens_per_clip": float(n.float().mean()),
            "what": "log-mel + encoder + ALSD beam search (NeMo align_length_sync_decoding, u_max = 2 T, score_norm), same batch, device-resident"}


def python_api_multi_gpu_rtfx(cfg, n_gpus: int, n_clips: int, seconds: float):
    """``load_model(devices=range(n_gpus))`` in THIS process, then ``transcribe_batch`` over n_gpus x n_clips clips."""
    from reazonspeech_b200.nemo.asr import TranscribeConfig, audio_from_numpy, load_model, transcribe_batch
    from reazonspeech_b200.synth import synth_clip
    model = load_model(synthetic=True, config=cfg, seed=0, max_batch=n_clips, devices=list(range(n_gpus)))
    audios = [audio_from_numpy(synth_clip(i, seconds), 16000) for i in range(n_gpus * n_clips)]
    conf = TranscribeConfig(verbose=False)
    transcribe_batch(model, audios * 4, conf)                   # warm-up with the measured call's own shape: workspaces and BOTH pinned staging sets on every device (cudaHostAlloc of the second 64 MB set inside the timed call halved the first measurement)
    t0 = time.perf_counter()
    res = transcribe_batch(model, audios * 4, conf)              # four engine batches per device
    dt = time.perf_counter() - t0
    return {"value": len(res) * seconds / dt, "unit": UNIT, "clips": len(res), "devices": n_gpus, "seconds": dt,
            "what": "one process, load_model(devices=[0..N-1]) + transcribe_batch(model, audios): numpy clips in, TranscribeResult out"}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, tokens: torch.Tensor, frames: torch.Tensor, n_tok: torch.Tensor):
    """Write what rs_transcribe_device returned (tokens / frames int32 [B, U], n_tok int32 [B]) as float32 .npy files.
    Entries past a clip's token count are unspecified by the C ABI and written as -1.  When the arrays exceed
    DUMP_BYTES, a fixed seeded sample of clips is written, with their batch indices in clips.npy."""
    B, U = tokens.shape
    clips = np.arange(B)
    per_clip = (2 * U + 2) * 4
    if B * per_clip > DUMP_BYTES:
        clips = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // per_clip, replace=False))
    n = n_tok.numpy()[clips]
    valid = np.arange(U)[None, :] < np.minimum(n, U)[:, None]
    arrays = {"tokens": np.where(valid, tokens.numpy()[clips], -1), "frames": np.where(valid, frames.numpy()[clips], -1),
              "n_tokens": n, "clips": clips}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float32))


def make_batch(n_clips: int, seconds: float, rank: int):
    from reazonspeech_b200.synth import synth_clip
    L = int(seconds * 16000) + 2 * PAD
    wav = torch.zeros(n_clips, L, dtype=torch.float32)
    for i in range(n_clips):
        wav[i, PAD:L - PAD] = torch.from_numpy(synth_clip(rank * n_clips + i, seconds))   # pad_audio: silence both sides
    return wav, torch.full((n_clips,), L, dtype=torch.int32)


def dist_setup(gpus: int):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        global HOST_GROUP                      # CPU-side rendezvous for the extras during which a rank must leave its GPU alone
        HOST_GROUP = dist.new_group(backend="gloo")
    return world, rank, local


HOST_GROUP = None


CPU_CLIPS = 8          # bounded CPU sample: the first clips of the SAME 32 x 30 s set, one transcribe() each (batch = 1)


def _cpu_setup(pin: bool):
    from oracle import nemo_restated as O
    from oracle.cpu_threads import physical_threads
    from reazonspeech_b200.config import ModelConfig
    from reazonspeech_b200.synth import synth_clip
    from reazonspeech_b200.weights import random_state_dict
    cfg = ModelConfig()
    sd = random_state_dict(cfg, seed=0)
    cores, how = physical_threads(pin=pin)          # deterministic: one thread per physical core of one NUMA node
    clip = lambda i, seconds: torch.from_numpy(np.pad(synth_clip(i, seconds), PAD))
    return O, cfg, sd, cores, how, clip


def cpu_oracle_rtfx(seconds: float, n_clips: int = CPU_CLIPS):
    """The reference algorithm (oracle port, fp32 PyTorch, batch=1 like transcribe.py:48-50) on the host cores, on the first
    ``n_clips`` clips of the GPU arm's own clip set."""
    O, cfg, sd, cores, how, clip = _cpu_setup(pin=False)
    n_before = torch.get_num_threads()
    O.transcribe_tokens(clip(1, 2.0), sd, cfg)                                  # warm-up (thread pool, oneDNN primitives)
    t0 = time.perf_counter()
    for i in range(n_clips):
        O.transcribe_tokens(clip(i, seconds), sd, cfg)
    dt = time.perf_counter() - t0
    torch.set_num_threads(n_before)
    return n_clips * seconds / dt, cores, how, dt


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; NeMo itself cannot be installed offline, DESIGN.md section 7)
    on the SAME clips as the GPU arm.  A step = one transcribe() of one 30 s clip of the set (batch = 1 is the only way
    the reference calls NeMo, pkg/nemo-asr/src/transcribe.py:48-50); K steps walk K clips of the 32."""
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    seconds = args.seconds
    O, cfg, sd, cores, how, clip = _cpu_setup(pin=True)
    for i in range(max(min(args.warmup, 3), 1)):
        O.transcribe_tokens(clip(31 - i, 2.0 if i else seconds), sd, cfg)       # first warm-up at full length, the rest short
    t0 = time.perf_counter()
    for k in range(args.steps):
        O.transcribe_tokens(clip(k % args.batch, seconds), sd, cfg)
    dt = time.perf_counter() - t0
    v = args.steps * seconds / dt
    sample = (f"{args.steps} steps x one {seconds:g} s clip of the same {args.batch}-clip set (batch=1, fp32, greedy), oracle port of the "
              f"NeMo path; {how}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic 16 kHz AM/FM clips; seeded random weights (619 M architecture)",
        "config": {"workload": f"nemo-asr FastConformer-RNNT 619M, batch={args.batch}x{seconds:g} s clips per GPU", "sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def decode_sensitivity(eng, run_step, n_tok_of, steps: int, targets=(50, 150, 250)):
    """Step time as a function of the decode load: the synthetic checkpoint's blank bias is shifted (device tensor, in place)
    until the batch emits about `target` tokens per 30 s clip, the step is timed, the bias is restored.  The emission rate of
    random weights is a property of one calibration; this makes the RTFx's dependence on it visible."""
    bias = eng.weights["joint.out.b"]
    blank = eng.cfg.blank
    base = float(bias[blank])
    out = []

    def tokens_at(shift):
        bias[blank] = base + shift
        run_step()
        torch.cuda.synchronize()
        return float(n_tok_of().float().mean())

    try:
        for target in targets:
            lo, hi = -12.0, 12.0                                   # tokens decrease as the blank bias rises
            for _ in range(16):
                mid = 0.5 * (lo + hi)
                if tokens_at(mid) > target:
                    lo = mid
                else:
                    hi = mid
            shift = 0.5 * (lo + hi)
            tok = tokens_at(shift)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(steps):
                run_step()
            ev1.record()
            torch.cuda.synchronize()
            out.append({"target_tokens_per_clip": target, "tokens_per_clip": tok, "blank_shift": shift, "max_tokens_in_a_clip": int(n_tok_of().max()),
                        "ms_per_step": ev0.elapsed_time(ev1) / steps})
    finally:
        bias[blank] = base
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="clips per GPU per step")
    ap.add_argument("--seconds", type=float, default=NOMINAL_SECONDS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip python_api / decode_sensitivity / config2 (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's tokens / frames / token counts (rank 0) "
                                                           "as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    world, rank, local = dist_setup(args.gpus)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from reazonspeech_b200.config import ModelConfig
    from reazonspeech_b200.engine import Engine
    from reazonspeech_b200.weights import random_state_dict

    cfg = ModelConfig()
    sd = random_state_dict(cfg, seed=0)
    eng = Engine(cfg, sd, f"cuda:{local}")
    del sd
    B = args.batch
    wav_host, len_host = make_batch(B, args.seconds, rank)
    wav_host = wav_host.pin_memory()
    L = wav_host.shape[1]
    wav_dev, len_dev = wav_host.to(dev), len_host.to(dev)
    U = eng.u_max(L)
    out_dev = (torch.zeros(B, U, dtype=torch.int32, device=dev), torch.zeros(B, U, dtype=torch.int32, device=dev),
               torch.zeros(B, dtype=torch.int32, device=dev))
    out_host = (torch.zeros(B, U, dtype=torch.int32).pin_memory(), torch.zeros(B, U, dtype=torch.int32).pin_memory(),
                torch.zeros(B, dtype=torch.int32).pin_memory())
    eng.ensure_workspace(B, L)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident timed region (`value`)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                      # nvidia-smi needs a few hundred ms to start: begin before the warm-up
    for _ in range(args.warmup):
        eng.transcribe_device(wav_dev, len_dev, U, out_dev)
    barrier()
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        eng.transcribe_device(wav_dev, len_dev, U, out_dev)
    ev1.record()
    barrier()
    launches = eng.launch_count - launches0
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop() if rank == 0 else None
    ms_step = ms_total / args.steps
    value = world * B * args.seconds / (ms_step / 1e3)
    n_tok = out_dev[2].cpu()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_dev[0].cpu(), out_dev[1].cpu(), n_tok)

    # ---------------- end-to-end through the host-buffer C-ABI call (`e2e`)
    for _ in range(2):
        eng.transcribe_host(wav_host, len_host, U, out_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.transcribe_host(wav_host, len_host, U, out_host)      # synchronises internally (tokens are on the host on return)
    barrier()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / args.steps)
    e2e_value = world * B * args.seconds / e2e_s
    h2d = wav_host.numel() * 4 + len_host.numel() * 4
    d2h = (out_host[0].numel() + out_host[1].numel() + out_host[2].numel()) * 4

    # ---------------- roofline of the dominant kernel (tcgen05 GEMM), CUDA events per launch
    sus, burst, hbm, src = measured_peaks()
    eng.enable_gemm_timing(True)
    for _ in range(args.steps):
        eng.transcribe_device(wav_dev, len_dev, U, out_dev)
    torch.cuda.synchronize(dev)
    g_ms, g_flops, g_n = eng.gemm_timing()
    eng.enable_gemm_timing(False)
    eng.enable_stage_timing(True)
    eng.transcribe_device(wav_dev, len_dev, U, out_dev)
    torch.cuda.synchronize(dev)
    stages = eng.stage_times_ms()
    eng.enable_stage_timing(False)
    decode_prof = eng.decode_cycles(B, L, U)
    if not any(v for k, v in decode_prof.items() if k != "iterations"):
        # (a build with -DRS_NO_DECODE_COUNTERS; the attention / GEMM timelines are compiled in only with RS_BUILD_FLAGS=-DRS_PROF)
        decode_prof = {"iterations": decode_prof["iterations"]}
    # per-kernel device time inside the pipeline (event pair around every launch; one extra, untimed step)
    eng.kernel_timing(True)
    eng.transcribe_device(wav_dev, len_dev, U, out_dev)
    kernel_ms = {k: {"launches": n, "ms": round(ms, 4)} for k, (n, ms) in sorted(eng.kernel_timing().items(), key=lambda kv: -kv[1][1])}
    eng.kernel_timing(False)
    attn_cycles = eng.attention_cycles()
    if not any(attn_cycles.values()):
        attn_cycles = None
    # memory-bound kernels against the measured copy bandwidth: ALGORITHMIC bytes (SURVEY.md section 8d) over the
    # in-pipeline time of their launches (event pairs above, so warm-L2 effects are included: a fraction can exceed 1)
    valid_T = eng.cfg.enc_frames(L)
    dm = eng.cfg.d_model

    def hbm_line(key, bytes_per_step, what):
        if key not in kernel_ms or kernel_ms[key]["ms"] <= 0:
            return None
        gbs = bytes_per_step / (kernel_ms[key]["ms"] * 1e-3) / 1e9
        return {"kernel": key, "bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm, "bytes_per_step": bytes_per_step, "what": what}

    n_ln = kernel_ms.get("launch_layernorm", {}).get("launches", 0)
    n_dw = kernel_ms.get("launch_conv_dw", {}).get("launches", 0)
    roofline_hbm = [r for r in (
        hbm_line("launch_logmel_fused", B * (L * 4 + eng.cfg.mel_valid(L) * eng.cfg.n_mels * 4), "log-mel frontend, one kernel: fp32 samples in, fp32 log-mel features + per-feature statistics out (2.98 MB per clip; the normalisation is applied by the consumer's load)"),
        hbm_line("launch_layernorm", n_ln * B * valid_T * dm * 6, "LayerNorm: fp32 row in, bf16 row out, per launch"),
        hbm_line("launch_conv_dw", n_dw * B * valid_T * dm * 4, "depthwise conv + BN + Swish: bf16 in, bf16 out, per launch"),
    ) if r is not None]
    # ALGORITHMIC FLOPs: the engine counts 2*M*N*K with M = B x frame capacity (a multiple of 8: 392 for 388 valid
    # frames); the roofline numerator keeps only the valid rows
    g_flops *= eng.cfg.enc_frames(L) / max(eng.enc_frames(L), 1)
    achieved = g_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    # DRAM bytes per launch of the dominant kernel cannot be measured without a profiler: they are read from the committed
    # summary of this round's `ncu --set full` capture of the same command (profiles/r02_gemm_traffic.json, written by
    # scripts/summarize_ncu.py); null when that file is absent
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
    roofline = {"bound": "tensor", "achieved": achieved, "peak": sus, "unit": "TFLOP/s", "frac": achieved / sus, "traffic": traffic,
                "traffic_source": traffic_src,
                "kernel": "gemm_bf16_tn_kernel (tcgen05.mma, all encoder/joint GEMMs)", "peak_source": f"{src} bf16_tflops_sustained",
                "launches_per_step": g_n // max(args.steps, 1), "gemm_ms_per_step": g_ms / max(args.steps, 1),
                "algorithmic_gflop_per_step": g_flops / max(args.steps, 1) / 1e9,
                "how": "CUDA events around every GEMM launch on its stream, separate pass of the same K steps"}

    # configs[2] of BASELINE.json (1024 clips sharded over 8 GPUs = 128 per GPU) next to the 32-per-GPU weak-scaling value
    config2 = None
    if (world == 8 or os.environ.get("RS_BENCH_CONFIG2") == "1") and not args.no_extras:
        # an extra: a rank that fails here must not leave the others waiting in a collective, so the timed part has no barrier
        # of its own and the two reductions below are reached by every rank whatever happened
        B2, ms_local, err2 = 128, 0.0, None
        n2 = max(args.steps // 4, 3)
        try:
            w2, l2 = make_batch(B2, args.seconds, rank)
            w2d, l2d = w2.to(dev), l2.to(dev)
            o2 = (torch.zeros(B2, U, dtype=torch.int32, device=dev), torch.zeros(B2, U, dtype=torch.int32, device=dev), torch.zeros(B2, dtype=torch.int32, device=dev))
            eng.ensure_workspace(B2, L)
            for _ in range(2):
                eng.transcribe_device(w2d, l2d, U, o2)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n2):
                eng.transcribe_device(w2d, l2d, U, o2)
            e1.record()
            torch.cuda.synchronize()
            ms_local = e0.elapsed_time(e1) / n2
            del w2d, l2d, o2
        except Exception as exc:
            err2 = f"{type(exc).__name__}: {exc}"[:300]
        ms2 = max_over_ranks(ms_local)
        failed = max_over_ranks(1.0 if err2 else 0.0)
        if failed:
            config2 = {"error": err2 or "another rank failed"}
        else:
            config2 = {"workload": f"nemo-asr FastConformer-RNNT 619M, {world * B2} x {args.seconds:g} s clips sharded by utterance across {world} GPUs ({B2} per GPU)",
                       "value": world * B2 * args.seconds / (ms2 / 1e3), "unit": UNIT, "ms_per_step": ms2, "steps": n2,
                       "timing": "CUDA events per rank around the steps (no barrier inside an extra), max over ranks"}
        eng.ensure_workspace(B, L)
    # the one-process multi-GPU model (load_model(devices=...)): rank 0 drives ALL `world` GPUs from its own process while the
    # other ranks idle at the barrier below -- the call a user makes on an 8-GPU box without torchrun
    api_multi = None
    if world > 1 and not args.no_extras:
        # The other ranks must not touch their GPUs meanwhile: an NCCL barrier is a kernel spinning on the device, and rank 0's
        # in-process replica for that device would be time-sliced against it (measured: 8.6 k RTFx instead of 2 x 35 k at two
        # GPUs).  They wait on the host (gloo) instead.
        import torch.distributed as dist
        barrier()
        if rank == 0:
            try:
                api_multi = python_api_multi_gpu_rtfx(eng.cfg, world, B, args.seconds)
            except Exception as exc:
                api_multi = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        dist.barrier(group=HOST_GROUP)
    if rank != 0:
        return
    cpu = None
    if not args.no_cpu_baseline and world == 1:          # the CPU arm is timed at N=1 only (it is the same host either way)
        v, cores, how, secs = cpu_oracle_rtfx(args.seconds)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"the first {CPU_CLIPS} clips of the same {B} x {args.seconds:g} s set, one transcribe() each (batch=1, fp32, greedy) "
                         f"through the oracle port: {secs:.1f} s of CPU work on {how}"}
    api = sens = alsd = None
    if world == 1 and not args.no_extras:
        try:
            alsd = alsd_rtfx(eng.cfg, wav_dev, len_dev, args.seconds)
        except Exception as exc:
            alsd = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            api = python_api_rtfx(eng, B, args.seconds, rank)
        except Exception as exc:      # an extra: reported, never fatal to the contract keys
            api = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            sens = decode_sensitivity(eng, lambda: eng.transcribe_device(wav_dev, len_dev, U, out_dev), lambda: out_dev[2].cpu(), max(args.steps // 2, 3))
        except Exception as exc:
            sens = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    print(json.dumps({
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic 16 kHz AM/FM clips; seeded random weights (619 M architecture, no checkpoint offline)",
        "config": {"workload": f"nemo-asr FastConformer-RNNT 619M, batch={B}x{args.seconds:g} s clips per GPU",
                   "samples_per_clip": L, "enc_frames": eng.cfg.enc_frames(L), "parallelism": f"utterance-sharded x{world}, no collective",
                   "l2": "per-step working set (~2 GB activations) exceeds the 126 MB L2; no explicit flush",
                   "tokens_per_clip": float(n_tok.float().mean())},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_s * 1e3},
        "roofline": roofline, "roofline_hbm": roofline_hbm, "stage_ms": stages, "kernel_ms": kernel_ms, "attention_cycles_cta": attn_cycles, "decode_cycles_cta0": decode_prof, "cpu_baseline": cpu, "python_api": api,
        "decode_sensitivity": sens, "alsd": alsd, "config2": config2, "python_api_multi_gpu": api_multi,
    }), flush=True)


if __name__ == "__main__":
    main()
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
