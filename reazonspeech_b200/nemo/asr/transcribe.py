"""``load_model`` / ``transcribe`` with the reference's signatures (pkg/nemo-asr/src/transcribe.py:9-60)
on top of the B200 engine, plus the batched ``transcribe_batch`` the reference lacks
(its evaluators leave ``_evaluate_batch`` unimplemented, pkg/evaluation/examples/rs-nemo/eval.py:31-32).

The object returned by ``load_model`` is a duck-typed stand-in for NeMo's EncDecRNNTBPEModel at
exactly the three points the reference touches it (SURVEY.md section 8b):
``model.transcribe(list_of_tensors, batch_size=..., return_hypotheses=True, verbose=...)``,
``hyp.y_sequence`` / ``hyp.timestamp`` and ``model.tokenizer.ids_to_text``; the reference's own
transcribe()/decode_hypothesis() therefore run unmodified on it (see INTEGRATION.md)."""
from __future__ import annotations

import glob
import math
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Union

import numpy as np
import torch

from ...config import ModelConfig
from ...engine import Engine
from ...tokenizer import PieceTableTokenizer, SentencePieceTokenizer, synthetic_pieces
from ...weights import load_nemo_archive, random_state_dict
from .audio import SAMPLERATE, norm_audio, pad_audio
from .decode import PAD_SECONDS, SECONDS_PER_STEP, build_result, decode_hypothesis
from .interface import AlignedCaption, AlignResult, AudioData, Caption, TranscribeConfig, TranscribeResult

HF_REPO = "reazon-research/reazonspeech-nemo-v2"
CAPTION_MARGIN = 25.0          # live captions lag the speech: search from this long before the display time (oneseg's _MARGIN)
CONFIDENCE_FRAMES = 30         # window of the min-mean caption confidence: 30 encoder frames = 2.4 s
ENV_CHECKPOINT = "REAZONSPEECH_NEMO_CHECKPOINT"
ENV_SYNTHETIC = "REAZONSPEECH_B200_SYNTHETIC"


@dataclass
class Hypothesis:
    """The two NeMo Hypothesis fields the reference reads (decode.py:40,44), ALSD-shaped:
    y_sequence = [blank, tok_0, ...]; timestamp[i] = frame_i + i + 1 so that decode.py:48's
    ``step - idx - 1`` recovers the emitting encoder frame."""
    y_sequence: torch.Tensor
    timestamp: List[int]
    score: float = 0.0

    @staticmethod
    def from_greedy(tokens: Sequence[int], frames: Sequence[int], blank: int) -> "Hypothesis":
        y = torch.tensor([blank, *[int(t) for t in tokens]], dtype=torch.long)
        return Hypothesis(y, [int(f) + i + 1 for i, f in enumerate(frames)])


class HostStaging:
    """Grow-only host buffers of one in-flight batch, reused across calls and pinned when a CUDA device is there:
    allocating (cudaHostAlloc) and zero-filling a fresh 64 MB pinned batch costs more than the batch's GPU time."""

    def __init__(self, pin: bool):
        self.pin = pin
        self._wav = self._lens = self._tok = self._frm = self._ntok = None

    def _grown(self, buf, numel: int, dtype):
        if buf is None or buf.numel() < numel:
            buf = torch.empty(int(numel * 1.25) + 16, dtype=dtype)
            if self.pin:
                buf = buf.pin_memory()
        return buf

    def stage(self, waves: Sequence[np.ndarray], pad: int):
        """Rows ``[zeros(pad) | wave | zeros(pad) | zeros to L]`` (pad_audio, audio.py:70-83, written in place) -> (wav [B, L], lens [B]).

        A batch whose waveforms are ALL 16-bit PCM (int16 arrays, e.g. ``audio_from_path(..., pcm16=True)``) is staged as
        int16 and scaled by 2^-15 on the device (rs_transcribe_batch_pcm16): half the pinned memory and PCIe bytes.  A mixed
        batch is staged as float32, int16 members converted the way a file decoder would (sample / 32768)."""
        B = len(waves)
        L = max(len(w) for w in waves) + 2 * pad
        L = (L + 3) & ~3                                # rows start 8 / 16-byte aligned: the kernel's vectorised staging load
        pcm = all(w.dtype == np.int16 for w in waves)
        if pcm:
            self._wav16 = self._grown(getattr(self, "_wav16", None), B * L, torch.int16)
            wav = self._wav16[: B * L].view(B, L)
        else:
            self._wav = self._grown(self._wav, B * L, torch.float32)
            wav = self._wav[: B * L].view(B, L)
        self._lens = self._grown(self._lens, B, torch.int32)
        lens = self._lens[:B]
        # the copies run in the library (rs_stage_rows: memcpy split over a few threads, interpreter lock released): the
        # same loop as numpy slice assignments cost ~0.5 ms per 30 s clip, as much as the GPU spends on it
        import ctypes as C
        from ...engine import load_library
        srcs = [np.ascontiguousarray(w if w.dtype in (np.int16, np.float32) else w.astype(np.float32)) for w in waves]
        ptr = (C.c_void_p * B)(*[a.ctypes.data for a in srcs])
        n = (C.c_int64 * B)(*[a.shape[0] for a in srcs])
        is16 = (C.c_int32 * B)(*[int(a.dtype == np.int16) for a in srcs])
        rc = load_library().rs_stage_rows(wav.data_ptr(), L, ptr, n, is16, int(pcm), B, pad, min(4, B))
        if rc != 0:
            raise RuntimeError(f"rs_stage_rows failed ({rc})")
        lens.copy_(torch.tensor([a.shape[0] + 2 * pad for a in srcs], dtype=torch.int32))
        return wav, lens

    def outputs(self, B: int, U: int):
        self._tok = self._grown(self._tok, B * U, torch.int32)
        self._frm = self._grown(self._frm, B * U, torch.int32)
        self._ntok = self._grown(self._ntok, B, torch.int32)
        return self._tok[: B * U].view(B, U), self._frm[: B * U].view(B, U), self._ntok[:B]


class B200RnntModel:
    """Engine + tokenizer behind NeMo's model surface."""

    def __init__(self, engine: Engine, tokenizer, max_batch: int = 64, decoding: str = "greedy", beam_size: int = 4):
        self.engine = engine
        self.cfg = engine.cfg
        self.tokenizer = tokenizer
        self.max_batch = max_batch
        self.decoding, self.beam_size = decoding, beam_size       # "greedy" (north_star's parity target) or "alsd" (the checkpoint's default)
        pin = torch.cuda.is_available()
        self._staging = (HostStaging(pin), HostStaging(pin))      # double buffer: stage batch k+1 while batch k runs

    # -- token-level batched path
    def iter_token_batches(self, waveforms: Sequence[np.ndarray], pad: int = 0):
        """16 kHz mono waveforms (each gets ``pad`` zero samples on both sides) -> yields ``(indices, [(tokens, frames)])``
        batch by batch.

        Utterances are sorted by length and cut into batches of at most ``max_batch`` so padding waste stays small.
        The engine call of batch k runs on a worker thread (ctypes drops the GIL) while this thread stages batch k+1
        into the other staging set and the caller post-processes batch k-1: on a long list the host work hides behind
        the GPU.  One engine call is in flight at a time (an engine is not re-entrant)."""
        from concurrent.futures import ThreadPoolExecutor
        if len(waveforms) == 0:
            return
        order = sorted(range(len(waveforms)), key=lambda i: len(waveforms[i]))
        batches = [order[lo:lo + self.max_batch] for lo in range(0, len(order), self.max_batch)]
        eng = self.engine
        eng.ensure_workspace(len(batches[0]), (len(waveforms[order[-1]]) + 2 * pad + 3) & ~3)   # once, on this thread (stage() rounds rows up to 4 samples)

        def run(staging, idx):
            wav, lens = staging.stage([waveforms[i] for i in idx], pad)
            out = staging.outputs(len(idx), eng.u_max(wav.shape[1]))
            return wav, lens, out

        def collect(done, idx):
            tokens, frames, ntok = done
            counts = ntok.tolist()
            return idx, [(tokens[r, :n].tolist(), frames[r, :n].tolist()) for r, n in enumerate(counts[: len(idx)])]

        if len(batches) == 1:                                         # nothing to overlap: skip the thread hand-off (one-clip calls)
            wav, lens, out = run(self._staging[0], batches[0])
            yield collect(eng.transcribe_host(wav, lens, out[0].shape[1], out), batches[0])
            return
        with ThreadPoolExecutor(max_workers=1) as pool:
            in_flight = None
            for k, idx in enumerate(batches):
                wav, lens, out = run(self._staging[k & 1], idx)
                nxt = (pool.submit(eng.transcribe_host, wav, lens, out[0].shape[1], out), idx)
                if in_flight is not None:
                    yield collect(in_flight[0].result(), in_flight[1])
                in_flight = nxt
            yield collect(in_flight[0].result(), in_flight[1])

    def transcribe_tokens(self, waveforms: Sequence[np.ndarray], pad: int = 0):
        """-> [(tokens, frames)] in input order."""
        results = [None] * len(waveforms)
        for idx, items in self.iter_token_batches(waveforms, pad):
            for i, item in zip(idx, items):
                results[i] = item
        return results

    def iter_token_batches_raw(self, waves: Sequence[np.ndarray], samplerate: int, pad: int = 0):
        """Like ``iter_token_batches`` for audio that still needs ``norm_audio`` (pkg/nemo-asr/src/audio.py:54-68): waveforms
        at ``samplerate`` (any rate), mono [n] or channels-first [c, n] with the SAME channel count, float or int16 PCM.  They
        are staged as they are (pinned), copied to the GPU and resampled / down-mixed / padded there (rs_resample_mono)
        straight into the buffer the engine transcribes from: the host never touches a sample arithmetically.  (scipy's
        resample_poly, which this kernel restates, costs the host ~10 ms per 30 s 48 kHz clip -- more than the whole engine.)"""
        if len(waves) == 0:
            return
        eng = self.engine
        waves = [w if w.ndim == 2 else w[None] for w in waves]
        C = waves[0].shape[0]
        if any(w.shape[0] != C for w in waves):
            raise ValueError("iter_token_batches_raw: all waveforms of a call must have the same number of channels")
        pcm = all(w.dtype == np.int16 for w in waves)
        order = sorted(range(len(waves)), key=lambda i: waves[i].shape[1])
        for lo in range(0, len(order), self.max_batch):
            idx = order[lo:lo + self.max_batch]
            L = (max(waves[i].shape[1] for i in idx) + 3) & ~3
            raw = torch.zeros(len(idx), C, L, dtype=torch.int16 if pcm else torch.float32)
            if torch.cuda.is_available():
                raw = raw.pin_memory()
            rows = raw.numpy()
            for r, i in enumerate(idx):
                w = waves[i]
                rows[r, :, : w.shape[1]] = w if (pcm or w.dtype != np.int16) else w.astype(np.float32) * np.float32(1.0 / 32768.0)
            lens = torch.tensor([waves[i].shape[1] for i in idx], dtype=torch.int32)
            with torch.cuda.device(eng.device):
                wav, wl = eng.resample_mono(raw.to(eng.device, non_blocking=True), lens.to(eng.device, non_blocking=True), samplerate, pad)
                tokens, frames, ntok = eng.transcribe_device(wav, wl)
                tokens, frames, counts = tokens.cpu(), frames.cpu(), ntok.cpu().tolist()
            yield idx, [(tokens[r, :n].tolist(), frames[r, :n].tolist()) for r, n in enumerate(counts)]

    # -- NeMo's call shape (transcribe.py:48-53): already padded tensors
    def transcribe_alsd(self, waveforms: Sequence[np.ndarray], pad: int = 0) -> List[Hypothesis]:
        """ALSD beam search (NeMo's align_length_sync_decoding, the strategy reazonspeech-nemo-v2 ships with): hypotheses exactly
        as NeMo hands them to the reference's decode.py -- y_sequence with the leading blank, timestamp = alignment steps."""
        eng = self.engine
        out: List[Optional[Hypothesis]] = [None] * len(waveforms)
        order = sorted(range(len(waveforms)), key=lambda i: len(waveforms[i]))
        for lo in range(0, len(order), self.max_batch):
            idx = order[lo:lo + self.max_batch]
            wav, lens = self._staging[0].stage([waveforms[i] for i in idx], pad)
            with torch.cuda.device(eng.device):
                x = wav.to(eng.device, non_blocking=True)
                if x.dtype == torch.int16:
                    x = x.to(torch.float32) * (1.0 / 32768.0)
                mel, mel_len = eng.log_mel(x, lens.to(eng.device))
                enc, enc_len = eng.encode(mel, mel_len)
                y, steps, n, score = [a.cpu() for a in eng.alsd(enc, enc_len, beam=self.beam_size)]
            for r, i in enumerate(idx):
                k = int(n[r])
                out[i] = Hypothesis(y[r, : k + 1].to(torch.long), steps[r, :k].tolist(), float(score[r]))
        return out

    def align_tokens(self, waveforms: Sequence[np.ndarray], token_lists: Sequence[Sequence[int]], pad: int = 0):
        """RNN-T forced alignment of known token sequences (rs_rnnt_align): 16 kHz mono waveforms (each gets ``pad`` zero
        samples on both sides) and one token-id list per waveform -> ``[(frames, token_log_probs, viterbi_log_prob,
        log_likelihood)]`` in input order; ``frames[i]`` is the encoder frame that emits token i on the best path.  Batches are
        cut by length, as in ``transcribe_alsd``."""
        eng = self.engine
        if "alsd.out.w3" not in eng.weights:
            raise RuntimeError("this model was loaded without the aligner weights: load it with load_model(..., aligner=True)")
        if len(token_lists) != len(waveforms):
            raise ValueError(f"align_tokens: {len(waveforms)} waveforms but {len(token_lists)} token lists")
        out: List[Optional[tuple]] = [None] * len(waveforms)
        order = sorted(range(len(waveforms)), key=lambda i: len(waveforms[i]))
        for lo in range(0, len(order), self.max_batch):
            idx = order[lo:lo + self.max_batch]
            wav, lens = self._staging[0].stage([waveforms[i] for i in idx], pad)
            U = max(1, max(len(token_lists[i]) for i in idx))
            targets = torch.zeros(len(idx), U, dtype=torch.int32)
            for r, i in enumerate(idx):
                targets[r, : len(token_lists[i])] = torch.tensor([int(t) for t in token_lists[i]], dtype=torch.int32)
            tgt_len = torch.tensor([len(token_lists[i]) for i in idx], dtype=torch.int32)
            with torch.cuda.device(eng.device):
                x = wav.to(eng.device, non_blocking=True)
                if x.dtype == torch.int16:
                    x = x.to(torch.float32) * (1.0 / 32768.0)
                mel, mel_len = eng.log_mel(x, lens.to(eng.device))
                enc, enc_len = eng.encode(mel, mel_len)
                frames, tok_logp, viterbi, loglik = [a.cpu() for a in eng.align(enc, enc_len, targets.to(eng.device), tgt_len.to(eng.device))]
            for r, i in enumerate(idx):
                k = len(token_lists[i])
                out[i] = (frames[r, :k].tolist(), tok_logp[r, :k].tolist(), float(viterbi[r]), float(loglik[r]))
        return out

    def align_caption_tokens(self, waveforms: Sequence[np.ndarray], windows: Sequence[Sequence[tuple]],
                             token_lists: Sequence[Sequence[Sequence[int]]], pad: int = 0):
        """Free-span alignment of known token sequences inside time windows of longer recordings (rs_rnnt_align_spans).
        ``waveforms``: 16 kHz mono recordings, each encoded ONCE with ``pad`` zero samples on both sides; ``windows[i]``: the
        (start, end) seconds, on recording i's own axis, of the window each of its captions is searched in; ``token_lists[i]``:
        the captions' token ids.  -> per recording, per caption ``(lo, frames, token_log_probs, path_logp, viterbi_log_prob,
        log_likelihood)`` or None (an empty window, or no tokens).  ``lo`` is the window's first encoder frame, ``frames`` the
        absolute encoder frame of every token on the best path and ``path_logp[t - lo]`` the path's log p at frame t of the
        window.  Recordings are cut into length-sorted batches as in ``align_tokens``; every batch is one encoder pass and one
        rs_rnnt_align_spans call over all of its recordings' captions."""
        eng = self.engine
        if "alsd.out.w3" not in eng.weights:
            raise RuntimeError("this model was loaded without the aligner weights: load it with load_model(..., aligner=True)")
        if not (len(waveforms) == len(windows) == len(token_lists)):
            raise ValueError(f"align_caption_tokens: {len(waveforms)} waveforms, {len(windows)} window lists, {len(token_lists)} token lists")
        out: List[List[Optional[tuple]]] = [[None] * len(w) for w in windows]
        pad_s = pad / SAMPLERATE
        order = sorted(range(len(waveforms)), key=lambda i: len(waveforms[i]))
        for lo_b in range(0, len(order), self.max_batch):
            idx = order[lo_b:lo_b + self.max_batch]
            wav, lens = self._staging[0].stage([waveforms[i] for i in idx], pad)
            with torch.cuda.device(eng.device):
                x = wav.to(eng.device, non_blocking=True)
                if x.dtype == torch.int16:
                    x = x.to(torch.float32) * (1.0 / 32768.0)
                mel, mel_len = eng.log_mel(x, lens.to(eng.device))
                enc, enc_len = eng.encode(mel, mel_len)
                T = enc_len.cpu().tolist()
                items = []                                               # (recording, caption, src, lo, hi, tokens)
                for r, i in enumerate(idx):
                    for j, ((start, end), toks) in enumerate(zip(windows[i], token_lists[i])):
                        lo, hi = window_frames(start, end, T[r], pad_s)
                        if lo < hi and len(toks) > 0:
                            items.append((i, j, r, lo, hi, [int(t) for t in toks]))
                if not items:
                    continue
                U = max(len(it[5]) for it in items)
                spans = torch.tensor([[it[2], it[3], it[4]] for it in items], dtype=torch.int32)
                targets = torch.zeros(len(items), U, dtype=torch.int32)
                for k, it in enumerate(items):
                    targets[k, : len(it[5])] = torch.tensor(it[5], dtype=torch.int32)
                tgt_len = torch.tensor([len(it[5]) for it in items], dtype=torch.int32)
                frames, tok_logp, path_logp, viterbi, loglik = [a.cpu() for a in eng.align_spans(
                    enc, enc_len, spans.to(eng.device), targets.to(eng.device), tgt_len.to(eng.device))]
            for k, (i, j, _, lo, hi, toks) in enumerate(items):
                n = len(toks)
                out[i][j] = (lo, frames[k, :n].tolist(), tok_logp[k, :n].tolist(), path_logp[k, : hi - lo].tolist(),
                             float(viterbi[k]), float(loglik[k]))
        return out

    def transcribe(self, audio, batch_size: int = 1, return_hypotheses: bool = True, verbose: bool = True, **_):
        waves = [a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a) for a in audio]
        if self.decoding == "alsd":
            out = self.transcribe_alsd(waves)
        else:
            out = [Hypothesis.from_greedy(t, f, self.cfg.blank) for t, f in self.transcribe_tokens(waves)]
        if return_hypotheses:
            return out
        return [self.tokenizer.ids_to_text(h.y_sequence.tolist()[1:]) for h in out]


def _find_checkpoint() -> Optional[str]:
    env = os.environ.get(ENV_CHECKPOINT)
    if env:
        return env
    hub = os.path.expanduser(os.environ.get("HF_HOME", "~/.cache/huggingface"))
    hits = glob.glob(os.path.join(hub, "hub", "models--" + HF_REPO.replace("/", "--"), "snapshots", "*", "*.nemo"))
    return sorted(hits)[-1] if hits else None


def load_model(device=None, *, checkpoint: Optional[str] = None, synthetic: Optional[bool] = None,
               config: Optional[ModelConfig] = None, seed: int = 0, max_batch: int = 64, devices: Optional[Sequence] = None,
               decoding: str = "greedy", beam_size: int = 4, aligner: bool = False):
    """Load the ReazonSpeech FastConformer-RNNT onto a B200.

    ``device``: None / "cuda" / "cuda:N" as in the reference (transcribe.py:9-22, eval.py:26).
    "cpu" raises: this engine has no CPU path.  ``decoding``: "greedy" (default: BASELINE.json's parity target) or "alsd", NeMo's
    align_length_sync_decoding beam search with ``beam_size`` -- the strategy the shipped checkpoint decodes with by default
    (pkg/nemo-asr/src/decode.py:29); it runs on the GPU too (csrc/decode_alsd.cu).  ``devices`` (e.g. ``range(8)`` or ``["cuda:0", "cuda:1"]``) loads one
    replica per listed GPU into THIS process and returns a model that deals every call's utterances across them
    (``multi_gpu.MultiGpuRnntModel``; same surface, results in input order).  Weights come from ``checkpoint`` (a .nemo file),
    $REAZONSPEECH_NEMO_CHECKPOINT or the local Hugging Face cache of reazonspeech-nemo-v2.  ``aligner=True`` uploads the
    weights ``align`` / ``align_batch`` need (the tripled predictor / joint matrices, as ``decoding="alsd"`` does).
    With ``synthetic=True`` (or $REAZONSPEECH_B200_SYNTHETIC=1) seeded random weights of the same
    architecture are used instead -- the only option offline."""
    if device is None:
        device = "cuda"
    if str(device).startswith("cpu"):
        raise RuntimeError("reazonspeech_b200: device='cpu' is not supported (hand-written sm_100a kernels only)")
    if synthetic is None:
        synthetic = os.environ.get(ENV_SYNTHETIC, "") not in ("", "0")
    path = checkpoint or (None if synthetic else _find_checkpoint())
    if path is not None:
        cfg, sd, tok = load_nemo_archive(path)
        tokenizer = SentencePieceTokenizer(tok) if tok else PieceTableTokenizer(synthetic_pieces(cfg.vocab_size))
        if decoding == "greedy" and not cfg.checkpoint_decoding.startswith("greedy"):
            import warnings                 # the reference never overrides the checkpoint's strategy (transcribe.py:26-28): say what differs
            warnings.warn(f"{path}: the checkpoint is configured for '{cfg.checkpoint_decoding}' decoding; this model decodes greedily "
                          f"(transcripts can differ from the reference's default).  Pass decoding='alsd' for NeMo's ALSD beam search.", stacklevel=2)
    elif synthetic:
        cfg = config or ModelConfig()
        sd = random_state_dict(cfg, seed)
        tokenizer = PieceTableTokenizer(synthetic_pieces(cfg.vocab_size))
    else:
        raise FileNotFoundError(
            f"no .nemo checkpoint for {HF_REPO}: pass checkpoint=..., set ${ENV_CHECKPOINT}, populate the Hugging Face "
            f"cache, or request seeded synthetic weights with synthetic=True / ${ENV_SYNTHETIC}=1")
    if decoding not in ("greedy", "alsd"):
        raise ValueError(f"decoding must be 'greedy' or 'alsd', got {decoding!r}")
    if devices is None:
        return B200RnntModel(Engine(cfg, sd, str(device), alsd=decoding == "alsd" or aligner), tokenizer, max_batch=max_batch,
                             decoding=decoding, beam_size=beam_size)
    if decoding != "greedy":
        raise ValueError("the one-process multi-GPU model decodes greedily; load one model per device for beam search")
    if aligner:
        raise NotImplementedError("the one-process multi-GPU model does not align; load one model per device for align()")
    names = [d if isinstance(d, str) else f"cuda:{int(d)}" for d in devices]
    if len(names) == 0 or len(set(names)) != len(names):
        raise ValueError(f"devices must name distinct GPUs, got {list(devices)!r}")
    from ...engine import pack_weights
    from .multi_gpu import MultiGpuRnntModel
    packed = pack_weights(sd, cfg)                                   # repacked once, uploaded once per device
    return MultiGpuRnntModel([B200RnntModel(Engine(cfg, None, n, packed=packed), tokenizer, max_batch=max_batch) for n in names])


def _prepare(audio: AudioData) -> np.ndarray:
    wave = pad_audio(norm_audio(audio), PAD_SECONDS).waveform
    return wave if wave.dtype == np.int16 else wave.astype(np.float32, copy=False)     # int16 = PCM, scaled on the device


def transcribe(model, audio: AudioData, config: Optional[TranscribeConfig] = None) -> TranscribeResult:
    """One utterance, same contract as the reference (transcribe.py:30-60)."""
    if config is None:
        config = TranscribeConfig()
    wave = torch.from_numpy(_prepare(audio))
    hyp = model.transcribe([wave], batch_size=1, return_hypotheses=True, verbose=config.verbose)[0]
    result = decode_hypothesis(model, hyp)
    if config.raw_hypothesis:
        result.hypothesis = hyp
    return result


def transcribe_batch(model, audios: Sequence[AudioData], config: Optional[TranscribeConfig] = None) -> List[TranscribeResult]:
    """Many utterances through one or a few engine launches; results in input order.

    Same per-utterance semantics as ``transcribe`` (norm_audio, 0.5 s of silence on both sides, greedy decode,
    decode_hypothesis); the padding is written straight into the staging buffer and the post-processing of one batch
    overlaps the engine call of the next.  A model object without ``iter_token_batches`` (e.g. a real NeMo model)
    is driven through its ``transcribe`` method instead."""
    if config is None:
        config = TranscribeConfig()
    out: List[Optional[TranscribeResult]] = [None] * len(audios)

    def finish(i, hyp):
        r = decode_hypothesis(model, hyp)
        if config.raw_hypothesis:
            r.hypothesis = hyp
        out[i] = r

    if hasattr(model, "iter_token_batches") and getattr(model, "decoding", "greedy") == "greedy":
        blank = model.cfg.blank
        pad = int(PAD_SECONDS * SAMPLERATE)
        # audio that still needs norm_audio (another rate, several channels) and is uniform in both goes to the GPU as it is:
        # resampling, down-mixing and padding run there (iter_token_batches_raw); anything else is normalised on the host
        raw_ok = (hasattr(model, "iter_token_batches_raw") and len(audios) > 0 and
                  len({(a.samplerate, np.asarray(a.waveform).ndim, np.asarray(a.waveform).shape[0] if np.asarray(a.waveform).ndim == 2 else 1)
                       for a in audios}) == 1 and
                  (audios[0].samplerate != SAMPLERATE or np.asarray(audios[0].waveform).ndim == 2))
        if raw_ok:
            batches = model.iter_token_batches_raw([np.asarray(a.waveform) for a in audios], audios[0].samplerate, pad=pad)
        else:
            batches = model.iter_token_batches([np.asarray(norm_audio(a).waveform) for a in audios], pad=pad)
        for idx, items in batches:
            for i, (tokens, frames) in zip(idx, items):
                finish(i, Hypothesis.from_greedy(tokens, frames, blank))
    else:
        tensors = [torch.from_numpy(_prepare(a)) for a in audios]
        hyps = model.transcribe(tensors, batch_size=max(len(tensors), 1), return_hypotheses=True, verbose=config.verbose)
        for i, hyp in enumerate(hyps):
            finish(i, hyp)
    return out


def align(model, audio: AudioData, text: Union[str, Sequence[int]], config: Optional[TranscribeConfig] = None) -> AlignResult:
    """When is a known transcript said in ``audio``, and how well does the audio support it: RNN-T forced alignment of
    ``text`` (a string, tokenised with ``model.tokenizer.text_to_ids``, or a list of token ids).  The audio is prepared as
    ``transcribe`` prepares it (norm_audio, 0.5 s of silence on both sides); subwords and segments carry the times of the
    frames that emit the tokens on the most likely alignment.  Needs ``load_model(..., aligner=True)``."""
    return align_batch(model, [audio], [text], config)[0]


def align_batch(model, audios: Sequence[AudioData], texts: Sequence[Union[str, Sequence[int]]],
                config: Optional[TranscribeConfig] = None) -> List[AlignResult]:
    """``align`` for many utterances through a few engine launches; results in input order."""
    if config is None:
        config = TranscribeConfig()
    if len(texts) != len(audios):
        raise ValueError(f"align_batch: {len(audios)} audios but {len(texts)} texts")
    ids = [model.tokenizer.text_to_ids(t) if isinstance(t, str) else [int(i) for i in t] for t in texts]
    waves = [np.asarray(norm_audio(a).waveform) for a in audios]
    out: List[AlignResult] = []
    for tokens, (frames, tok_logp, viterbi, loglik) in zip(ids, model.align_tokens(waves, ids, pad=int(PAD_SECONDS * SAMPLERATE))):
        steps = [f + i + 1 for i, f in enumerate(frames)]             # Hypothesis.from_greedy's convention
        r = build_result(model.tokenizer, tokens, steps)
        out.append(AlignResult(r.text, r.subwords, r.segments,
                               hypothesis=Hypothesis.from_greedy(tokens, frames, model.cfg.blank) if config.raw_hypothesis else None,
                               log_likelihood=loglik, viterbi_log_prob=viterbi, token_log_probs=tok_logp))
    return out


def window_frames(start: float, end: float, T: int, pad_seconds: float = PAD_SECONDS) -> tuple:
    """Encoder frames [lo, hi) of the window [start, end] seconds of a recording encoded with ``pad_seconds`` of silence on both
    sides, clamped to [0, T]: frame f covers [0.08 f - pad, 0.08 (f + 1) - pad) s of the recording, so lo is the frame that
    holds ``start`` and hi - 1 the frame that holds ``end``.  lo >= hi means an empty window."""
    lo = math.floor((start + pad_seconds) / SECONDS_PER_STEP)
    hi = math.floor((end + pad_seconds) / SECONDS_PER_STEP) + 1
    return min(max(lo, 0), T), min(max(hi, 0), T)


def min_mean_confidence(path_logp: Sequence[float], L: int = CONFIDENCE_FRAMES) -> float:
    """Mean of the per-frame path log-probabilities of a span of n frames when n <= L, else the minimum over its n - L + 1
    windows of L consecutive frames of their mean (CTC segmentation's ``score_min_mean_over_L``, on this model's scale)."""
    x = np.asarray(path_logp, np.float64)
    if len(x) <= L:
        return float(x.mean())
    c = np.concatenate(([0.0], np.cumsum(x)))
    return float(((c[L:] - c[:-L]) / L).min())


def add_space(captions: Sequence[AlignedCaption]) -> None:
    """The oneseg "lax" strategy (pkg/espnet-oneseg/src/align.py:46-51), in place, over consecutive captions in list order:
    half the gap between two captions, clamped to [0, 3] s, is added to the earlier one's end and taken from the later one's
    start."""
    for c0, c1 in zip(captions, captions[1:]):
        gap = max(min((c1.start_seconds - c0.end_seconds) / 2, 3), 0)
        c0.end_seconds += gap
        c1.start_seconds -= gap


def align_captions(model, audio: AudioData, captions: Sequence[Caption], *, before: float = CAPTION_MARGIN, after: float = 0.0,
                   strategy: str = "optim", with_asr: bool = False) -> List[Optional[AlignedCaption]]:
    """Where in ``audio`` is each caption said: free-span RNN-T alignment of every caption's text inside the window from
    ``before`` seconds ahead of its start to ``after`` seconds past its end (live captions lag the speech by up to ~25 s),
    the question ReazonSpeech's corpus builder answers with CTC segmentation (pkg/espnet-oneseg/src/align.py:22-44) and the
    one that re-timing an SRT / WebVTT file against its audio poses.  The recording is prepared as ``transcribe`` prepares it
    (norm_audio, 0.5 s of silence on both sides) and encoded once; every caption is placed independently.  Results in input
    order, None for a caption that could not be placed (an empty window, or text that tokenises to nothing).
    ``strategy="lax"`` widens consecutive placed captions into half the gap between them (at most 3 s each side), as the
    reference's "lax" strategy does; ``with_asr=True`` fills ``asr`` and ``cer`` from one greedy ``transcribe_batch`` of the
    placed slices.  Needs ``load_model(..., aligner=True)``."""
    return align_captions_batch(model, [audio], [captions], before=before, after=after, strategy=strategy, with_asr=with_asr)[0]


def align_captions_batch(model, audios: Sequence[AudioData], caption_lists: Sequence[Sequence[Caption]], *,
                         before: float = CAPTION_MARGIN, after: float = 0.0, strategy: str = "optim",
                         with_asr: bool = False) -> List[List[Optional[AlignedCaption]]]:
    """``align_captions`` for many recordings, cut into length-sorted batches; results in input order."""
    if strategy not in ("optim", "lax"):
        raise ValueError(f"strategy must be 'optim' or 'lax', got {strategy!r}")
    if len(caption_lists) != len(audios):
        raise ValueError(f"align_captions_batch: {len(audios)} audios but {len(caption_lists)} caption lists")
    for caps in caption_lists:
        for c in caps:
            if c.start_seconds > c.end_seconds:
                raise ValueError(f"caption {c.text!r} starts at {c.start_seconds} s, after its end {c.end_seconds} s")
    waves = [np.asarray(norm_audio(a).waveform) for a in audios]
    ids = [[model.tokenizer.text_to_ids(c.text) for c in caps] for caps in caption_lists]
    windows = [[(c.start_seconds - before, c.end_seconds + after) for c in caps] for caps in caption_lists]
    placed = model.align_caption_tokens(waves, windows, ids, pad=int(PAD_SECONDS * SAMPLERATE))
    out: List[List[Optional[AlignedCaption]]] = []
    for wave, caps, toks, res in zip(waves, caption_lists, ids, placed):
        duration = len(wave) / SAMPLERATE
        row: List[Optional[AlignedCaption]] = []
        for c, tokens, r in zip(caps, toks, res):
            if r is None:
                row.append(None)
                continue
            lo, frames, tok_logp, path_logp, viterbi, loglik = r
            steps = [f + i + 1 for i, f in enumerate(frames)]            # Hypothesis.from_greedy's convention
            start = min(max(SECONDS_PER_STEP * frames[0] - PAD_SECONDS, 0), duration)
            end = min(max(SECONDS_PER_STEP * frames[-1] - PAD_SECONDS, 0) + SECONDS_PER_STEP, duration)
            row.append(AlignedCaption(start, end, c.text, min_mean_confidence(path_logp[frames[0] - lo: frames[-1] - lo + 1]),
                                      viterbi, loglik, build_result(model.tokenizer, tokens, steps).subwords, tok_logp))
        out.append(row)
    if strategy == "lax":
        for row in out:
            add_space([r for r in row if r is not None])
    if with_asr:
        from ...evaluation.utils import calculate_cer, normalize
        slices, where = [], []
        for wave, row in zip(waves, out):
            for r in row:
                if r is not None:
                    slices.append(AudioData(wave[int(r.start_seconds * SAMPLERATE): int(r.end_seconds * SAMPLERATE)], SAMPLERATE))
                    where.append(r)
        for r, t in zip(where, transcribe_batch(model, slices) if slices else []):
            r.asr = t.text
            r.cer = calculate_cer(r.text, r.asr)["cer"] if normalize(r.text) else None
    return out
