"""Caption placement on the host, without a GPU: seconds -> window frames, result times and clipping, the None cases, input
order across length-sorted batches (B200RnntModel.align_caption_tokens over a stand-in engine), the "lax" widening, with_asr
on a caption that normalises to nothing, the min-mean confidence against the oracle, the SRT / WebVTT reader and the CLI's
--align-captions."""
import importlib

import numpy as np
import pytest
import torch

from oracle import align_spans_restated as S
from reazonspeech_b200.nemo.asr import Caption, cli
from reazonspeech_b200.nemo.asr.captions import parse_captions, read_captions
from reazonspeech_b200.nemo.asr.interface import AlignedCaption, Segment, TranscribeResult
from reazonspeech_b200.nemo.asr.writer import SRTWriter, VTTWriter
from reazonspeech_b200.tokenizer import PieceTableTokenizer, synthetic_pieces

T = importlib.import_module("reazonspeech_b200.nemo.asr.transcribe")
SR = 16000


# ---------------------------------------------------------------------------------------------- seconds -> frames
def test_window_frames():
    assert T.window_frames(1.0, 2.0, 100) == (18, 32)              # floor(1.5 / 0.08), floor(2.5 / 0.08) + 1
    assert T.window_frames(-0.5, 0.0, 100) == (0, 7)               # frame 0 starts at -0.5 s: the padding
    assert T.window_frames(-30.0, 5.0, 40) == (0, 40)              # clamped to [0, T]
    assert T.window_frames(50.0, 60.0, 40) == (40, 40)             # past the end: an empty window
    assert T.window_frames(-9.0, -8.0, 40) == (0, 0)               # before the start: an empty window
    lo, hi = T.window_frames(3.0, 3.0, 100)
    assert hi - lo == 1 and lo * 0.08 - 0.5 <= 3.0 < (lo + 1) * 0.08 - 0.5


def test_confidence_matches_the_oracle():
    rng = np.random.default_rng(3)
    for n in (1, 7, 29, 30, 31, 200):
        x = (-rng.exponential(1.0, n)).astype(np.float32).tolist()
        assert T.min_mean_confidence(x) == pytest.approx(S.span_confidence(x, 0, n - 1), rel=1e-12, abs=1e-12)
    assert T.CONFIDENCE_FRAMES == S.CONFIDENCE_FRAMES


# ---------------------------------------------------------------------------------------------- stand-in models
class StubModel:
    """align_caption_tokens returns frames it was told to; records what it was given."""

    def __init__(self, frames_for):
        self.tokenizer = PieceTableTokenizer(synthetic_pieces(127))
        self.frames_for = frames_for                     # caption text -> (lo, frames)
        self.calls = []

    def align_caption_tokens(self, waveforms, windows, token_lists, pad=0):
        self.calls.append((waveforms, windows, token_lists, pad))
        out = []
        for caps, toks in zip(windows, token_lists):
            row = []
            for w, t in zip(caps, toks):
                key = tuple(t)
                if not t or key not in self.frames_for:
                    row.append(None)
                    continue
                lo, fr = self.frames_for[key]
                path = [0.0] * (fr[-1] - lo + 5)
                for f in range(fr[0], fr[-1] + 1):
                    path[f - lo] = -0.25
                row.append((lo, list(fr), [-0.5] * len(t), path, -1.0 * len(t), -0.5 * len(t)))
            out.append(row)
        return out


def _audio(seconds):
    from reazonspeech_b200.nemo.asr.audio import audio_from_numpy
    return audio_from_numpy(np.zeros(int(seconds * SR), np.float32), SR)


def test_times_clipping_and_none():
    tok = PieceTableTokenizer(synthetic_pieces(127))
    a, b, c = (tuple(tok.text_to_ids(t)) for t in ("あいう", "かき", "さ"))
    model = StubModel({a: (10, [20, 21, 25]), b: (0, [2, 3]), c: (100, [131])})
    caps = [Caption(30.0, 31.0, "あいう"), Caption(0.0, 1.0, "かき"), Caption(5.0, 6.0, ""), Caption(9.0, 10.0, "さ")]
    got = T.align_captions(model, _audio(10.0), caps, before=25.0, after=0.5)
    waves, windows, toks, pad = model.calls[0]
    assert pad == 8000 and len(waves[0]) == 10 * SR
    assert windows == [[(5.0, 31.5), (-25.0, 1.5), (-20.0, 6.5), (-16.0, 10.5)]]
    assert toks[0][2] == []
    r0, r1, r2, r3 = got
    assert r2 is None                                                 # text that tokenises to nothing
    assert r0.start_seconds == pytest.approx(0.08 * 20 - 0.5) and r0.end_seconds == pytest.approx(0.08 * 25 - 0.5 + 0.08)
    assert r0.text == "あいう" and r0.viterbi_log_prob == -3.0 and r0.log_likelihood == -1.5
    assert r0.confidence == pytest.approx(-0.25) and r0.duration == pytest.approx(r0.end_seconds - r0.start_seconds)
    assert [w.seconds for w in r0.subwords] == pytest.approx([0.08 * f - 0.5 for f in (20, 21, 25)])
    assert r1.start_seconds == 0.0 and r1.end_seconds == pytest.approx(0.08)   # times inside the leading padding clip to 0
    assert r3.start_seconds == pytest.approx(0.08 * 131 - 0.5) and r3.end_seconds == 10.0   # clipped to the recording
    with pytest.raises(ValueError, match="after its end"):
        T.align_captions(model, _audio(10.0), [Caption(3.0, 2.0, "あ")])
    with pytest.raises(ValueError, match="strategy"):
        T.align_captions(model, _audio(10.0), caps, strategy="tight")


def test_lax_widens_into_half_the_gap():
    tok = PieceTableTokenizer(synthetic_pieces(127))
    texts = ["あ", "い", "う", "え", "お"]
    frames = {tuple(tok.text_to_ids("あ")): (0, [7, 11]), tuple(tok.text_to_ids("い")): (0, [25, 31]),
              tuple(tok.text_to_ids("え")): (0, [132, 136]), tuple(tok.text_to_ids("お")): (0, [134, 144])}
    caps = [Caption(i, i + 1.0, t) for i, t in enumerate(texts)]
    optim = T.align_captions(StubModel(frames), _audio(20.0), caps)
    lax = T.align_captions(StubModel(frames), _audio(20.0), caps, strategy="lax")
    assert optim[2] is None and lax[2] is None
    se = lambda r: (round(r.start_seconds, 6), round(r.end_seconds, 6))
    assert [se(r) for r in optim if r] == [(0.06, 0.46), (1.5, 2.06), (10.06, 10.46), (10.22, 11.1)]
    # gap 1.04 -> 0.52 each side; gap 7.96 -> 3.98 clamped to 3; overlap (-0.24) -> 0
    assert [se(r) for r in lax if r] == [(0.06, 0.98), (0.98, 5.06), (7.06, 10.46), (10.22, 11.1)]


def test_with_asr_and_an_empty_normalised_caption(monkeypatch):
    tok = PieceTableTokenizer(synthetic_pieces(127))
    from reazonspeech_b200.evaluation.utils import normalize
    assert normalize("。") == "" and tok.text_to_ids("。")
    frames = {tuple(tok.text_to_ids("あいう")): (0, [20, 30]), tuple(tok.text_to_ids("。")): (0, [40, 41])}
    seen = []

    def transcribe_batch(model, audios, config=None):
        seen.append([len(a.waveform) for a in audios])
        return [TranscribeResult("あいえ", [], []), TranscribeResult("あ", [], [])]

    monkeypatch.setattr(T, "transcribe_batch", transcribe_batch)
    got = T.align_captions(StubModel(frames), _audio(5.0), [Caption(1.0, 2.0, "あいう"), Caption(2.0, 3.0, "。")], with_asr=True)
    assert len(seen) == 1                                              # one batch for every placed slice
    assert seen[0][0] == int(got[0].end_seconds * SR) - int(got[0].start_seconds * SR)
    assert got[0].asr == "あいえ" and got[0].cer == pytest.approx(1 / 3)
    assert got[1].asr == "あ" and got[1].cer is None                   # calculate_cer would divide by zero


# ---------------------------------------------------------------------------------------------- batching over a stand-in engine
class FakeEngine:
    """Stands in for Engine: 'encodes' a batch into one frame per 1280 samples whose value is the row's sample count, and
    'aligns' every caption at the start of its window with viterbi = the value of its source row."""
    device = "cpu"
    weights = {"alsd.out.w3": None}

    def __init__(self):
        self.calls = []

    def log_mel(self, x, lens):
        return x, lens

    def encode(self, x, lens):
        T = int(x.shape[1]) // 1280
        enc = lens.to(torch.float32)[:, None, None].expand(x.shape[0], T, 1).contiguous()
        return enc, (lens // 1280).to(torch.int32)

    def align_spans(self, enc, enc_len, spans, targets, tgt_len):
        self.calls.append(spans.shape[0])
        K, U = targets.shape
        frames = spans[:, 1:2] + torch.arange(U, dtype=torch.int32)[None]
        F = int((spans[:, 2] - spans[:, 1]).max())
        vit = torch.stack([enc[int(s), int(lo), 0] for s, lo, _ in spans.tolist()]).to(torch.float64)
        return frames, torch.zeros(K, U), -torch.ones(K, F), vit, vit + 1


def test_caption_tokens_come_back_in_input_order(monkeypatch):
    import contextlib
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    eng = FakeEngine()
    model = T.B200RnntModel.__new__(T.B200RnntModel)
    model.engine, model.max_batch = eng, 2
    model._staging = (T.HostStaging(False), T.HostStaging(False))
    secs = [6.0, 2.0, 4.0, 3.0, 5.0]
    waves = [np.zeros(int(s * SR), np.float32) for s in secs]
    windows = [[(0.0, 1.0), (s - 1.0, s), (s + 5.0, s + 6.0)] for s in secs]
    toks = [[[1, 2], [3], [4]] for _ in secs]
    toks[3][1] = []
    out = model.align_caption_tokens(waves, windows, toks, pad=8000)
    assert eng.calls == [3, 4, 2]                                      # batches {2, 3}, {4, 5}, {6} seconds; empty items left out
    for s, w, row, tl in zip(secs, windows, out, toks):
        n = int(s * SR) + 16000
        assert row[2] is None                                          # past the end of the recording
        assert (row[1] is None) == (tl[1] == [])
        for (start, end), r, t in zip(w, row, tl):
            if r is None:
                continue
            lo, frames, tok_logp, path_logp, vit, ll = r
            assert (lo, len(path_logp)) == (T.window_frames(start, end, n // 1280)[0], T.window_frames(start, end, n // 1280)[1] - lo)
            assert frames == [lo + i for i in range(len(t))] and vit == n and ll == n + 1


def test_caption_tokens_need_the_aligner_weights():
    eng = FakeEngine()
    eng.weights = {}
    model = T.B200RnntModel.__new__(T.B200RnntModel)
    model.engine = eng
    with pytest.raises(RuntimeError, match="aligner=True"):
        model.align_caption_tokens([np.zeros(SR, np.float32)], [[(0.0, 1.0)]], [[[1]]])


def test_multi_gpu_model_does_not_align_captions():
    from reazonspeech_b200.nemo.asr import align_captions
    from reazonspeech_b200.nemo.asr.multi_gpu import MultiGpuRnntModel

    class Replica:
        cfg, max_batch = None, 8
        tokenizer = PieceTableTokenizer(synthetic_pieces(127))

    with pytest.raises(NotImplementedError):
        align_captions(MultiGpuRnntModel([Replica()]), _audio(1.0), [Caption(0.0, 1.0, "あ")])


# ---------------------------------------------------------------------------------------------- SRT / WebVTT reader
SEGS = [Segment(0.0, 1.5, "あいう"), Segment(61.25, 3725.125, "かき く"), Segment(3725.5, 3726.0, "さ")]


@pytest.mark.parametrize("writer", [SRTWriter, VTTWriter])
def test_read_captions_round_trips_the_writers(tmp_path, writer):
    p = tmp_path / f"x.{writer.ext}"
    with open(p, "w", encoding="utf-8") as f:
        w = writer(f)
        w.write_header()
        for s in SEGS:
            w.write(s)
    got = read_captions(str(p))
    assert [(c.start_seconds, c.end_seconds, c.text) for c in got] == [(s.start_seconds, s.end_seconds, s.text) for s in SEGS]


def test_read_hand_written_files(tmp_path):
    vtt = ("﻿WEBVTT - broadcast\r\nKind: captions\r\n\r\nNOTE this is\r\na comment\r\n\r\nSTYLE\r\n::cue { color: red }\r\n\r\n"
           "intro\r\n00:01.000 --> 00:02.500 align:start position:10%\r\nこんにちは\r\n世界\r\n\r\n"
           "01:00:00.250 --> 01:00:01.000\r\nさようなら\r\n")
    p = tmp_path / "a.vtt"
    p.write_bytes(vtt.encode("utf-8"))
    assert [(c.start_seconds, c.end_seconds, c.text) for c in read_captions(str(p))] == [
        (1.0, 2.5, "こんにちは 世界"), (3600.25, 3601.0, "さようなら")]
    srt = "1\r\n00:00:01,000 --> 00:00:02,000\r\nひとつ\r\nふたつ\r\n\r\n\r\n2\r\n00:00:03,5 --> 00:00:04,250\r\nみっつ\r\n"
    assert [(c.start_seconds, c.end_seconds, c.text) for c in parse_captions(srt)] == [(1.0, 2.0, "ひとつ ふたつ"), (3.5, 4.25, "みっつ")]
    # an SRT file whose first cue text happens to read WEBVTT further down is still SRT
    assert parse_captions("1\n00:00:00,000 --> 00:00:01,000\nWEBVTT\n")[0].text == "WEBVTT"
    with pytest.raises(ValueError):
        parse_captions("1\n00:00:xx,000 --> 00:00:01,000\nbad\n")


# ---------------------------------------------------------------------------------------------- CLI
def _wavs(tmp_path, secs):
    from scipy.io import wavfile
    paths = []
    for i, s in enumerate(secs):
        p = tmp_path / f"a{i}.wav"
        wavfile.write(p, SR, np.zeros(int(s * SR), np.int16))
        paths.append(str(p))
    return paths


def test_cli_exit_1_cases(tmp_path, capsys):
    paths = _wavs(tmp_path, (1.0, 2.0))
    srt = tmp_path / "c.srt"
    srt.write_text("1\n00:00:00,500 --> 00:00:01,000\nあ\n", encoding="utf-8")
    assert cli.main([f"--align-captions={srt}", *paths]) == 1
    assert "one audio file, got 2" in capsys.readouterr().err
    txt = tmp_path / "t.txt"
    txt.write_text("あ\n", encoding="utf-8")
    assert cli.main([f"--align-captions={srt}", f"--align={txt}", paths[0]]) == 1
    assert "cannot be combined" in capsys.readouterr().err
    assert cli.main([f"--align-captions={srt}"]) == 1
    assert "no audio file specified" in capsys.readouterr().err


def test_cli_writes_the_placed_captions(tmp_path, monkeypatch, capsys):
    paths = _wavs(tmp_path, (4.0,))
    vtt = tmp_path / "c.vtt"
    vtt.write_text("WEBVTT\n\n00:00:01.000 --> 00:00:02.000\nあ\n\n00:00:02.000 --> 00:00:03.000\nい\n\n"
                   "00:00:03.000 --> 00:00:03.500\nう\n", encoding="utf-8")
    seen = {}

    def load_model(*a, **k):
        seen["load"] = k
        return object()

    def align_captions(model, audio, captions, **k):
        seen["captions"] = [(c.start_seconds, c.end_seconds, c.text) for c in captions]
        seen["seconds"] = audio.seconds
        return [AlignedCaption(0.25, 0.75, "あ", -1.0, -2.0, -1.5), None, AlignedCaption(2.5, 3.25, "う", -1.0, -2.0, -1.5)]

    monkeypatch.setattr(T, "load_model", load_model)
    monkeypatch.setattr(T, "align_captions", align_captions)
    out = tmp_path / "o.tsv"
    assert cli.main(["--to=tsv", f"--align-captions={vtt}", "-o", str(out), paths[0]]) is None
    assert seen == {"load": {"aligner": True}, "captions": [(1.0, 2.0, "あ"), (2.0, 3.0, "い"), (3.0, 3.5, "う")], "seconds": 4.0}
    rows = [l.split("\t") for l in out.read_text().splitlines()[1:]]
    assert [(float(r[0]), float(r[1]), r[2]) for r in rows] == [(0.25, 0.75, "あ"), (2.5, 3.25, "う")]
    assert "1 of 3 captions could not be placed" in capsys.readouterr().err
