"""The CLI's --align option with a stub model (no GPU): transcript lines are matched to the AUDIO arguments in order, a line
count that differs is refused with exit status 1, and the aligned segments go through the same writers and time shift as
transcripts do.  Also the one-process multi-GPU model's refusal to align."""
import importlib

import numpy as np
import pytest

from reazonspeech_b200.nemo.asr import cli
from reazonspeech_b200.nemo.asr.interface import AlignResult, Segment


def _wavs(tmp_path, secs):
    from scipy.io import wavfile
    paths = []
    for i, s in enumerate(secs):
        p = tmp_path / f"a{i}.wav"
        wavfile.write(p, 16000, np.zeros(int(s * 16000), np.int16))
        paths.append(str(p))
    return paths


def test_align_line_count_mismatch_exits_1(tmp_path, capsys):
    paths = _wavs(tmp_path, (1.0, 2.0))
    lines = tmp_path / "t.txt"
    lines.write_text("あいう\n", encoding="utf-8")
    assert cli.main([f"--align={lines}", *paths]) == 1
    assert "1 transcript lines for 2 audio files" in capsys.readouterr().err


def test_align_writes_the_aligned_segments(tmp_path, monkeypatch):
    T = importlib.import_module("reazonspeech_b200.nemo.asr.transcribe")
    paths = _wavs(tmp_path, (2.0, 3.5))
    lines = tmp_path / "t.txt"
    lines.write_text("あいう\nかき く\n", encoding="utf-8")
    seen = {}

    def load_model(*a, **k):
        seen["load"] = k
        return object()

    def align_batch(model, audios, texts, config=None):
        seen["texts"] = list(texts)
        return [AlignResult(t, [], [Segment(0.25 * (i + 1), 0.75, t)], log_likelihood=-1.0) for i, t in enumerate(texts)]

    monkeypatch.setattr(T, "load_model", load_model)
    monkeypatch.setattr(T, "align_batch", align_batch)
    monkeypatch.setattr(T, "transcribe", lambda *a, **k: pytest.fail("--align must not transcribe"))
    monkeypatch.setattr(T, "transcribe_batch", lambda *a, **k: pytest.fail("--align must not transcribe"))
    out = tmp_path / "o.tsv"
    assert cli.main(["--to=tsv", f"--align={lines}", "-o", str(out), *paths]) is None
    assert seen["load"] == {"aligner": True} and seen["texts"] == ["あいう", "かき く"]
    rows = [l.split("\t") for l in out.read_text().splitlines()[1:]]
    assert [(float(r[0]), r[2]) for r in rows] == [(0.25, "あいう"), (2.5, "かき く")]     # second file shifted by the first's 2.0 s


def test_multi_gpu_model_does_not_align():
    from reazonspeech_b200.nemo.asr import align
    from reazonspeech_b200.nemo.asr.audio import audio_from_numpy
    from reazonspeech_b200.nemo.asr.multi_gpu import MultiGpuRnntModel

    class Replica:
        cfg, tokenizer, max_batch = None, None, 8

    with pytest.raises(NotImplementedError):
        align(MultiGpuRnntModel([Replica()]), audio_from_numpy(np.zeros(16000, np.float32), 16000), [1, 2])
