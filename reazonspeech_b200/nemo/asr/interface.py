"""Argument / result types of the ``reazonspeech.nemo.asr`` API.

Field names, order and defaults follow the reference dataclasses
(pkg/nemo-asr/src/interface.py:4-36) so results are interchangeable; the extra helpers are ours."""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Any, List, Optional

import numpy as np


@dataclass
class AudioData:
    """A waveform (float array, mono [n] or channels-first [c, n]) and its sample rate."""
    waveform: np.ndarray
    samplerate: int

    @property
    def seconds(self) -> float:
        return self.waveform.shape[-1] / float(self.samplerate)


@dataclass
class Subword:
    """One emitted token with the time of the encoder frame that emitted it."""
    seconds: float
    token_id: int
    token: str

    def as_dict(self) -> dict:
        return {"seconds": self.seconds, "token_id": self.token_id, "token": self.token}


@dataclass
class Segment:
    """A run of subwords ending at a sentence mark, a comma or a pause (decode.find_end_of_segment)."""
    start_seconds: float
    end_seconds: float
    text: str

    @property
    def duration(self) -> float:
        return self.end_seconds - self.start_seconds

    def as_dict(self) -> dict:
        return {"start_seconds": self.start_seconds, "end_seconds": self.end_seconds, "text": self.text}


@dataclass
class TranscribeResult:
    """What ``transcribe`` / ``transcribe_batch`` return.  ``hypothesis`` is only filled when the call was made with
    ``TranscribeConfig(raw_hypothesis=True)``; it then carries the engine's token ids and ALSD-shaped step counters."""
    text: str
    subwords: List[Subword]
    segments: List[Segment]
    hypothesis: Any = None

    def as_dict(self) -> dict:
        """Plain-Python form (no hypothesis) for JSON-lines outputs such as the evaluator's."""
        return {"text": self.text, "subwords": [w.as_dict() for w in self.subwords],
                "segments": [g.as_dict() for g in self.segments]}

    @property
    def token_ids(self) -> List[int]:
        return [w.token_id for w in self.subwords]


@dataclass
class AlignResult(TranscribeResult):
    """What ``align`` / ``align_batch`` return: the transcript's subwords and segments timed by the most likely alignment, plus
    ``log_likelihood`` (log p(text | audio) summed over every alignment: minus the RNN-T loss), ``viterbi_log_prob`` (log p of
    the best alignment alone) and ``token_log_probs`` (log p of every target token where that alignment emits it; one entry
    per token id, including ids that decode to no text and so have no subword)."""
    log_likelihood: float = 0.0
    viterbi_log_prob: float = 0.0
    token_log_probs: List[float] = field(default_factory=list)


@dataclass
class Caption:
    """A caption to be found in a recording: the text and the time it was displayed (for a live caption: some seconds after
    the words were said).  Field names and order follow the reference's oneseg ``Caption`` (pkg/espnet-oneseg/src/interface.py)."""
    start_seconds: float
    end_seconds: float
    text: str


@dataclass
class AlignedCaption:
    """What ``align_captions`` returns for a caption it placed.  Times are on the recording's own axis: ``start_seconds`` is
    the time of the frame that emits the caption's first token on the best path, ``end_seconds`` the time of the frame of its
    last token plus one frame (clipped to the recording).  ``confidence`` is the minimum, over windows of 30 encoder frames
    (2.4 s), of the mean per-frame log-probability of that path (the plain mean for a shorter span): the analogue of CTC
    segmentation's ``score_min_mean_over_L``, on this model's scale, not comparable with ESPnet's numbers.
    ``viterbi_log_prob`` is the best path's log p, ``log_likelihood`` the log p summed over every span and path of the window,
    ``token_log_probs`` the log p of every token id where the best path emits it.  ``asr`` / ``cer``: the engine's greedy
    transcript of the placed slice and its character error rate against ``text`` (``with_asr=True``; ``cer`` is None when
    the normalised caption is empty)."""
    start_seconds: float
    end_seconds: float
    text: str
    confidence: float
    viterbi_log_prob: float
    log_likelihood: float
    subwords: List[Subword] = field(default_factory=list)
    token_log_probs: List[float] = field(default_factory=list)
    asr: Optional[str] = None
    cer: Optional[float] = None

    @property
    def duration(self) -> float:
        return self.end_seconds - self.start_seconds


@dataclass
class TranscribeConfig:
    verbose: bool = True
    raw_hypothesis: bool = False
