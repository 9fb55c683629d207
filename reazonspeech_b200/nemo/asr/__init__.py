"""Drop-in for ``reazonspeech.nemo.asr`` (pkg/nemo-asr/src/__init__.py:1-3) plus ``transcribe_batch`` and forced alignment
(``align`` / ``align_batch``)."""
from .interface import AlignResult, TranscribeConfig
from .transcribe import align, align_batch, transcribe, transcribe_batch, load_model
from .audio import audio_from_numpy, audio_from_tensor, audio_from_path

__all__ = ["TranscribeConfig", "transcribe", "transcribe_batch", "load_model",
           "audio_from_numpy", "audio_from_tensor", "audio_from_path", "align", "align_batch", "AlignResult"]
