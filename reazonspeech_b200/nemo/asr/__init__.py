"""Drop-in for ``reazonspeech.nemo.asr`` (pkg/nemo-asr/src/__init__.py:1-3) plus ``transcribe_batch``, forced alignment
(``align`` / ``align_batch``) and caption placement in longer audio (``align_captions`` / ``align_captions_batch``)."""
from .interface import AlignedCaption, AlignResult, Caption, TranscribeConfig
from .transcribe import align, align_batch, align_captions, align_captions_batch, transcribe, transcribe_batch, load_model
from .audio import audio_from_numpy, audio_from_tensor, audio_from_path
from .captions import read_captions

__all__ = ["TranscribeConfig", "transcribe", "transcribe_batch", "load_model",
           "audio_from_numpy", "audio_from_tensor", "audio_from_path", "align", "align_batch", "AlignResult",
           "Caption", "AlignedCaption", "align_captions", "align_captions_batch", "read_captions"]
