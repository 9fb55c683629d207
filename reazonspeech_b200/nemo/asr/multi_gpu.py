"""One process, several B200s: the same model object surface as ``B200RnntModel`` over one engine replica per device.

north_star: "utterance batches shard embarrassingly across the 8 GPUs of one box (no NCCL on the hot path)".  The
reference's only scale-out is one spawned process per GPU, each with its own model, merged through files
(pkg/evaluation/src/base.py:194-212, examples/rs-nemo/eval.py:19-27).  Here ``load_model(devices=[0, 1, ...])`` keeps
everything in one process: a full weight replica, a worker thread and a pinned staging pair per device; the utterances of
a call are dealt to the devices by length (``sharding.shard_indices``: longest first to the least-loaded device), every
replica runs its own batched pipeline (staging of batch k+1 overlaps the engine call of batch k), results are merged by
utterance index, so the output order is the input order whatever the devices' relative speed.  No collective, no
peer-to-peer traffic: an utterance never leaves its device.  The engine's C calls select their device themselves
(cudaSetDevice per call, per thread) and ctypes drops the GIL while they run, so the replicas run concurrently.
"""
from __future__ import annotations

import queue
import threading
from typing import List, Sequence

import numpy as np

from ...sharding import shard_indices


class MultiGpuRnntModel:
    """``replicas``: ``B200RnntModel`` objects, one per device, same weights.  Duck-typed like a single replica:
    ``iter_token_batches`` / ``transcribe_tokens`` / ``transcribe`` / ``tokenizer`` / ``cfg``."""

    def __init__(self, replicas: Sequence):
        if len(replicas) == 0:
            raise ValueError("MultiGpuRnntModel needs at least one replica")
        self.replicas = list(replicas)
        self.cfg = self.replicas[0].cfg
        self.tokenizer = self.replicas[0].tokenizer
        self.max_batch = self.replicas[0].max_batch

    @property
    def devices(self) -> List[str]:
        return [str(r.engine.device) for r in self.replicas]

    def iter_token_batches(self, waveforms: Sequence[np.ndarray], pad: int = 0):
        """Yields ``(indices, [(tokens, frames)])`` per finished engine batch of any device, indices into ``waveforms``."""
        if len(waveforms) == 0:
            return
        shards = [s for s in shard_indices([len(w) for w in waveforms], len(self.replicas))]
        out: "queue.Queue" = queue.Queue()

        def work(replica, mine: List[int]):
            try:
                sub = [waveforms[i] for i in mine]
                for idx, items in replica.iter_token_batches(sub, pad):
                    out.put(([mine[j] for j in idx], items))
            except BaseException as exc:          # surfaced on the caller's thread: a dead device must not look like a slow one
                out.put(exc)
            finally:
                out.put(None)

        threads = [threading.Thread(target=work, args=(r, s), daemon=True) for r, s in zip(self.replicas, shards) if s]
        for t in threads:
            t.start()
        running, error = len(threads), None
        while running:
            item = out.get()
            if item is None:
                running -= 1
            elif isinstance(item, BaseException):
                error = error or item
            elif error is None:
                yield item
        for t in threads:
            t.join()
        if error is not None:
            raise error

    def transcribe_tokens(self, waveforms: Sequence[np.ndarray], pad: int = 0):
        """-> [(tokens, frames)] in input order."""
        results = [None] * len(waveforms)
        for idx, items in self.iter_token_batches(waveforms, pad):
            for i, item in zip(idx, items):
                results[i] = item
        return results

    def align_tokens(self, waveforms, token_lists, pad: int = 0):
        raise NotImplementedError("the one-process multi-GPU model does not align; load one model per device for align()")

    def align_caption_tokens(self, waveforms, windows, token_lists, pad: int = 0):
        raise NotImplementedError("the one-process multi-GPU model does not align; load one model per device for align_captions()")

    def transcribe(self, audio, batch_size: int = 1, return_hypotheses: bool = True, verbose: bool = True, **_):
        """NeMo's call shape (pkg/nemo-asr/src/transcribe.py:48-53) over all devices."""
        import torch
        from .transcribe import Hypothesis
        waves = [a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a) for a in audio]
        hyps = [Hypothesis.from_greedy(t, f, self.cfg.blank) for t, f in self.transcribe_tokens(waves)]
        if return_hypotheses:
            return hyps
        return [self.tokenizer.ids_to_text(h.y_sequence.tolist()[1:]) for h in hyps]
