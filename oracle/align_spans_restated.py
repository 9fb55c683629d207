"""CPU oracle of free-span RNN-T alignment: where inside a window of frames is a GIVEN token sequence said -- the question a
broadcast caption poses when it is searched for in the audio around its display time (rs_rnnt_align_spans).

THIS IS TEST INFRASTRUCTURE (see oracle/nemo_restated.py): only tests/, smoke() and the benchmark scripts may import it.

One caption has an encoder row ``src``, a frame window [lo, hi) of that row (W = hi - lo >= 1) and targets y_1..y_U (U >= 1).
Its lattice is exactly ``align_restated.lattice(enc[src, lo:hi], targets)``: nodes (t, u), t in [0, W), u in [0, U], each with
lb(t, u) and ly(t, u); the predictor state depends on u only and f on the frame only.  The path may begin at any node (t_s, 0)
at no cost and must end with the closing blank of some frame t_e at u = U:

    alpha(0, 0) = 0
    alpha(t, 0) = max(0 [fresh start], alpha(t-1, 0) + lb(t-1, 0))                     t >= 1
    alpha(t, u) = max(alpha(t-1, u) + lb(t-1, u), alpha(t, u-1) + ly(t, u-1))        u >= 1   (as align_restated)
    viterbi = max_t alpha(t, U) + lb(t, U)

The forward score is the same recursion with logaddexp in place of max: logaddexp(0, beta(t-1, 0) + lb(t-1, 0)) at u = 0 and
loglik = logsumexp_t beta(t, U) + lb(t, U), the end terms folded in ascending t.  Everything accumulates in float64 from the
fp32 lattice.  Identities: viterbi = max over t_s <= t_e of rnnt_viterbi(lat[t_s:t_e+1]).score and loglik = logsumexp over
t_s <= t_e of rnnt_forward(lat[t_s:t_e+1]).

Tie rules: at u = 0 an exact tie goes to the fresh start; at the end an exact tie goes to the earliest t_e; inside the lattice
the blank edge wins (as align_restated).  Every lb <= 0 (the lattice stores blank - lse with lse >= the row maximum), so with
these rules the best span is exactly [frames[0], frames[U-1]]: extra leading or trailing blanks never add to the score.

path_logp[t] for t in the span is lb(t, u_t) + the ly of the tokens the best path emits at t, u_t the path's u after frame t,
summed in fp32 in that order (the blank first, then the tokens from the last to the first -- the order of the GPU's backtrace);
frames outside the span hold 0.  Its sum is the Viterbi score up to fp32 rounding.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence

import numpy as np

CONFIDENCE_FRAMES = 30           # L: 30 encoder frames = 2.4 s, the window of span_confidence


@dataclass
class SpanPath:
    score: float                 # Viterbi log-probability of the best (span, path)
    frames: List[int]            # emitting window frame of every token
    tok_logp: List[float]        # ly(frames[u], u)
    path_logp: List[float]       # per window frame: the path's log p at that frame, 0 outside the span


def _sweep(lat: np.ndarray, viterbi: bool):
    W, U1 = lat.shape[0], lat.shape[1]
    U = U1 - 1
    lb = lat[..., 0].astype(np.float64)
    ly = lat[..., 1].astype(np.float64)
    a = np.full((W, U1), -np.inf)
    bp = np.zeros((W, U1), np.int8)                                  # 0 blank, 1 emit, 2 fresh start
    for t in range(W):
        for u in range(U1):
            if t == 0 and u == 0:
                a[0, 0], bp[0, 0] = 0.0, 2
                continue
            vb = a[t - 1, u] + lb[t - 1, u] if t > 0 else -np.inf
            if u == 0:
                if viterbi:
                    bp[t, 0] = 0 if vb > 0.0 else 2                   # exact tie: the fresh start
                    a[t, 0] = vb if bp[t, 0] == 0 else 0.0
                else:
                    a[t, 0] = np.logaddexp(0.0, vb)
                continue
            ve = a[t, u - 1] + ly[t, u - 1]
            if viterbi:
                bp[t, u] = ve > vb                                   # exact tie: the blank edge
                a[t, u] = ve if bp[t, u] else vb
            else:
                a[t, u] = np.logaddexp(vb, ve)
    best, t_e = -np.inf, 0
    for t in range(W):                                                # ascending t
        x = a[t, U] + lb[t, U]
        if t == 0:
            best = x
        elif viterbi:
            if x > best:                                             # exact tie: the earliest t_e
                best, t_e = x, t
        else:
            best = np.logaddexp(best, x)
    return bp, float(best), t_e


def rnnt_span_viterbi(lat: np.ndarray) -> SpanPath:
    """Best free-span path through a [W, U + 1, 2] lattice (U >= 1), float64, with the tie rules of the module docstring."""
    W, U = lat.shape[0], lat.shape[1] - 1
    assert W >= 1 and U >= 1
    bp, score, t = _sweep(lat, True)
    frames, logp = [0] * U, [0.0] * U
    path = np.zeros(W, np.float32)
    u = U
    acc = np.float32(lat[t, U, 0])
    while True:
        p = bp[t, u]
        if p == 1:
            u -= 1
            frames[u], logp[u] = t, float(lat[t, u, 1])
            acc = np.float32(acc + lat[t, u, 1])
        else:
            path[t] = acc
            if p == 2:
                break
            t -= 1
            acc = np.float32(lat[t, u, 0])
    return SpanPath(score, frames, logp, [float(x) for x in path])


def rnnt_span_forward(lat: np.ndarray) -> float:
    """log-sum-exp over every (start, end) pair and every monotone path between them of a [W, U + 1, 2] lattice, float64."""
    return _sweep(lat, False)[1]


def span_confidence(path_logp: Sequence[float], start: int, end: int, L: int = CONFIDENCE_FRAMES) -> float:
    """Confidence of a placed caption from the per-frame path log-probabilities of its span [start, end] (inclusive): the mean
    over the span when it has n <= L frames, else the minimum over the n - L + 1 windows of L consecutive frames of their mean.
    The analogue of CTC segmentation's ``score_min_mean_over_L``; it is not numerically comparable with ESPnet's score, which
    comes from another model with another output distribution."""
    x = np.asarray(path_logp[start:end + 1], np.float64)
    n = len(x)
    assert n >= 1
    if n <= L:
        return float(x.mean())
    return float(min(x[i:i + L].mean() for i in range(n - L + 1)))
