"""CPU oracle of RNN-T forced alignment: the (frame x token) lattice of a GIVEN token sequence, its best path (Viterbi) and
its log-likelihood summed over all paths (the forward algorithm; minus NeMo's RNN-T loss).

THIS IS TEST INFRASTRUCTURE (see oracle/nemo_restated.py): only tests/, smoke() and the benchmark scripts may import it.

For one utterance with T encoder frames and targets y_1..y_U (ids in [0, V), the blank V excluded):

    f_t = joint.enc(enc_t)                      (enc rounded to bf16 first with ``emulate``, as the greedy and ALSD oracles do)
    g_u = joint.pred(h_u)                       h_0: predictor state after the SOS step (zero input, zero state);
                                                h_u: after consuming y_1..y_u, teacher-forced
    z(t, u) = W_out relu(f_t + g_u) + b_out     over the V + 1 classes
    lb(t, u) = log_softmax(z)[blank],  ly(t, u) = log_softmax(z)[y_{u+1}]  (u < U)

    alpha(0, 0) = 0
    alpha(t, u) = op(alpha(t-1, u) + lb(t-1, u), alpha(t, u-1) + ly(t, u-1))
    score = alpha(T-1, U) + lb(T-1, U)          op = max: Viterbi;  op = logaddexp: log-likelihood

alpha is accumulated in float64 from the fp32 log-probabilities.  Where the two Viterbi candidates of a node are exactly
equal the back-pointer takes the blank edge from (t-1, u): the backtrace, which runs from the last node, then keeps moving back
in time before it takes a token, so every token lands on its earliest frame (an all-equal lattice puts them all on frame 0).
Token u is emitted at frame t where the best path takes the edge (t, u) -> (t, u+1).  There is no max_symbols bound (as in NeMo's RNN-T loss); U = 0 (all blanks) and U > T are valid.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence

import numpy as np
import torch
import torch.nn.functional as F

from reazonspeech_b200.config import ModelConfig
from .nemo_restated import StateDict, _q, joint_enc_proj, lstm_step


def pred_proj(targets: Sequence[int], sd: StateDict, cfg: ModelConfig) -> torch.Tensor:
    """g_u = joint.pred(h_u) for u = 0..U: float32 [U + 1, joint_hidden]."""
    emb = sd["decoder.prediction.embed.weight"]
    h = torch.zeros(cfg.pred_hidden); c = torch.zeros(cfg.pred_hidden)
    h, c = lstm_step(torch.zeros(cfg.pred_hidden), h, c, sd)                  # SOS step
    hs = [h]
    for y in targets:
        h, c = lstm_step(emb[int(y)], h, c, sd)
        hs.append(h)
    return F.linear(torch.stack(hs), sd["joint.pred.weight"], sd["joint.pred.bias"])


def lattice(enc: torch.Tensor, targets: Sequence[int], sd: StateDict, cfg: ModelConfig, emulate: bool = False,
            rows_per_chunk: int = 4096) -> np.ndarray:
    """enc float32 [T, d_model] -> float32 [T, U + 1, 2]: (lb, ly) of every node (ly at u = U is 0).  The joint is evaluated
    over chunks of frames so that the logits of at most ``rows_per_chunk`` nodes exist at a time."""
    targets = [int(y) for y in targets]
    assert all(0 <= y < cfg.vocab_size for y in targets)
    T, U = enc.shape[0], len(targets)
    with torch.no_grad():
        ep = joint_enc_proj(_q(enc, emulate), sd)
        g = pred_proj(targets, sd, cfg)
        W, b = sd["joint.joint_net.2.weight"], sd["joint.joint_net.2.bias"]
        out = np.zeros((T, U + 1, 2), np.float32)
        idx = torch.tensor(targets, dtype=torch.long)
        step = max(1, rows_per_chunk // (U + 1))
        for t0 in range(0, T, step):
            lp = torch.log_softmax(F.linear(torch.relu(ep[t0:t0 + step, None, :] + g[None]), W, b), dim=-1)   # [tc, U + 1, V + 1]
            out[t0:t0 + step, :, 0] = lp[..., cfg.blank].numpy()
            if U:
                out[t0:t0 + step, :U, 1] = lp[:, :U, :].gather(-1, idx.expand(lp.shape[0], U)[..., None])[..., 0].numpy()
    return out


@dataclass
class AlignPath:
    score: float                 # Viterbi log-probability of the best path
    frames: List[int]            # emitting frame of every token
    tok_logp: List[float]        # ly(frames[u], u)


def _sweep(lat: np.ndarray, viterbi: bool):
    T, W = lat.shape[0], lat.shape[1]
    lb = lat[..., 0].astype(np.float64)
    ly = lat[..., 1].astype(np.float64)
    a = np.full((T, W), -np.inf)
    bp = np.zeros((T, W), np.int8)
    a[0, 0] = 0.0
    for t in range(T):
        for u in range(W):
            if t == 0 and u == 0:
                continue
            vb = a[t - 1, u] + lb[t - 1, u] if t > 0 else -np.inf
            ve = a[t, u - 1] + ly[t, u - 1] if u > 0 else -np.inf
            if viterbi:
                bp[t, u] = ve > vb                                   # exact ties: the blank edge (earliest frame)
                a[t, u] = ve if bp[t, u] else vb
            else:
                a[t, u] = np.logaddexp(vb, ve)
    return a, bp, float(a[T - 1, W - 1] + lb[T - 1, W - 1])


def rnnt_viterbi(lat: np.ndarray) -> AlignPath:
    """Best path through a [T, U + 1, 2] lattice, float64; exact ties put a token on its earliest frame."""
    _, bp, score = _sweep(lat, True)
    T, U = lat.shape[0], lat.shape[1] - 1
    frames, logp = [0] * U, [0.0] * U
    t, u = T - 1, U
    while u > 0:
        if bp[t, u]:
            u -= 1
            frames[u], logp[u] = t, float(lat[t, u, 1])
        else:
            t -= 1
    return AlignPath(score, frames, logp)


def rnnt_forward(lat: np.ndarray) -> float:
    """log-sum-exp over every monotone path of a [T, U + 1, 2] lattice, float64 (= -RNN-T loss)."""
    return _sweep(lat, False)[2]


def path_score(lat: np.ndarray, frames: Sequence[int]) -> float:
    """Log-probability (float64) of the path that emits token u at frames[u] (non-decreasing) and blanks elsewhere."""
    T, U = lat.shape[0], lat.shape[1] - 1
    s, u = 0.0, 0
    for t in range(T):
        while u < U and frames[u] == t:
            s += float(lat[t, u, 1])
            u += 1
        s += float(lat[t, u, 0])
    assert u == U, "frames must be non-decreasing and inside [0, T)"
    return s
