"""The forced-alignment oracle (oracle/align_restated.py) against brute force, against torchaudio's RNN-T loss and against the
greedy oracle's own joint evaluations; the tokenizers' text_to_ids."""
import itertools

import numpy as np
import pytest
import torch

from oracle import align_restated as A
from oracle import nemo_restated as O


def _paths(T, U):
    """Every monotone path as the emitting frame of each token (non-decreasing, in [0, T))."""
    return itertools.combinations_with_replacement(range(T), U)


@pytest.mark.parametrize("T,U", [(1, 0), (1, 3), (3, 0), (2, 2), (4, 3), (5, 4), (5, 1)])
def test_viterbi_and_forward_equal_brute_force(T, U):
    rng = np.random.default_rng(100 * T + U)
    for _ in range(4):
        lat = (-rng.exponential(1.0, (T, U + 1, 2))).astype(np.float32)
        scores = {fr: A.path_score(lat, fr) for fr in _paths(T, U)}
        best = max(scores.values())
        lse = np.logaddexp.reduce(np.array(list(scores.values())))
        path = A.rnnt_viterbi(lat)
        assert abs(path.score - best) <= 1e-12 * max(1.0, abs(best))
        assert abs(A.rnnt_forward(lat) - lse) <= 1e-12 * max(1.0, abs(lse))
        argmax = max(scores, key=scores.get)                      # unique with continuous random values
        assert tuple(path.frames) == argmax
        assert path.tok_logp == [float(lat[t, u, 1]) for u, t in enumerate(path.frames)]


def test_ties_put_every_token_on_its_earliest_frame():
    lat = np.full((5, 4, 2), -0.5, np.float32)
    path = A.rnnt_viterbi(lat)
    assert path.frames == [0, 0, 0]


def test_forward_matches_torchaudio_rnnt_loss(tiny_cfg, tiny_sd):
    torchaudio = pytest.importorskip("torchaudio")
    rng = np.random.default_rng(7)
    T, U = 9, 5
    enc = torch.from_numpy(rng.standard_normal((T, tiny_cfg.d_model)).astype(np.float32))
    targets = rng.integers(0, tiny_cfg.vocab_size, U).tolist()
    lat = A.lattice(enc, targets, tiny_sd, tiny_cfg)
    with torch.no_grad():
        ep = O.joint_enc_proj(enc, tiny_sd)
        g = A.pred_proj(targets, tiny_sd, tiny_cfg)
        logits = torch.nn.functional.linear(torch.relu(ep[:, None] + g[None]), tiny_sd["joint.joint_net.2.weight"],
                                            tiny_sd["joint.joint_net.2.bias"])
        loss = torchaudio.functional.rnnt_loss(torch.log_softmax(logits, -1)[None], torch.tensor([targets], dtype=torch.int32),
                                               torch.tensor([T], dtype=torch.int32), torch.tensor([U], dtype=torch.int32),
                                               blank=tiny_cfg.blank, reduction="none")
    ref = -float(loss[0])
    got = A.rnnt_forward(lat)
    print(f"forward {got:.6f}, torchaudio {ref:.6f}")
    assert abs(got - ref) <= 1e-5 * abs(ref)


def test_lattice_on_the_greedy_path_equals_the_greedy_joint(tiny_cfg, tiny_sd):
    """Along the greedy hypothesis the lattice holds the log_softmax of exactly the logits rnnt_greedy evaluated there."""
    from reazonspeech_b200.synth import synth_clip
    wave = torch.from_numpy(np.pad(synth_clip(300, 2.5), 8000))
    with torch.no_grad():
        enc = O.encoder(O.log_mel(wave, tiny_cfg), tiny_sd, tiny_cfg, emulate=True)
    greedy = O.rnnt_greedy(enc, tiny_sd, tiny_cfg, emulate=True)
    assert greedy.tokens and max(np.bincount(greedy.frames)) < tiny_cfg.max_symbols   # no symbol cap on this clip
    lat = A.lattice(enc, greedy.tokens, tiny_sd, tiny_cfg, emulate=True)
    # replay the greedy loop's joint evaluations: (t, u) with u tokens emitted so far
    ep = O.joint_enc_proj(O._q(enc, True), tiny_sd)
    g = A.pred_proj(greedy.tokens, tiny_sd, tiny_cfg)
    W, b = tiny_sd["joint.joint_net.2.weight"], tiny_sd["joint.joint_net.2.bias"]
    u, checked = 0, 0
    for t in range(enc.shape[0]):
        while True:
            lp = torch.log_softmax(torch.nn.functional.linear(torch.relu(ep[t] + g[u]), W, b), -1)
            assert abs(float(lat[t, u, 0]) - float(lp[tiny_cfg.blank])) <= 1e-5
            if u < len(greedy.tokens) and greedy.frames[u] == t:
                assert abs(float(lat[t, u, 1]) - float(lp[greedy.tokens[u]])) <= 1e-5
                u += 1
                checked += 1
            else:
                break
    assert checked == len(greedy.tokens)
    path = A.rnnt_viterbi(lat)
    assert path.score >= A.path_score(lat, greedy.frames)


def test_piece_table_text_to_ids_round_trip():
    from reazonspeech_b200.tokenizer import PieceTableTokenizer, synthetic_pieces
    tok = PieceTableTokenizer(synthetic_pieces(3000))
    rng = np.random.default_rng(0)
    chars = [p for p in tok.pieces[2:]] + [" "]
    for n in (1, 5, 40):
        s = "".join(rng.choice(chars, n))
        s = "あ" + s.strip() + "。"
        ids = tok.text_to_ids(s)
        assert len(ids) == len(s) and tok.ids_to_text(ids) == s
    assert tok.text_to_ids("a b") == [0, 1, 0]                     # unknown -> 0, space -> the word-boundary piece
