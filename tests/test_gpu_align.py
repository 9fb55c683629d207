"""RNN-T forced alignment on the GPU (rs_rnnt_align, csrc/align.cu) against its CPU oracle (oracle/align_restated.py) on the
SAME encoder output: the lattice of log-probabilities, the Viterbi path and both scores; invariants, batch / chunk
invariance, argument errors; the Python API (align / align_batch)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import align_restated as A
from reazonspeech_b200.synth import synth_clip

CHUNK_ROWS = 128 * 1024                         # kAlignChunkRows (csrc/align.h)


@pytest.fixture(scope="module")
def align_engine(tiny_cfg, tiny_sd):
    from reazonspeech_b200.engine import Engine
    return Engine(tiny_cfg, tiny_sd, "cuda:0", alsd=True)


def _encode(eng, waves):
    L = max(len(w) for w in waves)
    x = torch.zeros(len(waves), L)
    for i, w in enumerate(waves):
        x[i, : len(w)] = torch.from_numpy(w)
    lens = torch.tensor([len(w) for w in waves], dtype=torch.int32)
    mel, mel_len = eng.log_mel(x.cuda(), lens.cuda())
    return eng.encode(mel, mel_len)


def _targets(tlists):
    U = max(1, max(len(t) for t in tlists))
    tg = torch.zeros(len(tlists), U, dtype=torch.int32)
    for i, t in enumerate(tlists):
        tg[i, : len(t)] = torch.tensor(t, dtype=torch.int32)
    return tg.cuda(), torch.tensor([len(t) for t in tlists], dtype=torch.int32).cuda()


def _align(eng, enc, enc_len, tlists, lattice=True):
    tg, tl = _targets(tlists)
    return [a.cpu() if a is not None else None for a in eng.align(enc, enc_len, tg, tl, lattice=lattice)]


@pytest.fixture(scope="module")
def cases(align_engine, tiny_cfg):
    """Five clips; targets of length 0, 1, random, the greedy transcript, and more than 2 T."""
    eng = align_engine
    waves = [np.pad(synth_clip(400 + i, s), 8000) for i, s in enumerate((2.0, 1.3, 2.7, 3.1, 1.0))]
    enc, enc_len = _encode(eng, waves)
    tk, fr, nt = [a.cpu() for a in eng.greedy(enc, enc_len)]
    T = enc_len.cpu().tolist()
    rng = np.random.default_rng(5)
    V = tiny_cfg.vocab_size
    tlists = [[], [int(rng.integers(V))], rng.integers(0, V, T[2] // 2).tolist(), tk[3, : int(nt[3])].tolist(),
              rng.integers(0, V, 2 * T[4] + 3).tolist()]
    assert len(tlists[3]) > 0
    res = _align(eng, enc, enc_len, tlists)
    greedy = [(tk[i, : int(nt[i])].tolist(), fr[i, : int(nt[i])].tolist()) for i in range(len(waves))]
    return dict(enc=enc, enc_len=enc_len, T=T, tlists=tlists, res=res, greedy=greedy)


def _oracle_lattice(case, i, sd, cfg):
    return A.lattice(case["enc"][i, : case["T"][i]].cpu(), case["tlists"][i], sd, cfg, emulate=True)


def test_lattice_matches_the_oracle(cases, tiny_cfg, tiny_sd):
    lat = cases["res"][4]
    worst = 0.0
    for i, tl in enumerate(cases["tlists"]):
        T, U = cases["T"][i], len(tl)
        ref = _oracle_lattice(cases, i, tiny_sd, tiny_cfg)
        got = lat[i, :T, : U + 1].numpy()
        d = max(float(np.abs(got[..., 0] - ref[..., 0]).max()), float(np.abs(got[:, :U, 1] - ref[:, :U, 1]).max()) if U else 0.0)
        print(f"utt{i}: T={T} U={U} max |lattice - oracle| = {d:.3g}")
        worst = max(worst, d)
    assert worst <= 1e-4


def test_dp_matches_the_oracle_on_the_engine_lattice(cases):
    frames, tok_logp, viterbi, loglik, lat = cases["res"]
    for i, tl in enumerate(cases["tlists"]):
        T, U = cases["T"][i], len(tl)
        L = lat[i, :T, : U + 1].numpy()
        if U == 0:
            L = L.copy(); L[..., 1] = 0.0
        path = A.rnnt_viterbi(L)
        assert frames[i, :U].tolist() == path.frames
        assert tok_logp[i, :U].tolist() == path.tok_logp
        assert abs(float(viterbi[i]) - path.score) <= 1e-9 * max(1.0, abs(path.score))
        ref = A.rnnt_forward(L)
        assert abs(float(loglik[i]) - ref) <= 1e-9 * max(1.0, abs(ref))


def test_end_to_end_matches_the_oracle(cases, tiny_cfg, tiny_sd):
    frames, _, viterbi, loglik, _ = cases["res"]
    differ = 0
    for i, tl in enumerate(cases["tlists"]):
        U = len(tl)
        ref_lat = _oracle_lattice(cases, i, tiny_sd, tiny_cfg)
        path, fwd = A.rnnt_viterbi(ref_lat), A.rnnt_forward(ref_lat)
        got = frames[i, :U].tolist()
        print(f"utt{i}: viterbi {float(viterbi[i]):.5f} (oracle {path.score:.5f}), loglik {float(loglik[i]):.5f} (oracle {fwd:.5f})")
        if got != path.frames:                     # admissible only as a near-tie of the two paths under the oracle
            differ += 1
            assert abs(A.path_score(ref_lat, got) - path.score) < 1e-3
        assert abs(float(viterbi[i]) - path.score) <= 1e-3 * max(1.0, abs(path.score))
        assert abs(float(loglik[i]) - fwd) <= 1e-3 * max(1.0, abs(fwd))
    assert differ <= 1


def test_invariants(cases):
    frames, tok_logp, viterbi, loglik, lat = cases["res"]
    for i, tl in enumerate(cases["tlists"]):
        T, U = cases["T"][i], len(tl)
        f = frames[i, :U].tolist()
        assert float(viterbi[i]) <= float(loglik[i]) and np.isfinite(float(loglik[i]))
        assert all(0 <= x < T for x in f) and all(a <= b for a, b in zip(f, f[1:]))
        L = lat[i, :T, : U + 1].numpy()
        assert abs(A.path_score(L, f) - float(viterbi[i])) <= 1e-9 * max(1.0, abs(float(viterbi[i])))
        assert frames[i, U:].eq(-1).all()
    # the greedy kernel's own decision path, aligned to its tokens, cannot beat the best path
    g_tok, g_frm = cases["greedy"][3]
    L = lat[3, : cases["T"][3], : len(g_tok) + 1].numpy()
    assert A.path_score(L, g_frm) <= float(viterbi[3]) + 1e-9


def test_batch_and_chunk_invariance(align_engine, tiny_cfg):
    """An utterance aligned alone equals the same utterance at position 3 of a batch of five, bit for bit, while the batch's
    lattice crosses chunk boundaries inside that utterance."""
    eng = align_engine
    waves = [np.pad(synth_clip(420 + i, s), 8000) for i, s in enumerate((5.0, 4.6, 5.3, 5.1, 4.8))]
    enc, enc_len = _encode(eng, waves)
    T = enc_len.cpu().tolist()
    rng = np.random.default_rng(9)
    tlists = [rng.integers(0, tiny_cfg.vocab_size, 1000).tolist() for _ in waves]
    offs = np.cumsum([0] + [T[i] * (len(tlists[i]) + 1) for i in range(5)])
    assert offs[3] // CHUNK_ROWS != (offs[4] - 1) // CHUNK_ROWS, offs          # utterance 3 straddles a chunk boundary
    batch = _align(eng, enc, enc_len, tlists)
    alone = _align(eng, enc[3:4].contiguous(), enc_len[3:4].contiguous(), [tlists[3]])
    for a, b in zip(alone[:4], batch[:4]):
        assert torch.equal(a[0], b[3])
    assert torch.equal(alone[4][0, : T[3]], batch[4][3, : T[3]])                # the lattice's valid nodes (the rest is unspecified)


def _raw_align(eng, enc, enc_len, targets, tgt_len, U_max):
    B, T = enc.shape[0], enc.shape[1]
    out = [torch.zeros(B, U_max, dtype=torch.int32, device="cuda"), torch.zeros(B, U_max, device="cuda"),
           torch.zeros(B, dtype=torch.float64, device="cuda"), torch.zeros(B, dtype=torch.float64, device="cuda")]
    rc = eng.lib.rs_rnnt_align(eng.h, enc.data_ptr(), enc_len.data_ptr(), B, T, targets.data_ptr(), tgt_len.data_ptr(), U_max,
                               *[o.data_ptr() for o in out], None, eng._stream())
    return rc, eng.lib.rs_last_error(eng.h).decode()


def test_invalid_arguments_are_reported(align_engine, tiny_engine, tiny_cfg):
    eng = align_engine
    enc, enc_len = _encode(eng, [np.pad(synth_clip(430, 1.0), 8000)] * 2)
    T = enc.shape[1]
    ok_t = torch.tensor([[1, 2, 3], [4, 5, 6]], dtype=torch.int32, device="cuda")
    ok_l = torch.tensor([3, 2], dtype=torch.int32, device="cuda")
    assert _raw_align(eng, enc, enc_len, ok_t, ok_l, 3)[0] == 0
    cases = [
        (enc_len, ok_t, torch.tensor([4, 2], dtype=torch.int32, device="cuda"), "tgt_len"),
        (enc_len, ok_t, torch.tensor([-1, 2], dtype=torch.int32, device="cuda"), "tgt_len"),
        (torch.tensor([0, 5], dtype=torch.int32, device="cuda"), ok_t, ok_l, "enc_len"),
        (torch.tensor([5, T + 1], dtype=torch.int32, device="cuda"), ok_t, ok_l, "enc_len"),
        (enc_len, torch.tensor([[1, tiny_cfg.vocab_size, 3], [4, 5, 6]], dtype=torch.int32, device="cuda"), ok_l, "target"),
        (enc_len, torch.tensor([[1, 2, 3], [-7, 5, 6]], dtype=torch.int32, device="cuda"), ok_l, "target"),
    ]
    for el, tg, tl, needle in cases:
        rc, msg = _raw_align(eng, enc, el, tg, tl, 3)
        print(rc, msg)
        assert rc == -1 and needle in msg                        # RS_ERR_INVALID_ARG
    # a target past tgt_len is padding and not checked
    assert _raw_align(eng, enc, enc_len, torch.tensor([[1, 2, 3], [4, 5, 999]], dtype=torch.int32, device="cuda"), ok_l, 3)[0] == 0
    rc, msg = _raw_align(tiny_engine, enc, enc_len, ok_t, ok_l, 3)
    assert rc == -5 and "alsd" in msg                            # RS_ERR_UNSUPPORTED
    torch.cuda.synchronize()                                     # the device is healthy after all of these


# ---------------------------------------------------------------------------------------------- production configuration
@pytest.fixture(scope="module")
def prod():
    from reazonspeech_b200.config import ModelConfig
    from reazonspeech_b200.engine import Engine
    from reazonspeech_b200.weights import random_state_dict
    cfg = ModelConfig()
    sd = random_state_dict(cfg, seed=0)
    return cfg, sd, Engine(cfg, sd, "cuda:0", alsd=True)


def test_production_config_matches_the_oracle(prod):
    cfg, sd, eng = prod
    waves = [np.pad(synth_clip(i, 30.0), 8000) for i in range(2)]            # the first two of bench.py's 30 s clips
    enc, enc_len = _encode(eng, waves)
    tk, _, nt = [a.cpu() for a in eng.greedy(enc, enc_len)]
    tlists = [tk[i, : int(nt[i])].tolist() for i in range(2)]
    frames, _, viterbi, loglik, lat = _align(eng, enc, enc_len, tlists)
    for i in range(2):
        T, U = int(enc_len[i]), len(tlists[i])
        ref = A.lattice(enc[i, :T].cpu(), tlists[i], sd, cfg, emulate=True)
        got = lat[i, :T, : U + 1].numpy()
        d = max(float(np.abs(got[..., 0] - ref[..., 0]).max()), float(np.abs(got[:, :U, 1] - ref[:, :U, 1]).max()))
        path = A.rnnt_viterbi(ref)
        print(f"production utt{i}: T={T} U={U} max |lattice - oracle| = {d:.3g}, viterbi {float(viterbi[i]):.4f} (oracle {path.score:.4f})")
        assert d <= 1e-4
        assert frames[i, :U].tolist() == path.frames
        assert float(viterbi[i]) <= float(loglik[i])


def test_production_config_long_clip(prod):
    cfg, sd, eng = prod
    enc, enc_len = _encode(eng, [np.pad(synth_clip(40, 150.0), 8000)])
    tk, _, nt = [a.cpu() for a in eng.greedy(enc, enc_len)]
    tl = tk[0, : int(nt[0])].tolist()
    T, U = int(enc_len[0]), len(tl)
    assert T * (U + 1) > 2 * CHUNK_ROWS, (T, U)                              # the lattice spans several chunks
    frames, tok_logp, viterbi, loglik, lat = _align(eng, enc, enc_len, [tl])
    f = frames[0, :U].tolist()
    print(f"150 s clip: T={T} U={U} nodes={T * (U + 1)} viterbi {float(viterbi[0]):.3f} loglik {float(loglik[0]):.3f}")
    assert all(0 <= x < T for x in f) and all(a <= b for a, b in zip(f, f[1:]))
    assert float(viterbi[0]) <= float(loglik[0]) and np.isfinite(float(loglik[0]))
    L = lat[0, :T, : U + 1].numpy()
    assert abs(A.path_score(L, f) - float(viterbi[0])) <= 1e-9 * abs(float(viterbi[0]))


# ---------------------------------------------------------------------------------------------- Python API
@pytest.fixture(scope="module")
def api_model(tiny_cfg):
    from reazonspeech_b200.nemo.asr import load_model
    return load_model(synthetic=True, config=tiny_cfg, aligner=True)


def test_align_api(api_model):
    from reazonspeech_b200.nemo.asr import align, align_batch, transcribe
    from reazonspeech_b200.nemo.asr.audio import audio_from_numpy
    from reazonspeech_b200.nemo.asr.decode import PAD_SECONDS
    audios = [audio_from_numpy(synth_clip(440 + i, s), 16000) for i, s in enumerate((2.5, 1.6, 3.2))]
    texts = [transcribe(api_model, a).text for a in audios]
    assert all(texts)
    single = [align(api_model, a, t) for a, t in zip(audios, texts)]
    for a, t, r in zip(audios, texts, single):
        secs = [w.seconds for w in r.subwords]
        assert r.text == t
        # times are on transcribe()'s axis: the clip plus its trailing 0.5 s of padding, where a forced token may land
        assert all(x <= y for x, y in zip(secs, secs[1:])) and all(0.0 <= x < a.seconds + PAD_SECONDS for x in secs)
        assert np.isfinite(r.log_likelihood) and r.viterbi_log_prob <= r.log_likelihood
        assert len(r.token_log_probs) == len(api_model.tokenizer.text_to_ids(t))
    batch = align_batch(api_model, audios, texts)
    for s, b in zip(single, batch):
        assert b.text == s.text and b.subwords == s.subwords and b.segments == s.segments
        assert b.token_log_probs == pytest.approx(s.token_log_probs, abs=1e-5)
        assert b.log_likelihood == pytest.approx(s.log_likelihood, rel=1e-6)
    ids = api_model.tokenizer.text_to_ids(texts[0])
    assert align(api_model, audios[0], ids).subwords == single[0].subwords          # token ids are accepted as well


def test_align_without_the_aligner_weights_raises(tiny_cfg):
    from reazonspeech_b200.nemo.asr import align, load_model
    from reazonspeech_b200.nemo.asr.audio import audio_from_numpy
    model = load_model(synthetic=True, config=tiny_cfg)
    with pytest.raises(RuntimeError, match="aligner=True"):
        align(model, audio_from_numpy(synth_clip(450, 1.0), 16000), "あ")
