"""Free-span RNN-T alignment on the GPU (rs_rnnt_align_spans, csrc/align.cu) against its CPU oracle
(oracle/align_spans_restated.py) on the SAME encoder output: several captions per encoder row, the lattice, the DP, end to
end; invariants against rs_rnnt_align; bit invariance across calls and lattice chunks; argument errors; the production
configuration on a 600 s recording; the Python API (align_captions / align_captions_batch)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import align_restated as A
from oracle import align_spans_restated as S
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


def _spans(eng, enc, enc_len, items, lattice=True):
    """items: [(src, lo, hi, tokens)] -> the outputs of Engine.align_spans on the host."""
    U = max(len(it[3]) for it in items)
    tg = torch.zeros(len(items), U, dtype=torch.int32)
    for k, it in enumerate(items):
        tg[k, : len(it[3])] = torch.tensor(it[3], dtype=torch.int32)
    sp = torch.tensor([it[:3] for it in items], dtype=torch.int32)
    tl = torch.tensor([len(it[3]) for it in items], dtype=torch.int32)
    out = eng.align_spans(enc, enc_len, sp.cuda(), tg.cuda(), tl.cuda(), lattice=lattice)
    return [a.cpu() for a in out]


@pytest.fixture(scope="module")
def cases(align_engine, tiny_cfg):
    """Two encoder rows, seven captions (K != B): windows with lo = 0, hi = enc_len, W = 1, U > W, and the greedy transcript."""
    eng = align_engine
    waves = [np.pad(synth_clip(500 + i, s), 8000) for i, s in enumerate((2.6, 3.4))]
    enc, enc_len = _encode(eng, waves)
    T = enc_len.cpu().tolist()
    tk, fr, nt = [a.cpu() for a in eng.greedy(enc, enc_len)]
    rng = np.random.default_rng(11)
    V = tiny_cfg.vocab_size
    r = lambda n: rng.integers(0, V, n).tolist()
    g1 = tk[1, : int(nt[1])].tolist()
    assert len(g1) > 0
    items = [(0, 0, T[0], r(3)), (0, 5, 6, r(2)), (1, 0, 10, r(4)), (1, 7, T[1], g1), (0, 3, 20, r(25)), (1, 12, 30, r(1)),
             (0, T[0] - 1, T[0], r(1))]
    res = _spans(eng, enc, enc_len, items)
    return dict(enc=enc, enc_len=enc_len, T=T, items=items, res=res)


def _oracle_lattice(enc, item, sd, cfg):
    src, lo, hi, toks = item
    return A.lattice(enc[src, lo:hi].cpu(), toks, sd, cfg, emulate=True)


def test_lattice_matches_the_oracle(cases, tiny_cfg, tiny_sd):
    lat = cases["res"][5]
    worst = 0.0
    for k, it in enumerate(cases["items"]):
        W, U = it[2] - it[1], len(it[3])
        ref = _oracle_lattice(cases["enc"], it, tiny_sd, tiny_cfg)
        got = lat[k, :W, : U + 1].numpy()
        d = max(float(np.abs(got[..., 0] - ref[..., 0]).max()), float(np.abs(got[:, :U, 1] - ref[:, :U, 1]).max()))
        print(f"caption{k}: src={it[0]} [{it[1]}, {it[2]}) U={U} max |lattice - oracle| = {d:.3g}")
        worst = max(worst, d)
    assert worst <= 1e-4


def test_dp_matches_the_oracle_on_the_engine_lattice(cases):
    frames, tok_logp, path_logp, viterbi, loglik, lat = cases["res"]
    for k, (src, lo, hi, toks) in enumerate(cases["items"]):
        W, U = hi - lo, len(toks)
        L = lat[k, :W, : U + 1].numpy().copy()
        L[:, U, 1] = 0.0
        path = S.rnnt_span_viterbi(L)
        assert frames[k, :U].tolist() == [lo + f for f in path.frames]
        assert frames[k, U:].eq(-1).all()
        assert tok_logp[k, :U].tolist() == path.tok_logp
        assert path_logp[k, :W].tolist() == path.path_logp and path_logp[k, W:].eq(0).all()
        assert abs(float(viterbi[k]) - path.score) <= 1e-9 * max(1.0, abs(path.score))
        ref = S.rnnt_span_forward(L)
        assert abs(float(loglik[k]) - ref) <= 1e-9 * max(1.0, abs(ref))


def test_end_to_end_matches_the_oracle(cases, tiny_cfg, tiny_sd):
    frames, _, _, viterbi, loglik, _ = cases["res"]
    differ = 0
    for k, it in enumerate(cases["items"]):
        lo, U = it[1], len(it[3])
        ref = _oracle_lattice(cases["enc"], it, tiny_sd, tiny_cfg)
        path, fwd = S.rnnt_span_viterbi(ref), S.rnnt_span_forward(ref)
        got = [f - lo for f in frames[k, :U].tolist()]
        print(f"caption{k}: viterbi {float(viterbi[k]):.5f} (oracle {path.score:.5f}), loglik {float(loglik[k]):.5f} (oracle {fwd:.5f})")
        if got != path.frames:                     # admissible only as a near-tie of the two paths under the oracle
            differ += 1
            assert abs(A.path_score(ref[got[0]:got[-1] + 1], [f - got[0] for f in got]) - path.score) < 1e-3
        assert abs(float(viterbi[k]) - path.score) <= 1e-3 * max(1.0, abs(path.score))
        assert abs(float(loglik[k]) - fwd) <= 1e-3 * max(1.0, abs(fwd))
    assert differ <= 1


def test_invariants_against_whole_window_alignment(align_engine, cases):
    eng = align_engine
    frames, tok_logp, path_logp, viterbi, loglik, lat = cases["res"]
    enc = cases["enc"]
    for k, (src, lo, hi, toks) in enumerate(cases["items"]):
        W, U = hi - lo, len(toks)
        f = frames[k, :U].tolist()
        assert all(lo <= x < hi for x in f) and all(a <= b for a, b in zip(f, f[1:]))
        assert float(viterbi[k]) <= float(loglik[k]) and np.isfinite(float(loglik[k]))
        # the best span is [frames[0], frames[U-1]]: path_logp is nonzero only there and sums to the score
        nz = [t for t in range(W) if float(path_logp[k, t]) != 0.0]
        assert set(nz) <= set(range(f[0] - lo, f[-1] - lo + 1))
        assert abs(float(path_logp[k, :W].double().sum()) - float(viterbi[k])) <= 1e-4 * max(1.0, abs(float(viterbi[k])))
        # rs_rnnt_align over the same window is one (start, end) candidate of the free span
        w = enc[src:src + 1, lo:hi].contiguous()
        tg = torch.tensor([toks], dtype=torch.int32, device="cuda")
        _, _, v_whole, l_whole = [a.cpu() for a in eng.align(w, torch.tensor([W], dtype=torch.int32, device="cuda"), tg,
                                                             torch.tensor([U], dtype=torch.int32, device="cuda"))]
        assert float(viterbi[k]) >= float(v_whole[0]) - 1e-6 * abs(float(v_whole[0]))
        assert float(loglik[k]) >= float(l_whole[0]) - 1e-6 * abs(float(l_whole[0]))
    # re-aligning inside the best span reproduces the result
    cropped = [(src, frames[k, 0].item(), frames[k, len(toks) - 1].item() + 1, toks) for k, (src, _, _, toks) in enumerate(cases["items"])]
    again = _spans(eng, enc, cases["enc_len"], cropped, lattice=False)
    for k, (_, lo, hi, toks) in enumerate(cropped):
        U = len(toks)
        assert torch.equal(again[0][k, :U], frames[k, :U])
        assert abs(float(again[3][k]) - float(viterbi[k])) <= 1e-12 * max(1.0, abs(float(viterbi[k])))


def test_bit_invariance_alone_and_across_chunks(align_engine, tiny_cfg):
    """A caption aligned alone equals the same caption at position 3 of a K = 5 call, bit for bit, while that call's lattice
    crosses a chunk boundary inside it."""
    eng = align_engine
    waves = [np.pad(synth_clip(520 + i, s), 8000) for i, s in enumerate((5.2, 4.7))]
    enc, enc_len = _encode(eng, waves)
    T = enc_len.cpu().tolist()
    rng = np.random.default_rng(13)
    V = tiny_cfg.vocab_size
    items = [(0, 0, T[0], rng.integers(0, V, 1000).tolist()), (1, 2, T[1], rng.integers(0, V, 1000).tolist()),
             (0, 4, T[0] - 3, rng.integers(0, V, 1000).tolist()), (1, 1, T[1] - 1, rng.integers(0, V, 1000).tolist()),
             (0, 0, 30, rng.integers(0, V, 900).tolist())]
    offs = np.cumsum([0] + [(hi - lo) * (len(t) + 1) for _, lo, hi, t in items])
    assert offs[3] // CHUNK_ROWS != (offs[4] - 1) // CHUNK_ROWS, offs          # caption 3 straddles a chunk boundary
    batch = _spans(eng, enc, enc_len, items)
    alone = _spans(eng, enc, enc_len, [items[3]])
    W = items[3][2] - items[3][1]
    for i in (0, 1, 3, 4):                                    # frames, tok_logp, viterbi, loglik
        assert torch.equal(alone[i][0], batch[i][3])
    for i in (2, 5):                                          # path_logp and the lattice over the caption's window
        assert torch.equal(alone[i][0, :W], batch[i][3, :W])


def _raw(eng, enc, enc_len, spans, targets, tgt_len, U_max, F_max):
    K = spans.shape[0]
    out = [torch.zeros(K, U_max, dtype=torch.int32, device="cuda"), torch.zeros(K, U_max, device="cuda"),
           torch.zeros(K, max(F_max, 1), device="cuda"), torch.zeros(K, dtype=torch.float64, device="cuda"),
           torch.zeros(K, dtype=torch.float64, device="cuda")]
    rc = eng.lib.rs_rnnt_align_spans(eng.h, enc.data_ptr(), enc_len.data_ptr(), enc.shape[0], enc.shape[1], K, spans.data_ptr(),
                                     targets.data_ptr(), tgt_len.data_ptr(), U_max, out[0].data_ptr(), out[1].data_ptr(),
                                     out[2].data_ptr(), F_max, out[3].data_ptr(), out[4].data_ptr(), None, eng._stream())
    return rc, eng.lib.rs_last_error(eng.h).decode()


def test_invalid_arguments_are_reported(align_engine, tiny_engine, tiny_cfg):
    eng = align_engine
    enc, enc_len = _encode(eng, [np.pad(synth_clip(530, 1.0), 8000), np.pad(synth_clip(531, 1.4), 8000)])
    T = enc_len.cpu().tolist()
    I = lambda x: torch.tensor(x, dtype=torch.int32, device="cuda")
    ok_s, ok_t, ok_l = I([[0, 0, T[0]], [1, 2, 9], [0, 3, 4]]), I([[1, 2, 3], [4, 5, 6], [7, 8, 9]]), I([3, 2, 1])
    F = max(T[0], 7)
    assert _raw(eng, enc, enc_len, ok_s, ok_t, ok_l, 3, F)[0] == 0
    cases = [
        (I([[0, 0, T[0]], [2, 2, 9], [0, 3, 4]]), ok_t, ok_l, F, "src"),
        (I([[0, 0, T[0]], [-1, 2, 9], [0, 3, 4]]), ok_t, ok_l, F, "src"),
        (I([[0, -1, T[0]], [1, 2, 9], [0, 3, 4]]), ok_t, ok_l, F, "window"),
        (I([[0, 0, T[0] + 1], [1, 2, 9], [0, 3, 4]]), ok_t, ok_l, F + 1, "window"),
        (I([[0, 0, T[0]], [1, 9, 9], [0, 3, 4]]), ok_t, ok_l, F, "window"),
        (ok_s, ok_t, I([3, 0, 1]), F, "tgt_len"),
        (ok_s, ok_t, I([3, 4, 1]), F, "tgt_len"),
        (ok_s, ok_t, ok_l, T[0] - 1, "F_max"),
        (ok_s, I([[1, 2, 3], [4, tiny_cfg.vocab_size, 6], [7, 8, 9]]), ok_l, F, "target"),
        (ok_s, I([[1, 2, 3], [4, 5, 6], [-3, 8, 9]]), ok_l, F, "target"),
    ]
    for sp, tg, tl, f_max, needle in cases:
        rc, msg = _raw(eng, enc, enc_len, sp, tg, tl, 3, f_max)
        print(rc, msg)
        assert rc == -1 and needle in msg                        # RS_ERR_INVALID_ARG
    rc, msg = _raw(tiny_engine, enc, enc_len, ok_s, ok_t, ok_l, 3, F)
    assert rc == -5 and "alsd" in msg                            # RS_ERR_UNSUPPORTED
    torch.cuda.synchronize()                                     # the device is healthy after all of these
    assert _raw(eng, enc, enc_len, ok_s, ok_t, ok_l, 3, F)[0] == 0


# ---------------------------------------------------------------------------------------------- production configuration
@pytest.fixture(scope="module")
def prod():
    from reazonspeech_b200.config import ModelConfig
    from reazonspeech_b200.engine import Engine
    from reazonspeech_b200.weights import random_state_dict
    cfg = ModelConfig()
    sd = random_state_dict(cfg, seed=0)
    return cfg, sd, Engine(cfg, sd, "cuda:0", alsd=True)


def test_production_600s_recording(prod):
    """Captions of 24 tokens cut from the greedy transcript of a 600 s recording (decoded per 30 s piece: in one piece this
    untrained checkpoint emits only a few dozen tokens), each searched for in the 25 s before it, in the encoding of the whole
    recording."""
    cfg, sd, eng = prod
    x = synth_clip(0, 600.0)
    enc, enc_len = _encode(eng, [np.pad(x, 8000)])
    T = int(enc_len[0])
    pieces = [np.pad(x[i:i + 480000], 8000) for i in range(0, len(x), 480000)]
    tk, fr, nt = [a.cpu() for a in eng.greedy(*_encode(eng, pieces))]
    toks, frs = [], []
    for i in range(len(pieces)):
        toks += tk[i, : int(nt[i])].tolist()
        frs += [f + 375 * i for f in fr[i, : int(nt[i])].tolist()]        # 30 s = 375 frames
    items = []
    for i in range(0, len(toks) - 23, 24):
        hi = min(T, frs[i + 23] + 1)
        items.append((0, max(0, frs[i] - 312), hi, toks[i:i + 24]))
    assert len(items) >= 50, len(toks)
    frames, tok_logp, path_logp, viterbi, loglik, lat = _spans(eng, enc, enc_len, items)
    assert np.isfinite(viterbi.numpy()).all() and np.isfinite(loglik.numpy()).all()
    assert np.isfinite(path_logp.numpy()).all() and np.isfinite(tok_logp.numpy()).all()
    for k, (_, lo, hi, tl) in enumerate(items):
        W, U = hi - lo, len(tl)
        L = lat[k, :W, : U + 1].numpy().copy()
        L[:, U, 1] = 0.0
        path = S.rnnt_span_viterbi(L)
        assert frames[k, :U].tolist() == [lo + f for f in path.frames], k
        assert path_logp[k, :W].tolist() == path.path_logp, k
        assert abs(float(viterbi[k]) - path.score) <= 1e-9 * max(1.0, abs(path.score))
        ref = S.rnnt_span_forward(L)
        assert abs(float(loglik[k]) - ref) <= 1e-9 * max(1.0, abs(ref))
    for k in (0, len(items) // 2):
        _, lo, hi, tl = items[k]
        W, U = hi - lo, len(tl)
        ref = A.lattice(enc[0, lo:hi].cpu(), tl, sd, cfg, emulate=True)
        got = lat[k, :W, : U + 1].numpy()
        d = max(float(np.abs(got[..., 0] - ref[..., 0]).max()), float(np.abs(got[:, :U, 1] - ref[:, :U, 1]).max()))
        print(f"production caption{k}: W={W} U={U} max |lattice - oracle| = {d:.3g}")
        assert d <= 1e-4
    placed = sum(abs(int(frames[k, 0]) - frs[24 * k]) <= 2 for k in range(len(items)))
    print(f"600 s: T={T} captions={len(items)} placed within 2 frames of the greedy frame: {placed}")


# ---------------------------------------------------------------------------------------------- Python API
@pytest.fixture(scope="module")
def api_model(tiny_cfg):
    from reazonspeech_b200.nemo.asr import load_model
    return load_model(synthetic=True, config=tiny_cfg, aligner=True)


def _caption_set(model, audio):
    from reazonspeech_b200.nemo.asr import Caption, transcribe
    r = transcribe(model, audio)
    assert len(r.subwords) >= 4
    w = r.subwords
    h = len(w) // 2
    return [Caption(w[0].seconds + 1.0, w[h - 1].seconds + 1.5, "".join(x.token for x in w[:h])),
            Caption(w[h].seconds + 0.5, w[-1].seconds + 0.2, "".join(x.token for x in w[h:])),
            Caption(0.2, 0.4, ""),                                                       # tokenises to nothing
            Caption(audio.seconds + 30.0, audio.seconds + 31.0, w[0].token)]             # the window lies past the end


def test_align_captions_matches_the_engine(api_model):
    from reazonspeech_b200.nemo.asr import align_captions
    from reazonspeech_b200.nemo.asr.audio import audio_from_numpy, norm_audio, pad_audio
    from reazonspeech_b200.nemo.asr.decode import PAD_SECONDS
    from reazonspeech_b200.nemo.asr.transcribe import min_mean_confidence, window_frames
    audio = audio_from_numpy(synth_clip(540, 6.0), 16000)
    caps = _caption_set(api_model, audio)
    got = align_captions(api_model, audio, caps, before=3.0)
    assert got[2] is None and got[3] is None
    eng = api_model.engine
    wave = pad_audio(norm_audio(audio), PAD_SECONDS).waveform.astype(np.float32)
    enc, enc_len = _encode(eng, [wave])
    T = int(enc_len[0])
    for c, r in zip(caps[:2], got[:2]):
        lo, hi = window_frames(c.start_seconds - 3.0, c.end_seconds, T)
        toks = api_model.tokenizer.text_to_ids(c.text)
        frames, tok_logp, path_logp, viterbi, loglik = _spans(eng, enc, enc_len, [(0, lo, hi, toks)], lattice=False)
        f = frames[0, : len(toks)].tolist()
        assert r.text == c.text
        assert r.viterbi_log_prob == pytest.approx(float(viterbi[0]), rel=1e-6)
        assert r.log_likelihood == pytest.approx(float(loglik[0]), rel=1e-6)
        assert r.token_log_probs == pytest.approx(tok_logp[0, : len(toks)].tolist(), abs=1e-5)
        assert r.start_seconds == pytest.approx(max(0.08 * f[0] - 0.5, 0))
        assert r.end_seconds == pytest.approx(min(max(0.08 * f[-1] - 0.5, 0) + 0.08, audio.seconds))
        assert r.confidence == pytest.approx(min_mean_confidence(path_logp[0, f[0] - lo: f[-1] - lo + 1].tolist()))
        assert r.start_seconds <= r.end_seconds and r.viterbi_log_prob <= r.log_likelihood
        assert len(r.token_log_probs) == len(toks) and len(r.subwords) <= len(toks)


def test_align_captions_batch_lax_and_asr(api_model):
    from reazonspeech_b200.nemo.asr import align_captions, align_captions_batch
    from reazonspeech_b200.nemo.asr.audio import audio_from_numpy
    from reazonspeech_b200.nemo.asr.transcribe import add_space
    audios = [audio_from_numpy(synth_clip(550 + i, s), 16000) for i, s in enumerate((7.0, 4.5, 5.5))]
    caps = [_caption_set(api_model, a) for a in audios]
    api_model.max_batch = 2                                   # two length-sorted batches
    try:
        batch = align_captions_batch(api_model, audios, caps)
    finally:
        api_model.max_batch = 64
    for a, c, b in zip(audios, caps, batch):
        single = align_captions(api_model, a, c)
        assert [x is None for x in single] == [x is None for x in b]
        for s, x in zip(single, b):
            if s is not None:
                assert (s.start_seconds, s.end_seconds, s.subwords) == (x.start_seconds, x.end_seconds, x.subwords)
                assert x.viterbi_log_prob == pytest.approx(s.viterbi_log_prob, rel=1e-6)
    lax = align_captions(api_model, audios[0], caps[0], strategy="lax", with_asr=True)
    ref = [x for x in align_captions(api_model, audios[0], caps[0]) if x is not None]
    add_space(ref)
    assert [(x.start_seconds, x.end_seconds) for x in lax if x is not None] == [(x.start_seconds, x.end_seconds) for x in ref]
    for x in lax:
        if x is not None:
            assert isinstance(x.asr, str) and (x.cer is None or x.cer >= 0.0)


def test_align_captions_without_the_aligner_weights_raises(tiny_cfg):
    from reazonspeech_b200.nemo.asr import Caption, align_captions, load_model
    from reazonspeech_b200.nemo.asr.audio import audio_from_numpy
    model = load_model(synthetic=True, config=tiny_cfg)
    with pytest.raises(RuntimeError, match="aligner=True"):
        align_captions(model, audio_from_numpy(synth_clip(560, 2.0), 16000), [Caption(0.0, 1.0, "あ")])
