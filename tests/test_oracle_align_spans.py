"""The free-span alignment oracle (oracle/align_spans_restated.py) against brute force over every (start, end) pair and every
monotone path, its identities with the whole-window oracle (oracle/align_restated.py), the three tie rules, the per-frame path
log-probabilities and the min-mean confidence."""
import itertools

import numpy as np
import pytest

from oracle import align_restated as A
from oracle import align_spans_restated as S


def _lattice(rng, W, U):
    """Log-softmax-like lattice: every entry <= 0, as align_lattice produces."""
    lat = np.log(rng.uniform(0.02, 1.0, (W, U + 1, 2))).astype(np.float32)
    lat[:, U, 1] = 0.0
    return lat


def _paths(n, U):
    return itertools.combinations_with_replacement(range(n), U)


def _brute(lat):
    W, U = lat.shape[0], lat.shape[1] - 1
    best, terms = -np.inf, []
    for ts in range(W):
        for te in range(ts, W):
            sub = lat[ts:te + 1]
            for fr in _paths(te - ts + 1, U):
                s = A.path_score(sub, fr)
                best = max(best, s)
                terms.append(s)
    return best, float(np.logaddexp.reduce(np.array(terms)))


@pytest.mark.parametrize("seed", range(12))
def test_span_scores_equal_brute_force(seed):
    rng = np.random.default_rng(seed)
    W, U = int(rng.integers(1, 6)), int(rng.integers(1, 4))
    lat = _lattice(rng, W, U)
    vit, fwd = _brute(lat)
    path = S.rnnt_span_viterbi(lat)
    assert abs(path.score - vit) <= 1e-12 * max(1.0, abs(vit))
    assert abs(S.rnnt_span_forward(lat) - fwd) <= 1e-12 * max(1.0, abs(fwd))
    assert path.frames == sorted(path.frames) and all(0 <= f < W for f in path.frames)
    assert A.path_score(lat[path.frames[0]:path.frames[-1] + 1], [f - path.frames[0] for f in path.frames]) == path.score


@pytest.mark.parametrize("seed", range(8))
def test_identities_over_sub_lattices(seed):
    rng = np.random.default_rng(100 + seed)
    W, U = int(rng.integers(1, 7)), int(rng.integers(1, 4))
    lat = _lattice(rng, W, U)
    subs = [(ts, te) for ts in range(W) for te in range(ts, W)]
    vit = max(A.rnnt_viterbi(lat[ts:te + 1]).score for ts, te in subs)
    fwd = float(np.logaddexp.reduce(np.array([A.rnnt_forward(lat[ts:te + 1]) for ts, te in subs])))
    assert abs(S.rnnt_span_viterbi(lat).score - vit) <= 1e-12 * max(1.0, abs(vit))
    assert abs(S.rnnt_span_forward(lat) - fwd) <= 1e-12 * max(1.0, abs(fwd))


def test_tie_at_u0_goes_to_the_fresh_start():
    lat = np.full((4, 2, 2), -1.0, np.float32)
    lat[:, 0, 0] = 0.0                                   # alpha(t-1, 0) + lb = 0: an exact tie with the fresh start
    bp, _, _ = S._sweep(lat, True)
    assert (bp[:, 0] == 2).all()


def test_tie_at_the_end_goes_to_the_earliest_frame():
    lat = np.zeros((4, 2, 2), np.float32)
    lat[:, 0, 1] = -1.0                                  # emitting the token costs the same at every frame
    lat[:, 1, 0] = -0.5
    path = S.rnnt_span_viterbi(lat)
    assert path.frames == [0] and path.score == -1.5
    assert path.path_logp == [-1.5, 0.0, 0.0, 0.0]


def test_tie_inside_goes_to_the_blank_edge():
    lat = np.full((2, 3, 2), -10.0, np.float32)
    lat[0, 0, 1], lat[0, 1, 0], lat[1, 0, 1] = -1.0, -1.0, -2.0     # y1 at 0 then a blank, or y1 at 1: both -2 at node (1, 1)
    lat[1, 1, 1], lat[1, 2, 0] = -1.0, -1.0
    path = S.rnnt_span_viterbi(lat)
    assert path.score == -4.0 and path.frames == [0, 1]
    assert path.path_logp == [-2.0, -2.0]


@pytest.mark.parametrize("seed", range(10))
def test_best_span_path_logp_and_cropping(seed):
    rng = np.random.default_rng(200 + seed)
    W, U = int(rng.integers(3, 40)), int(rng.integers(1, 6))
    lat = _lattice(rng, W, U)
    path = S.rnnt_span_viterbi(lat)
    f0, f1 = path.frames[0], path.frames[-1]
    # the best span is [frames[0], frames[U-1]]: path_logp is nonzero exactly there (random entries are < 0)
    assert [i for i, x in enumerate(path.path_logp) if x != 0.0] == list(range(f0, f1 + 1))
    assert abs(sum(path.path_logp) - path.score) <= 1e-5 * max(1.0, abs(path.score))
    assert path.tok_logp == [float(lat[f, u, 1]) for u, f in enumerate(path.frames)]
    # the whole-window Viterbi of the best span is the same path
    whole = A.rnnt_viterbi(lat[f0:f1 + 1])
    assert whole.score == path.score and whole.frames == [f - f0 for f in path.frames]
    # cropping the lattice to the best span reproduces the score and shifts the frames
    crop = S.rnnt_span_viterbi(lat[f0:f1 + 1])
    assert crop.score == path.score and crop.frames == [f - f0 for f in path.frames]
    assert crop.path_logp == path.path_logp[f0:f1 + 1]
    assert S.rnnt_span_forward(lat) >= path.score


def test_span_covers_a_whole_window_path():
    """The span score is at least the whole-window Viterbi score, which is one of the (start, end) candidates."""
    rng = np.random.default_rng(7)
    for _ in range(10):
        lat = _lattice(rng, int(rng.integers(1, 30)), int(rng.integers(1, 5)))
        assert S.rnnt_span_viterbi(lat).score >= A.rnnt_viterbi(lat).score
        assert S.rnnt_span_forward(lat) >= A.rnnt_forward(lat)


def test_confidence():
    L = S.CONFIDENCE_FRAMES
    assert L == 30
    x = [0.0] * 3 + [-1.0, -2.0, -3.0] + [0.0] * 2
    assert S.span_confidence(x, 3, 5) == pytest.approx(-2.0)                          # n < L: the mean
    y = list(np.linspace(-2.0, 0.0, L))
    assert S.span_confidence(y, 0, L - 1) == pytest.approx(float(np.mean(y)))        # n = L: the mean
    z = [-0.1] * 100
    z[60:70] = [-5.0] * 10                                                           # n > L: the worst window of L frames
    got = S.span_confidence(z, 0, 99)
    assert got == pytest.approx((20 * -0.1 + 10 * -5.0) / L)
    assert got < float(np.mean(z))
