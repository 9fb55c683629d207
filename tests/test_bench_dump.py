"""bench.py --dump-outputs: what the timed path returned, written as float32 .npy files (no GPU involved)."""
import sys

import numpy as np
import pytest
import torch

import bench


def _outputs(B, U, seed=0):
    g = torch.Generator().manual_seed(seed)
    tokens = torch.randint(0, 3000, (B, U), generator=g, dtype=torch.int32)
    frames = torch.randint(0, 392, (B, U), generator=g, dtype=torch.int32)
    n_tok = torch.randint(0, U + 5, (B,), generator=g, dtype=torch.int32)        # may exceed U: the true emission count
    n_tok[0] = 0
    return tokens, frames, n_tok


def test_dump_writes_float32_with_unspecified_entries_masked(tmp_path):
    tokens, frames, n_tok = _outputs(6, 20)
    bench.dump_outputs(str(tmp_path), tokens, frames, n_tok)
    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert sorted(got) == ["clips", "frames", "n_tokens", "tokens"]
    assert all(a.dtype == np.float32 for a in got.values())
    assert np.array_equal(got["n_tokens"], n_tok.numpy()) and np.array_equal(got["clips"], np.arange(6))
    for b in range(6):
        n = min(int(n_tok[b]), 20)
        assert np.array_equal(got["tokens"][b, :n], tokens[b, :n].numpy()) and np.array_equal(got["frames"][b, :n], frames[b, :n].numpy())
        assert (got["tokens"][b, n:] == -1).all() and (got["frames"][b, n:] == -1).all()


def test_dump_of_a_large_batch_is_a_fixed_sample_within_the_cap(tmp_path, monkeypatch):
    B, U = 50, 16
    monkeypatch.setattr(bench, "DUMP_BYTES", 7 * (2 * U + 2) * 4 + 3)
    tokens, frames, n_tok = _outputs(B, U)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), tokens, frames, n_tok)
    assert sum(np.load(p).nbytes for p in (tmp_path / "a").glob("*.npy")) <= bench.DUMP_BYTES
    clips = np.load(tmp_path / "a" / "clips.npy").astype(np.int64)
    assert len(clips) == 7 and np.array_equal(clips, np.sort(clips)) and len(set(clips)) == 7
    for name in ("clips", "tokens", "frames", "n_tokens"):
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "n_tokens.npy"), n_tok.numpy()[clips])


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bad_arguments_are_refused_before_any_work(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
