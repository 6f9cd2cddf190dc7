"""bench.py --dump-outputs without a GPU: the per-window decode results are written field by field, slots the library leaves
unwritten are masked, and an output over the size limit becomes the same seeded sample of windows every time."""
import os

import numpy as np

import bench
from whisperkit_b200._lib import wk_decode_result


def fake_results(n):
    res = (wk_decode_result * n)()
    for i in range(n):
        res[i].n_tokens = i % 5
        res[i].avg_logprob = -0.25 * i
        res[i].steps = 3 + i
        for j in range(226):            # stale contents past n_tokens must not reach the dump
            res[i].tokens[j] = 1000 + j
            res[i].token_logprobs[j] = -7.0
    return res


def test_dump_writes_every_field_masked(tmp_path):
    bench.dump_outputs(str(tmp_path), fake_results(6), first_window=64)
    names = {f[:-4] for f in os.listdir(tmp_path)}
    assert names == {n for n, _ in wk_decode_result._fields_} | {"window_index"}
    tok, lp = np.load(tmp_path / "tokens.npy"), np.load(tmp_path / "token_logprobs.npy")
    assert tok.dtype == np.float64 and tok.shape == (6, 226) and lp.dtype == np.float32
    assert list(tok[3, :4]) == [1000, 1001, 1002, -1] and (tok[0] == -1).all()
    assert list(lp[3, :4]) == [-7.0, -7.0, -7.0, 0.0]
    np.testing.assert_array_equal(np.load(tmp_path / "window_index.npy"), np.arange(64, 70))
    np.testing.assert_array_equal(np.load(tmp_path / "steps.npy"), np.arange(3, 9))
    assert np.load(tmp_path / "avg_logprob.npy").dtype == np.float32


def test_dump_over_the_limit_is_a_fixed_sample(tmp_path):
    res = fake_results(40)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res, first_window=0, limit=10 * 3000, suffix="_rank1")
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    idx = np.load(tmp_path / "a" / "window_index_rank1.npy")
    assert 0 < len(idx) < 40 and total <= 10 * 3000 + 128 * len(os.listdir(tmp_path / "a"))   # + one .npy header per file
    assert (np.diff(idx) > 0).all()
    for f in os.listdir(tmp_path / "a"):
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
    steps = np.load(tmp_path / "a" / "steps_rank1.npy")
    np.testing.assert_array_equal(steps, 3 + idx)          # every field is sampled at the same windows
