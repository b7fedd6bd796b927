"""bench.py --dump-outputs: the files written for a search result (host logic only; no GPU)."""
import os

import numpy as np

import bench
import meilisearch_b200 as mb


def _result(n, seed=0):
    r = mb.SearchResult(n, 20)
    rng = np.random.default_rng(seed)
    r.documents_ids[:] = rng.integers(0, 2**32 - 1, r.documents_ids.shape, dtype=np.uint32)
    r.n_candidates[:] = rng.integers(0, 2**40, n, dtype=np.uint64)
    r.score_rank[:] = rng.integers(0, 2**32 - 1, r.score_rank.shape, dtype=np.uint32)
    r.score_sim[:] = rng.random(r.score_sim.shape, dtype=np.float32)
    return r


def test_dump_holds_every_result_array_exactly(tmp_path):
    r = _result(64)
    bench.dump_outputs(r, str(tmp_path))
    assert sorted(os.listdir(tmp_path)) == sorted(name + ".npy" for name in bench.RESULT_ARRAYS)
    for name in bench.RESULT_ARRAYS:
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype in (np.float32, np.float64)
        assert np.array_equal(a, getattr(r, name)), name


def test_large_batch_dump_is_a_fixed_sample_below_64mb(tmp_path):
    r = _result(20000)
    bench.dump_outputs(r, str(tmp_path / "a"))
    bench.dump_outputs(r, str(tmp_path / "b"))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) < 64e6
    rows = np.load(tmp_path / "a" / "query_index.npy")
    assert 0 < len(rows) < 20000
    assert np.array_equal(rows, np.load(tmp_path / "b" / "query_index.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "documents_ids.npy"), r.documents_ids[rows.astype(np.int64)])
