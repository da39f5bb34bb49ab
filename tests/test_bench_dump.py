"""bench.py --dump-outputs on a stand-in for the library's Results (CPU only): the files are float32, depend only on the
arguments, hold exactly the sampled pairs' matches, and stay under the size cap even when every query row matches."""
import os

import numpy as np

import bench
from oracle import DMATCH_DTYPE


class _Results:
    def __init__(self, counts, seed):
        rng = np.random.default_rng(seed)
        self.n_pairs = len(counts)
        self.m = np.zeros(int(np.sum(counts)), DMATCH_DTYPE)
        self.m["queryIdx"] = rng.integers(0, 8000, len(self.m))
        self.m["trainIdx"] = rng.integers(0, 8000, len(self.m))
        self.m["distance"] = rng.random(len(self.m), dtype=np.float32)
        self.off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)

    def fetch(self):
        pass

    def all_matches(self):
        return self.m.copy(), self.off.copy()


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_is_float32_repeatable_and_exact(tmp_path):
    counts = np.random.default_rng(0).integers(0, 2500, 2368)
    pairs = np.random.default_rng(1).integers(0, 1000, (2368, 2)).astype(np.int32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), _Results(counts, 7), pairs, 8000)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == ["distance", "match_counts", "pairs", "query_idx", "sample", "train_idx"]
    for k in a:
        assert a[k].dtype == np.float32 and a[k].tobytes() == b[k].tobytes(), k
    assert (a["pairs"] == pairs).all() and (a["match_counts"] == counts).all()
    r = _Results(counts, 7)
    sample = a["sample"].astype(np.int64)
    assert len(sample) < len(pairs) and (np.diff(sample) > 0).all()
    ref = np.concatenate([r.m[r.off[k]:r.off[k + 1]] for k in sample])
    assert (a["query_idx"] == ref["queryIdx"]).all() and (a["train_idx"] == ref["trainIdx"]).all()
    assert (a["distance"] == ref["distance"]).all()


def test_dump_stays_under_the_cap_when_every_row_matches(tmp_path):
    for n_pairs, n_feat in ((2368, 8000), (9472, 4000)):
        d = tmp_path / f"{n_pairs}"
        pairs = np.zeros((n_pairs, 2), np.int32)
        bench.dump_outputs(str(d), _Results(np.full(n_pairs, n_feat), 3), pairs, n_feat)
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= bench.DUMP_BYTES


def test_dump_keeps_every_pair_when_they_fit(tmp_path):
    counts = np.array([3, 0, 5, 1])
    bench.dump_outputs(str(tmp_path), _Results(counts, 9), np.arange(8).reshape(4, 2), 64)
    a = _load(tmp_path)
    assert (a["sample"] == np.arange(4)).all() and len(a["query_idx"]) == counts.sum()
