"""SURF tc16 fast mode (sweep_win.cu, 9 MMA slots per tile) against the oracle and against exact mode ($ESFM_TC16_EXACT=1, 13 slots).

The fast sweep ranks with the query rounded to one fp16 term; rows its error bound cannot settle are re-swept exactly (the fallback
sweep).  These tests build rows the fast values cannot settle -- near-ties at the ratio boundary, train rows a hair apart, duplicates,
non-unit norms -- check the answers against oracle.match, that the fallback really ran, and that both modes return the same matches.
Magnitudes outside tc16's input range (and the fallback at the smallest magnitude it keeps) are in test_gpu_input_range.py.
"""
import os

import numpy as np
import pytest

import oracle
from easysfm_b200 import synth
from util import justify_l2

pytestmark = pytest.mark.gpu


def _context(exact):
    import easysfm_b200 as esfm
    old = os.environ.get("ESFM_TC16_EXACT")
    os.environ["ESFM_TC16_EXACT"] = "1" if exact else "0"
    try:
        c = esfm.Context(0)                 # the knob is read when the context is created
    finally:
        if old is None:
            del os.environ["ESFM_TC16_EXACT"]
        else:
            os.environ["ESFM_TC16_EXACT"] = old
    c.set_l2_engine("tc16")
    return c


@pytest.fixture(scope="module")
def fast():
    c = _context(False)
    yield c
    c.close()


@pytest.fixture(scope="module")
def exact():
    c = _context(True)
    yield c
    c.close()


def _unit(x):
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def near_ties(seed):
    """Query rows whose two nearest train rows are (a) at d1 / d2 = 0.8 within 1e-4, (b) a hair apart, so that the fast sweep's
    error (the dropped b_q.t term) outweighs their difference, (c) exact duplicates."""
    rng = np.random.default_rng(seed)
    T = _unit(rng.standard_normal((900, 64)))
    Q = _unit(rng.standard_normal((700, 64)))
    for k in range(150):                                       # (a)
        t1, t2 = T[2 * k], T[2 * k + 1]
        s = 0.8 * (1 + rng.uniform(-1e-4, 1e-4))
        w = s / (1 + s)
        Q[k] = (1 - w) * t1 + w * t2
    for k in range(150):                                       # (b): t' = t + 2^-12 * noise, q next to both
        t = 300 + k
        T[450 + k] = _unit((T[t] + 2.0 ** -12 * rng.standard_normal(64))[None])[0]
        Q[150 + k] = _unit((T[t] + 0.02 * rng.standard_normal(64))[None])[0]
    Q[300:340] = T[600:640]                                    # (c)
    T[640:680] = T[600:640]
    return Q, T


def test_near_ties_fall_back_and_match_the_oracle(fast):
    Q, T = near_ties(21)
    before = fast.stats()["fallback_rows"]
    for ratio in (0.8, float("inf")):
        for cc in (False, True):
            got = fast.match_descriptors(Q, T, ratio, cc)
            justify_l2(Q, T, ratio, cc, got, oracle.match(Q, T, ratio, cc))
    assert fast.stats()["fallback_rows"] - before > 0


@pytest.mark.parametrize("scale_q,scale_t", [(1.0, 1.0), (1 / 16, 1.0), (16.0, 1 / 16), (4.0, 4.0)])
def test_fast_equals_exact(fast, exact, scale_q, scale_t):
    """Contention data (graded queries around shared train rows, duplicates, rows between two train rows) at several scales."""
    rng = np.random.default_rng(17)
    T = _unit(rng.standard_normal((1100, 64)))
    Q = _unit(rng.standard_normal((1500, 64)))

    def jitter(row, s):
        return _unit((row + s * rng.standard_normal(64))[None])[0]
    for k in range(300):
        Q[int(rng.integers(0, 1500))] = jitter(T[int(rng.integers(0, 200))], float(rng.uniform(0.0, 0.12)))
    for k in range(40):
        Q[int(rng.integers(0, 1500))] = T[int(rng.integers(200, 220))]
    for k in range(60):
        a, b = int(rng.integers(0, 200)), int(rng.integers(220, 260))
        T[b] = jitter(T[a], 0.01)
        Q[int(rng.integers(0, 1500))] = jitter(T[a], 0.005)
    Q = (Q * np.float32(scale_q)).astype(np.float32)
    T = (T * np.float32(scale_t)).astype(np.float32)
    for ratio in (0.8, 1.0, float("inf")):
        for cc in (False, True):
            a = fast.match_descriptors(Q, T, ratio, cc)
            b = exact.match_descriptors(Q, T, ratio, cc)
            assert len(a) == len(b)
            for f in ("queryIdx", "trainIdx", "distance"):
                np.testing.assert_array_equal(a[f], b[f])
            justify_l2(Q, T, ratio, cc, a, oracle.match(Q, T, ratio, cc))


def test_bench_shape_needs_no_fallback(fast, exact):
    """Frames of bench.py's SURF generator (8000 unit rows, sigma 0.02): no row reaches the fallback sweep, and every pair's
    matches equal exact mode's."""
    import torch
    data = synth.surf_like_torch(4, 8000, 4, torch.device("cuda:0")).cpu().numpy()
    frames = [np.ascontiguousarray(data[i]) for i in range(4)]
    out = []
    for c in (fast, exact):
        before = c.stats()["fallback_rows"]
        bank = c.bank_from_frames(frames)
        res = bank.match_all_pairs(0.8, True)
        out.append([res.pair_at(k) for k in range(res.n_pairs)])
        bank.close()
        if c is fast:
            assert c.stats()["fallback_rows"] == before
    assert sum(len(m) for _, _, m in out[0]) > 10000
    for (i, j, a), (i2, j2, b) in zip(*out):
        assert (i, j) == (i2, j2) and len(a) == len(b)
        for f in ("queryIdx", "trainIdx", "distance"):
            np.testing.assert_array_equal(a[f], b[f])
