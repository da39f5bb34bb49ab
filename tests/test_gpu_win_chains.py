"""SURF tc16 chain keys (sweep_win.cu): the sweep keeps the two largest maxima of 8-column chains per row, and finalize learns the
best chain's own second by evaluating that chain exactly.

Every case places a row's nearest and second-nearest train rows in the same chain, across a chain boundary, or in frames that are a
single chain, and checks the answers against oracle.match -- in fast mode (9 MMA slots, fallback sweep) and with $ESFM_TC16_EXACT=1.
"""
import os

import numpy as np
import pytest

import oracle
from test_gpu_tc16_fast import near_ties
from util import justify_l2

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["fast", "exact"])
def mode_ctx(request):
    import easysfm_b200 as esfm
    old = os.environ.get("ESFM_TC16_EXACT")
    os.environ["ESFM_TC16_EXACT"] = "1" if request.param == "exact" else "0"
    try:
        c = esfm.Context(0)                 # the knob is read when the context is created
    finally:
        if old is None:
            del os.environ["ESFM_TC16_EXACT"]
        else:
            os.environ["ESFM_TC16_EXACT"] = old
    c.set_l2_engine("tc16")
    yield c
    c.close()


def _unit(x):
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def _between(t1, t2, s):
    """The point on segment t1 -> t2 at d(q, t1) / d(q, t2) = s."""
    w = s / (1 + s)
    return ((1 - w) * t1 + w * t2).astype(np.float32)


def _check(c, Q, T, ratios=(0.8, float("inf"))):
    """Against oracle.match: the same train row within 1e-5 relative, any other difference explained by a float64 near-tie."""
    for ratio in ratios:
        for cc in (False, True):
            justify_l2(Q, T, ratio, cc, c.match_descriptors(Q, T, ratio, cc), oracle.match(Q, T, ratio, cc))


# (nearest, second) column placements: inside one chain (also at its first / last column and in the frame's last, partial chain), and
# across the chain boundaries 7|8, 63|64 (the two 32-column loads of a unit), 127|128 (two tiles)
_IN_CHAIN = [(16, 17), (23, 22), (0, 7), (56, 63), (64, 71), (120, 127), (128, 135), (200, 203), (498, 497), (499, 496)]
_ACROSS = [(7, 8), (8, 7), (63, 64), (64, 63), (127, 128), (128, 127), (255, 256)]


@pytest.mark.parametrize("nt", [500, 37])
def test_in_chain_second_decides_the_ratio_test(mode_ctx, nt):
    """The second neighbour sits in the nearest one's chain at d1 / d2 = 0.9 (fails at 0.8) or 0.7 (passes), and every other column is
    far: the second chain alone would pass every row."""
    rng = np.random.default_rng(5 + nt)
    T = _unit(rng.standard_normal((nt, 64)))
    Q = _unit(rng.standard_normal((300, 64)))
    places = [(a % nt, b % nt) for a, b in _IN_CHAIN + _ACROSS]
    places = [(a, b) for a, b in places if a != b]
    if nt == 37:                                # the last chain is columns 32..36
        places += [(32, 36), (36, 33), (31, 32), (35, 34)]
    k = 0
    want_pass = []
    for a, b in places:
        for s in (0.9, 0.7, 0.85, 0.75):
            Q[k] = _between(T[a], T[b], s)
            want_pass.append((k, a, s < 0.8))
            k += 1
    got = mode_ctx.match_descriptors(Q, T, 0.8, False)
    kept = {int(m["queryIdx"]): int(m["trainIdx"]) for m in got}
    for q, a, ok in want_pass:
        assert (kept.get(q) == a) if ok else (q not in kept), (q, a, ok, kept.get(q))
    _check(mode_ctx, Q, T)


@pytest.mark.parametrize("nt", [2, 3, 7, 8, 9, 15, 16, 17])
def test_small_train_frames(mode_ctx, nt):
    """Train frames of one chain, a chain and a bit, two chains: rows near a train row must pass, rows between two must not."""
    rng = np.random.default_rng(100 + nt)
    T = _unit(rng.standard_normal((nt, 64)))
    Q = _unit(rng.standard_normal((200, 64)))
    for k in range(60):
        Q[k] = _unit((T[k % nt] + 0.05 * rng.standard_normal(64))[None])[0]
    for k in range(60, 100):
        a, b = int(rng.integers(0, nt)), int(rng.integers(0, nt))
        if a != b:
            Q[k] = _between(T[a], T[b], float(rng.uniform(0.6, 1.0)))
    got = mode_ctx.match_descriptors(Q, T, 0.8, False)
    assert len(got) >= 55, len(got)                 # the rows next to a train row pass (unless that row is itself near another)
    _check(mode_ctx, Q, T, ratios=(0.8, 1.0, float("inf")))


def test_exact_ties_pick_the_lowest_index(mode_ctx):
    """Duplicate train rows inside one chain and in different chains (also across units and tiles): equal distances, lowest index."""
    rng = np.random.default_rng(9)
    T = _unit(rng.standard_normal((400, 64)))
    dups = [(3, 5), (6, 9), (10, 11, 12), (20, 90), (40, 70, 140), (130, 135, 300), (255, 256), (391, 399)]
    for grp in dups:
        for j in grp[1:]:
            T[j] = T[grp[0]]
    Q = _unit(rng.standard_normal((200, 64)))
    k = 0
    for grp in dups:
        Q[k] = T[grp[0]]                                              # d1 = d2 = 0
        Q[k + 1] = _unit((T[grp[0]] + 0.03 * rng.standard_normal(64))[None])[0]
        Q[k + 2] = _between(T[grp[0]], T[(grp[0] + 1) % 400], 0.5)
        k += 3
    _check(mode_ctx, Q, T, ratios=(0.8, 1.0, float("inf")))
    got = mode_ctx.match_descriptors(Q, T, float("inf"), False)
    kept = {int(m["queryIdx"]): int(m["trainIdx"]) for m in got}
    for i, grp in enumerate(dups):
        assert kept[3 * i] == grp[0] and kept[3 * i + 1] == grp[0], (grp, kept.get(3 * i), kept.get(3 * i + 1))


def _rival_scene(rng, second_in_chain, rival_nearer):
    """Query row q sits 0.1 from train row t and survives the ratio test.  A rival query row r has its nearest train row t' and its
    second t, with d(r, t') / d(r, t) < 0.8, so r survives too and only histogram B speaks for it at t.  t sits in t''s chain
    (second_in_chain) or in another chain, and r is nearer to t than q (rival_nearer: q must lose the cross-check) or farther."""
    T = _unit(rng.standard_normal((300, 64)))
    Q = _unit(rng.standard_normal((200, 64)))
    u = T[40].astype(np.float64)
    basis = np.linalg.qr(np.stack([u, rng.standard_normal(64), rng.standard_normal(64)], 1))[0]
    e1, e2 = basis[:, 1], basis[:, 2]
    tp = 41 if second_in_chain else 52                      # t' next to t = 40: chain 5, or chain 6
    T[tp] = u + 0.12 * e1
    Q[7] = u - 0.1 * e2                                     # q: d(q, t) = 0.1, d(q, t') = 0.156
    Q[150] = u + (0.075 if rival_nearer else 0.16) * e1     # r: d(r, t) = 0.075 or 0.16, d(r, t') = 0.045 or 0.04
    return Q.astype(np.float32), T.astype(np.float32), 7, 150, 40, tp


@pytest.mark.parametrize("second_in_chain", [True, False])
@pytest.mark.parametrize("rival_nearer", [True, False])
def test_histogram_b_takes_the_in_chain_second(mode_ctx, second_in_chain, rival_nearer):
    rng = np.random.default_rng(31 + 2 * second_in_chain + rival_nearer)
    Q, T, q, r, t, tp = _rival_scene(rng, second_in_chain, rival_nearer)
    D = np.sqrt(((Q[:, None, :].astype(np.float64) - T[None, :, :]) ** 2).sum(-1))
    assert np.argsort(D[r])[:2].tolist() == [tp, t] and D[r, tp] < 0.8 * D[r, t]
    assert np.argmin(D[q]) == t and (D[r, t] < D[q, t]) == rival_nearer
    got = mode_ctx.match_descriptors(Q, T, 0.8, True)
    kept = {int(m["queryIdx"]): int(m["trainIdx"]) for m in got}
    assert kept.get(r) == tp
    assert (q not in kept) if rival_nearer else (kept.get(q) == t), kept.get(q)
    _check(mode_ctx, Q, T)


def _chain_order(n):
    """A train-row order for near_ties' frame that puts its rows a hair apart (300 + k, 450 + k) and its duplicates (600 + k, 640 + k)
    next to each other inside one chain, and its pairs at d1 / d2 = 0.8 (2k, 2k + 1) at an odd offset: every fourth pair straddles a
    chain boundary."""
    order = [r for k in range(150) for r in (300 + k, 450 + k)] + [r for k in range(40) for r in (600 + k, 640 + k)] + [680]
    order += list(range(300))
    return np.array(order + [i for i in range(n) if i not in set(order)])


def test_near_ties_in_chain_fall_back_and_match_the_oracle(mode_ctx):
    Q, T = near_ties(21)
    T = np.ascontiguousarray(T[_chain_order(len(T))])
    _check(mode_ctx, Q, T)
