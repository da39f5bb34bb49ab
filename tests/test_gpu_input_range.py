"""SURF matching across the descriptor values the library accepts, and frames at the largest sizes the bank accepts.

Each SURF engine is correct on a range of component magnitudes (DESIGN.md section 5.0, "Input range"): tc16 rounds components to fp16,
tc and ffma keep running thresholds below fixed sentinels.  A bank outside the context's engine's range is swept by the next engine that
covers it (tc16 -> tc -> ffma); non-finite components and magnitudes beyond every engine are refused at commit.  These tests judge every
answer against oracle.match with justify_l2, at magnitudes from 2^-20 to past fp16's range, in banks whose frames differ in scale, at the
largest SURF and ORB frames a bank accepts, and check that one row more is refused.

The oracle's answers for the large frames are computed once per session and shared by the engine parametrisations.
"""
import os

import numpy as np
import pytest

import oracle
from util import LazyDist64, assert_matches_equal, justify_l2, near

pytestmark = pytest.mark.gpu

FP16_MAX = 65504.0
RATIOS = (0.8, 1.0, float("inf"))


def _unit(x):
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def contention(seed, nq=1500, nt=1100):
    """test_gpu_parity.test_cross_check_contention's SURF rows: queries at graded distances from shared train rows, exact duplicates,
    queries between two train rows."""
    rng = np.random.default_rng(seed)
    T = _unit(rng.standard_normal((nt, 64)))
    Q = _unit(rng.standard_normal((nq, 64)))

    def jitter(row, s):
        return _unit((row + s * rng.standard_normal(64))[None])[0]
    for k in range(nq // 5):
        Q[int(rng.integers(0, nq))] = jitter(T[int(rng.integers(0, 200))], float(rng.uniform(0.0, 0.12)))
    for k in range(40):
        Q[int(rng.integers(0, nq))] = T[int(rng.integers(200, 220))]
    for k in range(60):
        a, b = int(rng.integers(0, 200)), int(rng.integers(220, 260))
        T[b] = jitter(T[a], 0.01)
        Q[int(rng.integers(0, nq))] = jitter(T[a], 0.005)
    return Q, T


def _scaled(Q, T, sq, st):
    return (Q * np.float32(sq)).astype(np.float32), (T * np.float32(st)).astype(np.float32)


def _check_all(c, Q, T):
    for ratio in RATIOS:
        for cc in (False, True):
            justify_l2(Q, T, ratio, cc, c.match_descriptors(Q, T, ratio, cc), oracle.match(Q, T, ratio, cc))


# (query scale, train scale).  2^17 puts the largest components of unit rows (about 0.5) past fp16's 65504; 2^50 is past the tc
# sweep's range (2^44), so such a bank runs on ffma whatever the context's engine.
MAGNITUDES = [(2.0 ** -20, 2.0 ** -20), (2.0 ** -20, 2.0 ** -19), (2.0 ** -12, 2.0 ** -12), (2.0 ** -12, 2.0 ** -11), (1.0, 1.0),
              (1.0, 2.0), (2.0 ** 8, 2.0 ** 8), (2.0 ** 15, 2.0 ** 15), (2.0 ** 15, 2.0 ** 16), (2.0 ** 17, 2.0 ** 17),
              (2.0 ** 17, 2.0 ** 16), (2.0 ** 50, 2.0 ** 50)]


@pytest.mark.parametrize("sq,st", MAGNITUDES, ids=[f"q2^{np.log2(a):g}-t2^{np.log2(b):g}" for a, b in MAGNITUDES])
def test_magnitude_sweep(ctx, sq, st):
    Q, T = _scaled(*contention(17), sq, st)
    _check_all(ctx, Q, T)


def test_straddles_fp16_range(ctx):
    """Rows at 2^15 with a few components above 65504 in both frames: the rest of the bank is inside fp16's range, those are not."""
    Q, T = _scaled(*contention(23), 2.0 ** 15, 2.0 ** 15)
    rng = np.random.default_rng(5)
    for M in (Q, T):
        rows = rng.choice(len(M), 6, replace=False)
        M[rows, rng.integers(0, 64, 6)] = np.float32(70000.0) * rng.choice([-1, 1], 6).astype(np.float32)
    assert np.abs(T).max() > FP16_MAX and (np.abs(T) > FP16_MAX).sum() == 6
    _check_all(ctx, Q, T)


def test_mixed_scale_bank(ctx):
    """Six frames from 2^-20 to past fp16's range in one bank: every ordered pair, also the ones that never touch the large frame."""
    scales = [2.0 ** -20, 2.0 ** -12, 1.0, 2.0 ** 8, 2.0 ** 15, 2.0 ** 17]
    frames = []
    for k, s in enumerate(scales):
        Q, _ = contention(40 + k, nq=600, nt=300)
        frames.append((Q * np.float32(s)).astype(np.float32))
    frames[-1][3, 7] = np.float32(90000.0)
    bank = ctx.bank_from_frames(frames)
    pairs = [(i, j) for i in range(6) for j in range(6) if i != j]
    for ratio, cc in ((0.8, True), (float("inf"), False)):
        res = bank.match_pairs(pairs, ratio, cc)
        assert res.n_pairs == 30
        for k in range(res.n_pairs):
            i, j, m = res.pair_at(k)
            justify_l2(frames[i], frames[j], ratio, cc, m, oracle.match(frames[i], frames[j], ratio, cc))
    bank.close()


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
def fast_exact():
    a, b = _context(False), _context(True)
    yield a, b
    a.close()
    b.close()


def test_small_magnitudes_fall_back_or_leave_tc16(fast_exact):
    """At 2^-4 (largest component about 2^-5, twice the smallest tc16 keeps) the fast sweep's bound flags rows for the exact fallback sweep;
    at 2^-20 fp16's subnormal step is larger than the distances' differences, and the bank runs on tc instead: no fallback rows.  Both
    modes give the same matches byte for byte, and the oracle's."""
    fast, exact = fast_exact
    for s, want_fallback in ((2.0 ** -4, True), (2.0 ** -20, False)):
        Q, T = _scaled(*contention(17), s, s)
        before = fast.stats()["fallback_rows"]
        for ratio in RATIOS:
            for cc in (False, True):
                a = fast.match_descriptors(Q, T, ratio, cc)
                b = exact.match_descriptors(Q, T, ratio, cc)
                assert len(a) == len(b)
                for f in ("queryIdx", "trainIdx", "distance"):
                    np.testing.assert_array_equal(a[f], b[f])
                justify_l2(Q, T, ratio, cc, a, oracle.match(Q, T, ratio, cc))
        assert (fast.stats()["fallback_rows"] > before) == want_fallback, s


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf, 2.0 ** 60])
def test_out_of_domain_components_are_refused(ctx, bad):
    """A NaN or infinite component, or one beyond every engine's range, is refused at commit -- through a bank and through
    match_descriptors -- instead of producing matches."""
    import easysfm_b200 as esfm
    Q, T = contention(3, nq=200, nt=300)
    T[77, 5] = np.float32(bad)
    with pytest.raises(esfm.EsfmError) as e:
        ctx.bank_from_frames([Q, T])
    assert e.value.code == 1 and "frame 1" in str(e.value)
    with pytest.raises(esfm.EsfmError):
        ctx.match_descriptors(T, Q, 0.8, True)
    justify_l2(Q, T[:77], 0.8, True, ctx.match_descriptors(Q, T[:77], 0.8, True), oracle.match(Q, T[:77], 0.8, True))   # still usable


# ---- the largest frames ------------------------------------------------------------------------------------------------------------
BIG_SURF = 70000
SURF_DUPS = (32767, 65535)          # rows 32767 / 32768 and 65535 / 65536 of the big frame are equal
_CACHE = {}


def _surf_big():
    if "surf" not in _CACHE:
        rng = np.random.default_rng(7)
        big = _unit(rng.standard_normal((BIG_SURF, 64)))
        small = [_unit(rng.standard_normal((n, 64))) for n in (1500, 3000)]
        for k, r in enumerate(SURF_DUPS):
            big[r + 1] = big[r]
            for s in small:
                s[10 + k] = big[r]                                  # queries equal to the duplicated rows
                s[20 + k] = _unit((big[r] + 0.01 * rng.standard_normal(64))[None])[0]
        frames = [big] + small
        pairs = [(0, 1), (0, 2), (1, 0), (2, 0)]
        refs = {(p, cc): oracle.match(frames[p[0]], frames[p[1]], 0.8, cc) for p in pairs for cc in (False, True)}
        knn = {p: oracle.knn2(frames[p[0]], frames[p[1]]) for p in pairs}
        _CACHE["surf"] = (frames, pairs, refs, knn)
    return _CACHE["surf"]


def test_surf_frame_past_2_16_rows(ctx):
    """A 70,000-row frame against 1,500- and 3,000-row frames, as query frame and as train frame: match_pairs with and without the
    cross-check, and knn2_pair, whose duplicates at rows 32767 / 32768 and 65535 / 65536 rank lowest index first."""
    frames, pairs, refs, knn = _surf_big()
    bank = ctx.bank_from_frames(frames)
    for cc in (False, True):
        res = bank.match_pairs(pairs, 0.8, cc)
        for k, p in enumerate(pairs):
            q, t, m = res.pair_at(k)
            assert (q, t) == p
            justify_l2(frames[q], frames[t], 0.8, cc, m, refs[(p, cc)], D=LazyDist64(frames[q], frames[t]))
            if p[0] == 0 and cc:             # of two equal query rows only the lower one can be the train row's nearest
                for r in SURF_DUPS:
                    assert r + 1 not in set(m["queryIdx"].tolist())
    for p in pairs:
        idx, dist = bank.knn2_pair(*p)
        ridx, rdist = knn[p]
        if p[1] == 0:
            for k, r in enumerate(SURF_DUPS):
                assert idx[10 + k].tolist() == [r, r + 1] and dist[10 + k].tolist() == [0.0, 0.0]
        D = LazyDist64(frames[p[0]], frames[p[1]])
        np.testing.assert_allclose(dist, rdist, rtol=1e-5, atol=1e-12)
        for q, r in zip(*np.nonzero(idx != ridx)):            # a different index only at a float64 near-tie
            row = np.sort(D[q])
            assert near(row[r], D[q][idx[q, r]]) and (near(row[0], row[1]) or near(row[1], row[min(2, len(row) - 1)])), (p, q, r)
    bank.close()


def _max_rows(ctx, kind):
    """The largest frame a bank of `kind` accepts, found by refusal of esfm_bank_set_frame_rows (host-side, nothing allocated)."""
    import easysfm_b200 as esfm
    b = esfm.Bank(ctx, kind, 1)
    lo, hi = 1, 1 << 22
    while lo < hi:
        mid = (lo + hi + 1) // 2
        try:
            b.set_frame_rows(0, mid)
            lo = mid
        except esfm.EsfmError as e:
            assert e.code == 5
            hi = mid - 1
    b.close()
    return lo


def _orb_big(n):
    if ("orb", n) not in _CACHE:
        rng = np.random.default_rng(9)
        big = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        small = rng.integers(0, 256, (2000, 32), dtype=np.uint8)
        for k in range(50):                                       # near copies, duplicates at the frame's last rows
            small[k] = big[n - 1 - k]
            small[k][k % 32] ^= np.uint8(1 << (k % 8))
        big[n - 2] = big[n - 1]
        small[60] = big[n - 1]
        frames = [big, small]
        refs = {(p, cc): oracle.match(frames[p[0]], frames[p[1]], 0.8, cc) for p in ((0, 1), (1, 0)) for cc in (False, True)}
        knn = {p: oracle.knn2(frames[p[0]], frames[p[1]]) for p in ((0, 1), (1, 0))}
        _CACHE[("orb", n)] = (frames, refs, knn)
    return _CACHE[("orb", n)]


def test_orb_frame_at_the_row_limit(ctx):
    """A frame of exactly the largest accepted row count, in both roles, bit-exact against the oracle on every Hamming engine."""
    import easysfm_b200 as esfm
    n = _max_rows(ctx, esfm.KIND_B256)
    assert n > 32768                                              # past the Z key's limit: the +-1 encoding on the tc engine
    frames, refs, knn = _orb_big(n)
    bank = ctx.bank_from_frames(frames)
    for cc in (False, True):
        res = bank.match_pairs([(0, 1), (1, 0)], 0.8, cc)
        for k, p in enumerate(((0, 1), (1, 0))):
            q, t, m = res.pair_at(k)
            assert (q, t) == p
            assert_matches_equal(m, refs[(p, cc)])
    for p in ((0, 1), (1, 0)):
        idx, dist = bank.knn2_pair(*p)
        np.testing.assert_array_equal(idx, knn[p][0])
        np.testing.assert_array_equal(dist, knn[p][1])
    assert knn[(1, 0)][0][60].tolist() == [n - 2, n - 1]
    bank.close()


def test_one_row_over_the_limit_is_refused(ctx):
    """set_frame refuses a frame one row longer than the largest accepted, for both kinds, with ERR_CAPACITY; the SURF frame
    (2^20 + 1 rows, 268 MB of zero pages) is never read."""
    import easysfm_b200 as esfm
    for kind, cols, dtype in ((esfm.KIND_B256, 32, np.uint8), (esfm.KIND_F32X64, 64, np.float32)):
        n = _max_rows(ctx, kind)
        if kind == esfm.KIND_F32X64:
            assert n == 1 << 20
        b = esfm.Bank(ctx, kind, 1)
        with pytest.raises(esfm.EsfmError) as e:
            b.set_frame(0, np.zeros((n + 1, cols), dtype))
        assert e.value.code == 5
        b.close()
