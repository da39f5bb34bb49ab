"""The tc16 cross-check where its histograms cannot decide (finalize.cu, two-phase): banks with repeated structure, poison rows and
rivals that really win, sent through the verification sweep and checked against the oracle on every engine family.

Phase 1 decides a claimant (the best survivor of the ratio test at its train row) only when no other row's best value (histogram A)
or second value (histogram B) lies at or below its own.  A "poison" query row equal to two identical train rows puts mass in bucket 0
-- in A when it fails the ratio test (ratio 0.8, 1.0), in B when it passes (ratio inf, second value 0) -- so every claimant of its pair
goes to the verification sweep; `verified_rows` counts them.  Each case also holds claimants the cross-check has to drop: a
ratio-failing row nearer to the claimant's train row, a row for which that train row is the second neighbour, and a ratio-failing row
at the claimant's own distance (the lowest index wins the tie).

Rows are built from bit strings: ORB rows are the 256 bits, SURF rows are 64 bits mapped to +-1/16, so that 1/2 d^2 = hamming / 128
exactly.  Competing SURF distances therefore tie exactly or differ by more than 1e-4 relative (sweep ranking error cannot justify a
difference); the borderline ratio h1 / h2 = 0.64 never occurs in the designs.  Oracle answers are computed once per session."""
import os

import numpy as np
import pytest

import oracle
from easysfm_b200 import scheduler, synth
from golden_util import frames_of, load
from util import LazyDist64, assert_matches_equal, dist64, justify_l2

pytestmark = pytest.mark.gpu

RATIOS = (0.8, 1.0, float("inf"))
NBITS = {"orb": 256, "surf": 64}
FULL = {"orb": 4000, "surf": 8000}          # the benchmark's frame sizes: a gather list of about a whole train frame
_CACHE = {}
_ORB_BYTES = {}                             # ORB answers of the first engine that ran a case: the others must equal them byte for byte


class _env:
    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        os.environ.update({k: str(v) for k, v in self.kv.items()})

    def __exit__(self, *exc):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _context(l2, exact=None):
    import easysfm_b200 as esfm
    with _env(**({} if exact is None else {"ESFM_TC16_EXACT": "1" if exact else "0"})):
        c = esfm.Context(0)                 # ESFM_TC16_EXACT is read when the context is created
    c.set_l2_engine(l2)
    return c


@pytest.fixture(scope="module")
def ffma():
    c = _context("ffma")
    yield c
    c.close()


@pytest.fixture(scope="module")
def fast():
    c = _context("tc16", exact=False)
    yield c
    c.close()


@pytest.fixture(scope="module")
def exact():
    c = _context("tc16", exact=True)
    yield c
    c.close()


def _rows(bits, kind):
    """bool [n, NBITS[kind]] -> ORB uint8 [n, 32] or SURF float32 [n, 64] (+-1/16: 1/2 d^2 = hamming / 128)."""
    if kind == "orb":
        return np.ascontiguousarray(np.packbits(bits, axis=1))
    return np.ascontiguousarray(np.where(bits, np.float32(1 / 16), np.float32(-1 / 16)).astype(np.float32))


def _flip(rng, row, n, avoid=()):
    """row with n bits flipped outside `avoid`; returns (new row, flipped positions)."""
    free = np.setdiff1d(np.arange(row.size), np.asarray(avoid, np.int64))
    pos = rng.choice(free, n, replace=False)
    r = row.copy()
    r[pos] ^= True
    return r, pos


def structured_pair(kind, n, g, seed):
    """Query and train frames of n rows whose ratio test at 0.8 leaves g claimants, each of a different train row, plus one poison row.
    Claimants: plain ones (their train row's only near query row, kept), and three kinds of rival, about g / 16 each:
      a) a ratio-failing row at 4 from t (tied at 4 with t' = t + 8 bits), claimant at 5: the claimant is dropped;
      b) a row at 3 from its own t_x and 7 from t (t is its second neighbour), claimant at 8: dropped;
      c) a ratio-failing row at the claimant's own distance 4: the lower query index wins.
    The rest are random rows, which fail the ratio test at 0.8."""
    rng = np.random.default_rng(seed)
    nb = NBITS[kind]
    k = min(max(1, g // 16), (n - g - 2) // 2)
    n_a, n_b, n_c = (1, 0, 0) if g < 5 else (k, k, k)
    n_plain = g - n_a - 2 * n_b - n_c
    assert n_plain >= 0 and n_plain + 2 * (n_a + n_b + n_c) + 2 <= n
    T = rng.random((n, nb)) < 0.5
    Q = rng.random((n, nb)) < 0.5
    ti = qi = 0

    def take_t(row):
        nonlocal ti
        T[ti] = row
        ti += 1

    def take_q(row):
        nonlocal qi
        Q[qi] = row
        qi += 1
    for _ in range(n_plain):
        t = T[ti].copy(); ti += 1
        take_q(_flip(rng, t, 4)[0])
    for kind_r, count in (("a", n_a), ("b", n_b), ("c", n_c)):
        for _ in range(count):
            t = T[ti].copy(); ti += 1
            if kind_r == "b":
                tx, C = _flip(rng, t, 10)
                take_t(tx)
                s = t.copy(); s[C[:7]] ^= True                          # d(s, t) = 7, d(s, t_x) = 3
                take_q(s)
                take_q(_flip(rng, t, 8, avoid=C)[0])                    # d(q, t) = 8, d(q, t_x) = 18
            else:
                t2, A = _flip(rng, t, 8)
                take_t(t2)
                r = t.copy(); r[A[:4]] ^= True                          # d(r, t) = d(r, t') = 4: fails at 0.8 and 1.0
                take_q(r)
                take_q(_flip(rng, t, 5 if kind_r == "a" else 4, avoid=A)[0])   # 5 / 13 or 4 / 12
    p = rng.random(nb) < 0.5                                            # poison: one query row, two identical train rows
    take_t(p); take_t(p); take_q(p)
    pq, pt = rng.permutation(n), rng.permutation(n)
    return _rows(Q[pq], kind), _rows(T[pt], kind)


def _refs(key, Q, T, ratios=RATIOS):
    """Oracle answers of a pair, with and without the cross-check, computed once per session."""
    if key not in _CACHE:
        _CACHE[key] = {(r, cc): oracle.match(Q, T, r, cc) for r in ratios for cc in (False, True)}
    return _CACHE[key]


def _verified(c):
    return c.stats()["verified_rows"]


def _is_tc16(c, kind):
    return (c.l2_engine() if kind == "surf" else c.hamming_engine()) == "tc16"


def _check_pair(ctx, kind, Q, T, key, ffma=None):
    """Every ratio with the cross-check (and, for ORB, without it): the oracle's answer, the verification sweep counted on tc16
    (exactly the claimants at ratio 0.8), nothing counted elsewhere.  SURF on tc16 is also judged against the ffma engine."""
    refs = _refs(key, Q, T)
    D = dist64(Q, T) if kind == "surf" and len(Q) * len(T) <= 4_000_000 else (LazyDist64(Q, T) if kind == "surf" else None)
    claimants = len(set(refs[(0.8, False)]["trainIdx"].tolist()))
    for ratio in RATIOS:
        assert len(refs[(ratio, False)]) > len(refs[(ratio, True)]), ratio      # the cross-check has something to remove
        for cc in ((True, False) if kind == "orb" else (True,)):
            before = _verified(ctx)
            got = ctx.match_descriptors(Q, T, ratio, cc)
            delta = _verified(ctx) - before
            ref = refs[(ratio, cc)]
            if kind == "orb":
                assert_matches_equal(got, ref)
                prev = _ORB_BYTES.setdefault((key, ratio, cc), got.tobytes())
                assert prev == got.tobytes()
            else:
                justify_l2(Q, T, ratio, cc, got, ref, D=D)
                if ffma is not None and _is_tc16(ctx, kind):
                    justify_l2(Q, T, ratio, cc, got, ffma.match_descriptors(Q, T, ratio, cc), D=D)
            if not (cc and _is_tc16(ctx, kind)):
                assert delta == 0, (ratio, cc, delta)
            elif ratio == 0.8:
                assert delta == claimants, (delta, claimants)
            else:
                assert delta > 0, ratio
    return claimants


@pytest.mark.parametrize("g", [1, 127, 128, 129, 300, "full"])
@pytest.mark.parametrize("kind", ["orb", "surf"])
def test_gather_list_sizes_across_tile_edges(ctx, ffma, kind, g):
    """Gather lists of 1, 127, 128, 129 and 300 train rows (1200-row frames), and of about a whole train frame (the benchmark's
    frame sizes): the gathered query operand spans one tile, a tile and a row, several tiles, a partial last tile."""
    n = FULL[kind] if g == "full" else 1200
    want = n - 2 * max(1, n // 64) - 2 if g == "full" else g
    Q, T = structured_pair(kind, n, want, seed=1000 + want)
    got = _check_pair(ctx, kind, Q, T, (kind, n, want), ffma)
    if kind == "orb":
        assert got == want                      # 256-bit random rows never pass the ratio test at 0.8
    else:
        assert abs(got - want) <= 2             # (64-bit ones may, rarely)


@pytest.mark.parametrize("g", [5, 200, "full"])
@pytest.mark.parametrize("kind", ["orb", "surf"])
def test_verification_split_across_units(ctx, ffma, kind, g):
    """One pair of 8000-row frames per call: the forward sweep splits the pair into many units, and the verification launch
    reuses that split for 5, 200 or about 8000 gathered rows (most units empty, or a few tiles spread over units)."""
    n = 8000
    want = n - 2 * (n // 64) - 2 if g == "full" else g
    Q, T = structured_pair(kind, n, want, seed=1000 + want)
    _check_pair(ctx, kind, Q, T, (kind, n, want), ffma)


def repeated_bank(kind, n_frames, seed):
    """Frames of 1000-2000 rows sampled from a shared world of landmarks (8 % of the bits flipped per view), a tenth of them seen
    twice in the same frame (repeated structure: a query row between two copies fails the ratio test near a claimant's distance);
    every second frame also holds the same poison row three times."""
    rng = np.random.default_rng(seed)
    nb = NBITS[kind]
    flip = 0.08 if kind == "orb" else 0.03
    sizes = rng.integers(1000, 2001, n_frames)
    world = rng.random((4 * 2000, nb)) < 0.5
    poison = rng.random(nb) < 0.5
    frames = []
    for f, n in enumerate(sizes):
        n_dup = n // 10
        n_poison = 3 if f % 2 == 0 else 0
        ids = rng.choice(len(world), n - n_dup - n_poison, replace=False)
        ids = np.concatenate([ids, rng.choice(ids, n_dup, replace=False)])
        rows = world[ids] ^ (rng.random((len(ids), nb)) < flip)
        rows = np.concatenate([rows, np.repeat(poison[None], n_poison, 0)])
        frames.append(_rows(rows[rng.permutation(n)], kind))
    return frames


def _bank_case(kind, ctx):
    key = ("bank", kind)
    if key not in _CACHE:
        frames = repeated_bank(kind, 36, seed=7 if kind == "orb" else 8)
        pairs = scheduler.all_pairs(len(frames))
        sel = np.sort(np.random.default_rng(9).choice(len(pairs), 60, replace=False))
        refs = {int(k): _refs(("bank", kind, int(k)), frames[pairs[k][0]], frames[pairs[k][1]]) for k in sel}
        _CACHE[key] = (frames, pairs, refs)
    frames, pairs, refs = _CACHE[key]
    assert len(pairs) >= 4 * ctx.sm_count       # units_per_pair == 1
    return frames, pairs, refs


@pytest.mark.parametrize("kind", ["orb", "surf"])
def test_bench_batch_shape_with_lists_in_many_pairs(ctx, kind):
    """630 pairs in one all-pairs call (one CTA per pair), verification lists in many pairs at once; 60 pairs against the oracle.
    The pairs between two poisoned frames send every claimant to the verification sweep: on tc16 the counter covers at least
    their claimants."""
    frames, pairs, refs = _bank_case(kind, ctx)
    bank = ctx.bank_from_frames(frames)
    for ratio in RATIOS:
        for cc in ((True, False) if kind == "orb" else (True,)):
            before = _verified(ctx)
            res = bank.match_all_pairs(ratio, cc)
            delta = _verified(ctx) - before
            forced = 0
            for k, ref in refs.items():
                i, j, m = res.pair_at(k)
                assert (i, j) == tuple(int(x) for x in pairs[k])
                if kind == "orb":
                    assert_matches_equal(m, ref[(ratio, cc)])
                elif m.tobytes() != ref[(ratio, cc)].tobytes():
                    justify_l2(frames[i], frames[j], ratio, cc, m, ref[(ratio, cc)], D=LazyDist64(frames[i], frames[j]))
                if i % 2 == 0 and j % 2 == 0:
                    forced += len(set(ref[(0.8, False)]["trainIdx"].tolist())) if ratio == 0.8 else 1
            assert sum(len(r[(ratio, False)]) for r in refs.values()) > sum(len(r[(ratio, True)]) for r in refs.values())
            if cc and _is_tc16(ctx, kind):
                assert forced > 0 and delta >= forced, (ratio, delta, forced)
            else:
                assert delta == 0
            res.close()
    bank.close()


@pytest.mark.parametrize("kind", ["orb", "surf"])
def test_chunk_edges_keep_the_lists(ctx, kind):
    """The batch of the previous test in chunks of 1, 7 and 64 pairs: byte-identical matches and counts, and the same number of
    verified train rows as one chunk."""
    frames, _, _ = _bank_case(kind, ctx)
    bank = ctx.bank_from_frames(frames)
    before = _verified(ctx)
    whole = bank.match_all_pairs(0.8, True)
    n_verified = _verified(ctx) - before
    ref_all, ref_off = whole.all_matches()
    assert (n_verified > 0) == _is_tc16(ctx, kind)
    for chunk in (1, 7, 64):
        with _env(ESFM_CHUNK_PAIRS=chunk):
            assert bank.chunk_pairs() == chunk
            before = _verified(ctx)
            parts = bank.match_all_pairs(0.8, True)
            assert _verified(ctx) - before == n_verified, chunk
        got_all, got_off = parts.all_matches()
        assert got_all.tobytes() == ref_all.tobytes() and (got_off == ref_off).all(), chunk
        assert (parts.pair_counts() == whole.pair_counts()).all()
        parts.close()
    whole.close()
    bank.close()


def _unit(x):
    return (x / np.linalg.norm(x, axis=-1, keepdims=True)).astype(np.float32)


def _orth(rng, *dirs):
    """a random unit vector orthogonal to `dirs` (float64)"""
    v = rng.standard_normal(64)
    for d in dirs:
        v -= (v @ d) * d
    return v / np.linalg.norm(v)


def fast_mode_pair(seed):
    """test_gpu_tc16_fast.near_ties (rows at d1 / d2 = 0.8 within 1e-4, train rows a hair apart, exact duplicates of duplicated
    train rows -- poison rows) plus 20 ratio-failing rivals nearer to a claimant's train row and 20 rows for which a claimant's
    train row is the second neighbour."""
    from test_gpu_tc16_fast import near_ties
    Q, T = near_ties(seed)
    rng = np.random.default_rng(seed + 1)
    for k in range(20):
        t = T[700 + k].astype(np.float64)
        u = _orth(rng); v = _orth(rng, u)
        T[720 + k] = t + 0.53 * u                   # t'
        Q[340 + k] = t + 0.25 * u                   # d(r, t) = 0.25, d(r, t') = 0.28: fails at 0.8
        Q[360 + k] = t + 0.30 * v                   # claimant at 0.30: dropped
        t2 = T[760 + k].astype(np.float64)
        u = _orth(rng); v = _orth(rng, u)
        T[740 + k] = t2 + 0.5 * u                   # t_x
        Q[380 + k] = t2 + 0.29 * u                  # d(s, t_x) = 0.21, d(s, t2) = 0.29
        Q[400 + k] = t2 + 0.32 * v                  # claimant at 0.32: dropped
    return np.ascontiguousarray(Q, np.float32), np.ascontiguousarray(T, np.float32)


def test_surf_fast_mode_fallback_and_verification_in_one_pair(ctx, fast, exact):
    """The gather buffer carries the fallback list first, then phase 1's verification list: rows of both kinds in one pair.  Fast
    mode re-sweeps rows and verifies train rows, and returns exactly the bytes of exact mode; both pass against the oracle."""
    Q, T = fast_mode_pair(21)
    refs = _refs(("fast", 21), Q, T)
    D = dist64(Q, T)
    for ratio in RATIOS:
        assert len(refs[(ratio, False)]) > len(refs[(ratio, True)])
        fb, vr = fast.stats()["fallback_rows"], _verified(fast)
        a = fast.match_descriptors(Q, T, ratio, True)
        assert fast.stats()["fallback_rows"] > fb and _verified(fast) > vr, ratio
        b = exact.match_descriptors(Q, T, ratio, True)
        assert a.tobytes() == b.tobytes(), ratio
        justify_l2(Q, T, ratio, True, a, refs[(ratio, True)], D=D)
        justify_l2(Q, T, ratio, True, ctx.match_descriptors(Q, T, ratio, True), refs[(ratio, True)], D=D)


def margin_bank(scale, n_pairs, seed):
    """Pairs of a 2-row query frame (claimant q, rival r) and a 2-row train frame (t, t'), rows of norm `scale` (four components
    of scale / 2, the offsets in the other 60): r fails the ratio test (d(r, t') = d(r, t) / 0.9) and is nearer to t than q is.
    Their 1/2 d^2 sit within 1e-4 of the bucket boundary 8 / 512, the offsets swept over the pairs: in half of them both lie below
    it with q + 1e-5 (phase 1's margin on unit rows) still below, in the other half on either side of it.  The sweep's error grows
    with the squared norms, so a margin that did not would let phase 1 decide q although r is nearer."""
    rng = np.random.default_rng(seed)
    B = 8 / 512
    frames = []
    for k in range(n_pairs):
        S = rng.choice(64, 4, replace=False)
        t = np.zeros(64)
        t[S] = scale / 2
        u = rng.standard_normal(64); u[S] = 0; u /= np.linalg.norm(u)
        v = rng.standard_normal(64); v[S] = 0; v -= (v @ u) * u; v /= np.linalg.norm(v)
        if k % 2 == 0:
            q_val = B - 1e-5 - rng.uniform(1e-6, 9e-5)
            r_val = q_val - rng.uniform(2e-6, 1e-4)
        else:
            q_val = B + rng.uniform(1e-6, 1e-4)
            r_val = B - rng.uniform(1e-6, 1e-4)
        rho = np.sqrt(2 * r_val)
        q = t + np.sqrt(2 * q_val) * v
        r = t + rho * u
        t2 = t + (rho + rho / 0.9) * u
        frames += [np.array([q, r], np.float32), np.array([t, t2], np.float32)]
    return frames


def _check_margin_bank(contexts, scale):
    """q and r lie at least 6e-5 apart relative in d, so the answers are compared exactly: with the cross-check at ratio 0.8 every
    pair's answer is empty (the claimant loses to the ratio-failing rival), without it q -> t; at 1.0 and inf r -> t.  On tc16 every
    claimant at ratio 0.8 has to go to the verification sweep."""
    n = 48
    frames = margin_bank(scale, n, seed=int(scale))
    pairs = [[2 * k, 2 * k + 1] for k in range(n)]
    refs = [_refs(("margin", scale, k), frames[2 * k], frames[2 * k + 1]) for k in range(n)]
    for ref in refs:
        assert len(ref[(0.8, True)]) == 0 and ref[(0.8, False)][["queryIdx", "trainIdx"]].tolist() == [(0, 0)]
        assert ref[(1.0, True)][["queryIdx", "trainIdx"]].tolist() == [(1, 0)]
    for c in contexts:
        bank = c.bank_from_frames(frames)
        for ratio in RATIOS:
            for cc in (True, False):
                before = _verified(c)
                res = bank.match_pairs(pairs, ratio, cc)
                delta = _verified(c) - before
                for k in range(n):
                    assert_matches_equal(res.pair_at(k)[2], refs[k][(ratio, cc)], exact_distance=False)
                if not (cc and _is_tc16(c, "surf")):
                    assert delta == 0
                elif ratio == 0.8:
                    assert delta == n, delta
                res.close()
        bank.close()


@pytest.mark.parametrize("scale", [16.0, 64.0])
def test_surf_phase1_margin_at_non_unit_magnitudes(fast, exact, scale):
    """Phase 1 compares a claimant's direct-form 1/2 d^2 with the sweep's values of its rivals: a margin that ignores the rows'
    norms lets a rival pushed across a bucket boundary by the sweep's error leave the claimant decided (with the absolute 1e-5
    margin it did at norm 64).  Exact mode and fast mode, whose rows of this magnitude all go to the exact fallback sweep."""
    _check_margin_bank((fast, exact), scale)


@pytest.mark.xfail(strict=True, reason="ffma / tc decide the cross-check on the column minimum ranked in expansion form; when it names "
                                        "the claimant itself, finalize keeps it unchecked, and at norms 16 and 64 the ranking error exceeds "
                                        "the gap to a nearer rival (DESIGN 5.3)")
@pytest.mark.parametrize("scale", [16.0, 64.0])
@pytest.mark.parametrize("engine", ["ffma", "tc"])
def test_surf_one_sweep_cross_check_at_non_unit_magnitudes(engine, scale):
    """The same pairs on the engines that decide the cross-check with column minima in one sweep."""
    c = _context(engine)
    try:
        _check_margin_bank((c,), scale)
    finally:
        c.close()


def test_bench_banks_verify_no_rows(ctx):
    """DESIGN 5.3: on the benchmark's generators (four 8000-row SURF frames of synth.surf_like_torch, four 4000-row ORB frames of
    synth.orb_like) the histograms decide every claimant and the verification sweep has nothing to do."""
    import torch
    data = synth.surf_like_torch(4, 8000, 4, torch.device("cuda:0")).cpu().numpy()
    for frames in ([np.ascontiguousarray(data[i]) for i in range(4)], synth.orb_like(4, 4000, seed=4)):
        bank = ctx.bank_from_frames(frames)
        before = _verified(ctx)
        res = bank.match_all_pairs(0.8, True)
        assert _verified(ctx) == before
        assert res.n_matches > 4000
        res.close()
        bank.close()


@pytest.mark.parametrize("kind", ["orb", "surf"])
def test_entry_points_agree(ctx, kind):
    """The per-pair entry, the batch entry and esfm_multi_* (device 0 listed twice) return the same bytes on verification cases."""
    import easysfm_b200 as esfm
    Q, T = structured_pair(kind, 1200, 129, seed=1129)
    F, G = structured_pair(kind, 1200, 300, seed=1300)
    frames = [Q, T, F, G]
    pairs = [[0, 1], [2, 3], [1, 0], [3, 2]]
    bank = ctx.bank_from_frames(frames)
    with esfm.MultiContext([0, 0]) as multi:
        multi.set_engines(l2=ctx.l2_engine(), hamming=ctx.hamming_engine())
        mb = multi.bank_from_frames(frames)
        for ratio in (0.8, float("inf")):
            batch = bank.match_pairs(pairs, ratio, True)
            many = mb.match_pairs(pairs, ratio, True)
            for k, (i, j) in enumerate(pairs):
                one = ctx.match_descriptors(frames[i], frames[j], ratio, True)
                assert one.tobytes() == batch.pair_at(k)[2].tobytes() == many.pair_at(k)[2].tobytes(), (ratio, i, j)
            batch.close(); many.close()
        mb.close()
    bank.close()


def _tiled_views(seed, tiles):
    """A patch of orb_util.image tiled tiles x tiles with small per-tile noise, and a second view of it shifted by (5, 9) pixels."""
    from orb_util import image
    rng = np.random.default_rng(seed)
    patch = image(seed, 120, 160, 14).astype(np.int16)
    big = np.block([[patch + rng.integers(-3, 4, patch.shape) for _ in range(tiles)] for _ in range(tiles)])
    big = np.clip(big, 0, 255).astype(np.uint8)
    return np.ascontiguousarray(big[:-9, :-5]), np.ascontiguousarray(big[9:, 5:])


@pytest.mark.parametrize("tiles", [3, 4])
def test_orb_repeated_texture_from_extraction(ctx, tiles):
    """ORB descriptors extracted on the device from a tiled texture and a shifted view of it: duplicates and Hamming ties
    everywhere, as repeated structure gives.  Bit-exact against the oracle; on tc16 the verification sweep runs."""
    a, b = _tiled_views(40 + tiles, tiles)
    _, Q = ctx.orb_extract(a, 3000)
    _, T = ctx.orb_extract(b, 3000)
    refs = _refs(("tiled", tiles), Q, T)
    n_verified = 0
    for ratio in RATIOS:
        for cc in (True, False):
            before = _verified(ctx)
            assert_matches_equal(ctx.match_descriptors(Q, T, ratio, cc), refs[(ratio, cc)])
            n_verified += _verified(ctx) - before
    assert (n_verified > 0) == _is_tc16(ctx, "orb"), n_verified


def test_fountain_images_through_the_verification_sweep(ctx):
    """The 11 fountain images' ORB(8000) descriptors, all 55 pairs with the cross-check, bit-exact against cv2's answers; real
    images leave train rows undecided, and tc16 verifies them."""
    from golden_util import as_matches
    z = load("fountain_orb.npz")
    fr = frames_of(z)
    bank = ctx.bank_from_frames(fr)
    before = _verified(ctx)
    res = bank.match_all_pairs(0.8, True)
    n_verified = _verified(ctx) - before
    for k in range(res.n_pairs):
        i, j, m = res.pair_at(k)
        assert_matches_equal(m, as_matches(z[f"m_r80_c1_{i}_{j}_idx"], z[f"m_r80_c1_{i}_{j}_dist"]))
    # at most every claimant (the distinct train rows of the ratio test's survivors), and on tc16 fewer: the histograms decide some
    claimants = sum(len(set(z[f"m_r80_c0_{i}_{j}_idx"][:, 1].tolist())) for i, j, _ in res)
    if _is_tc16(ctx, "orb"):
        assert 0 < n_verified < claimants, (n_verified, claimants)
    else:
        assert n_verified == 0
    res.close()
    bank.close()
