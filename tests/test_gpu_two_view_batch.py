"""GPU: esfm_two_view_batch the way an all-pairs job calls it, against the numpy oracle (oracle/two_view_oracle.py).

  * one batch of 8,300 pairs: three chunks of the batch loop (4096 pairs each), per-pair cameras, random_rate 20, first_pair and seed
    other than 0; real scenes at the chunk edges are compared with the oracle, hypothesis sequence for hypothesis sequence;
  * the same pairs split into other calls, and the same call repeated, give the same bytes;
  * parameter edges: max_iters around the 64-hypothesis round, ransac_prob, ransac_thre, random_rate against the inlier count, cheirality_dist;
  * degenerate scenes (planar, collinear, pure rotation, tiny baseline, distant points, repeated and identical correspondences, x1 == x2),
    where the GPU's and the oracle's minimal solvers may return different solutions: every output finite and consistent with the GPU's own E
    under the oracle's deterministic stages;
  * esfm_two_view_depth on its own for every random_rate up to INT_MAX."""
import numpy as np
import pytest

from easysfm_b200 import capi
from oracle import two_view_oracle as tvo
from two_view_util import DEGENERATE, degenerate_scene, random_K, scene

pytestmark = pytest.mark.gpu

CHUNK = 4096                  # pairs per chunk of esfm_two_view_batch's loop (two_view.cu)
EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def tctx():
    """Two-view verification does not depend on the matching engine: one context for the module."""
    c = capi.Context(0)
    yield c
    c.close()


def _same_up_to_sign(E, F, tol):
    return min(np.abs(E - F).max(), np.abs(E + F).max()) <= tol


def _concat(pairs):
    off = np.cumsum([0] + [len(p[0]) for p in pairs]).astype(np.int64)
    p1 = np.concatenate([np.asarray(p[0], np.float32).reshape(-1, 2) for p in pairs])
    p2 = np.concatenate([np.asarray(p[1], np.float32).reshape(-1, 2) for p in pairs])
    return off, p1, p2


def _t2(K, thre):
    return (thre / ((K[0, 0] + K[1, 1]) / 2.0)) ** 2


def check_equals_oracle(got, mask, x1, x2, K, ref, thre=1.0, tag=None):
    """The rules of test_two_view_batch_equals_oracle: same number of hypotheses, E to 1e-6 up to sign, masks equal except at matches whose
    Sampson error sits on the threshold, and (when no such match moved the counts) R, t to 1e-6, n_good +-1, depth to rtol 1e-6."""
    assert got["n_matches"] == len(x1), tag
    assert bool(got["ok"]) == (ref["E"] is not None), tag
    assert got["iters"] == ref["iters"], (tag, got["iters"], ref["iters"])
    if ref["E"] is None:
        assert not mask.any() and got["n_inliers"] == 0 and not got["E"].any(), tag
        return
    assert _same_up_to_sign(got["E"], ref["E"], 1e-6), tag
    t2 = _t2(K, thre)
    err = tvo.sampson_errors(ref["E"], tvo.normalise(x1, K), tvo.normalise(x2, K))
    diff = mask.astype(bool) != ref["mask"].astype(bool)
    assert np.all(np.abs(err[diff] - t2) <= 1e-6 * t2), tag
    if diff.any():
        return                                                        # (a borderline match moves the counts below)
    assert got["n_inliers"] == ref["n_inliers"], tag
    np.testing.assert_allclose(got["R"], ref["R"], atol=1e-6, err_msg=str(tag))
    np.testing.assert_allclose(got["t"], ref["t"], atol=1e-6, err_msg=str(tag))
    assert abs(int(got["n_good"]) - ref["n_good"]) <= 1, tag
    np.testing.assert_allclose(got["depth"], ref["depth"], rtol=1e-6, err_msg=str(tag))


# --------------------------------------------------------------------------------------------------------------------------------------
# a. one all-pairs-shaped batch across three chunks
# --------------------------------------------------------------------------------------------------------------------------------------
N_PAIRS = 8300
FIRST_PAIR = 123457
SEED = 0x5EEDF00D
RATE = 20
EDGES = [0, CHUNK - 1, CHUNK, CHUNK + 1, 2 * CHUNK - 1, 2 * CHUNK, N_PAIRS - 1]


def _big_batch():
    rng = np.random.default_rng(2024)
    others = np.setdiff1d(np.arange(N_PAIRS), EDGES)
    real = sorted(set(EDGES) | set(rng.choice(others, 25, replace=False).tolist()))
    Ks = np.stack([random_K(rng) for _ in range(N_PAIRS)])
    pairs, kinds = [], []
    for k in range(N_PAIRS):
        if k in real:
            n, noise, outl = int(rng.integers(300, 601)), rng.uniform(0.2, 0.5), rng.uniform(0.0, 0.3)
            kinds.append("real")
        elif k % 3 == 0:
            n, noise, outl = int(rng.integers(0, 5)), 0.3, 0.0
            kinds.append("tiny")
        elif k % 3 == 1:
            n, noise, outl = int(rng.integers(5, 7)), 0.3, 0.0
            kinds.append("five")
        else:
            n, noise, outl = int(rng.integers(30, 81)), 0.3, rng.uniform(0.0, 0.4)
            kinds.append("filler")
        _, x1, x2, R, t = scene(n, noise, outl, 10_000 + k, K=Ks[k])
        pairs.append((x1, x2, R, t))
    off, p1, p2 = _concat(pairs)
    return real, kinds, Ks, pairs, off, p1, p2


@pytest.fixture(scope="module")
def big(tctx):
    real, kinds, Ks, pairs, off, p1, p2 = _big_batch()
    mask, res = tctx.two_view_batch(off, p1, p2, Ks, 1.0, 0.99, max_iters=1000, seed=SEED, first_pair=FIRST_PAIR, random_rate=RATE)
    return dict(real=real, kinds=kinds, Ks=Ks, pairs=pairs, off=off, p1=p1, p2=p2, mask=mask, res=res)


def test_chunked_batch_equals_oracle(big):
    """Real scenes at both sides of every chunk boundary and 25 others, each with its own camera, its own sampler key (first_pair + k) and
    every 20th inlier triangulated for the depth, are the oracle's."""
    off, mask, res = big["off"], big["mask"], big["res"]
    assert len(res) == N_PAIRS
    most_inliers = {}
    for k in big["real"]:
        x1, x2 = big["pairs"][k][:2]
        ref = tvo.estimate_two_view(x1, x2, big["Ks"][k], 0.99, 1.0, 1000, seed=SEED, pair=FIRST_PAIR + k, random_rate=RATE)
        check_equals_oracle(res[k], mask[off[k]:off[k + 1]], x1, x2, big["Ks"][k], ref, tag=k)
        assert res[k]["ok"], k
        most_inliers[k] = int(res[k]["n_inliers"])
    # tv_pose_kernel numbers the inliers 128 matches at a time: boundary scenes with more than 128 inliers carry the count across blocks
    assert sum(most_inliers[k] > 128 for k in EDGES) >= 3


def test_chunked_batch_small_pairs(big):
    """Pairs of fewer than five matches are never verified; pairs of exactly five or six take the oracle's path."""
    off, mask, res, kinds = big["off"], big["mask"], big["res"], big["kinds"]
    tiny = [k for k in range(N_PAIRS) if kinds[k] == "tiny"]
    assert {int(off[k + 1] - off[k]) for k in tiny} == {0, 1, 2, 3, 4}
    for k in tiny:
        r = res[k]
        assert r["ok"] == 0 and r["n_inliers"] == 0 and r["iters"] == 0 and not mask[off[k]:off[k + 1]].any(), k
        assert r["n_matches"] == off[k + 1] - off[k]
    five = [k for k in range(N_PAIRS) if kinds[k] == "five"]
    for k in five[:10] + [k for k in five if k >= CHUNK][:10] + five[-10:]:
        x1, x2 = big["pairs"][k][:2]
        ref = tvo.estimate_two_view(x1, x2, big["Ks"][k], 0.99, 1.0, 1000, seed=SEED, pair=FIRST_PAIR + k, random_rate=RATE)
        check_equals_oracle(res[k], mask[off[k]:off[k + 1]], x1, x2, big["Ks"][k], ref, tag=k)
    for f in ("E", "R", "t", "depth"):
        assert np.isfinite(res[f]).all(), f
    assert np.array_equal(res["n_matches"], np.diff(off))
    cs = np.concatenate([[0], np.cumsum(mask, dtype=np.int64)])
    assert np.array_equal(res["n_inliers"], cs[off[1:]] - cs[off[:-1]])


def test_batch_split_and_repeat_are_byte_identical(tctx, big):
    """Where the batch is split into calls does not change a byte: slices that straddle the chunk boundaries, with the matching first_pair
    and cameras, reproduce the full run, and the full run repeated reproduces itself."""
    off, p1, p2, Ks = big["off"], big["p1"], big["p2"], big["Ks"]
    for a, b in [(4000, 4200), (8100, N_PAIRS), (CHUNK - 1, CHUNK + 1), (1, 2 * CHUNK + 3)]:
        m, r = tctx.two_view_batch(off[a:b + 1] - off[a], p1[off[a]:off[b]], p2[off[a]:off[b]], Ks[a:b], 1.0, 0.99, max_iters=1000, seed=SEED,
                                   first_pair=FIRST_PAIR + a, random_rate=RATE)
        assert m.tobytes() == big["mask"][off[a]:off[b]].tobytes(), (a, b)
        assert r.tobytes() == big["res"][a:b].tobytes(), (a, b)
    m, r = tctx.two_view_batch(off, p1, p2, Ks, 1.0, 0.99, max_iters=1000, seed=SEED, first_pair=FIRST_PAIR, random_rate=RATE)
    assert m.tobytes() == big["mask"].tobytes() and r.tobytes() == big["res"].tobytes()


# --------------------------------------------------------------------------------------------------------------------------------------
# c. parameter edges
# --------------------------------------------------------------------------------------------------------------------------------------
# (n, noise, outliers): the stopping rule fires after ~10 to ~60 hypotheses on the first five scenes and after ~150 on the last, so the max_iters
# caps below bind on some scenes and not on others.  The last scene costs the oracle ~10 ms a hypothesis: only the capped runs take it.
EDGE_SCENES = [(400, 0.3, 0.1), (350, 0.25, 0.25), (450, 0.2, 0.2), (300, 0.3, 0.15), (500, 0.3, 0.35), (400, 0.3, 0.5)]
N_EASY = 5
EDGE_SEED, EDGE_FIRST = 99, 777


@pytest.fixture(scope="module")
def edge_scenes():
    rng = np.random.default_rng(5)
    out = []
    for k, (n, noise, outl) in enumerate(EDGE_SCENES):
        K = random_K(rng)
        _, x1, x2, _, _ = scene(n, noise, outl, 500 + k, K=K)
        out.append((K, x1, x2))
    return out


def _run_edges(tctx, sc, first=0, **kw):
    """One batch call over the scenes sc, which are edge_scenes[first:first + len(sc)] (so each keeps its sampler key)."""
    off, p1, p2 = _concat([(x1, x2) for _, x1, x2 in sc])
    Ks = np.stack([K for K, _, _ in sc])
    prm = dict(ransac_thre=1.0, ransac_prob=0.99, max_iters=1000, random_rate=1, cheirality_dist=50.0)
    prm.update(kw)
    mask, res = tctx.two_view_batch(off, p1, p2, Ks, seed=EDGE_SEED, first_pair=EDGE_FIRST + first, **prm)
    return [(mask[off[k]:off[k + 1]], res[k]) for k in range(len(sc))], prm


def _oracle(K, x1, x2, k, prm):
    return tvo.estimate_two_view(x1, x2, K, prm["ransac_prob"], prm["ransac_thre"], prm["max_iters"], seed=EDGE_SEED, pair=EDGE_FIRST + k,
                                 random_rate=prm["random_rate"], dist=prm["cheirality_dist"])


@pytest.mark.parametrize("kw", [dict(max_iters=v) for v in (1, 5, 63, 64, 65, 130)] + [dict(ransac_prob=v) for v in (0.5, 0.999999)]
                         + [dict(ransac_thre=v) for v in (0.3, 3.0)] + [dict(cheirality_dist=8.0)],
                         ids=lambda kw: "-".join(f"{k}={v}" for k, v in kw.items()))
def test_parameter_edges_equal_oracle(tctx, edge_scenes, kw):
    sc = edge_scenes if "max_iters" in kw else edge_scenes[:N_EASY]
    got, prm = _run_edges(tctx, sc, **kw)
    for k, ((K, x1, x2), (mask, r)) in enumerate(zip(sc, got)):
        ref = _oracle(K, x1, x2, k, prm)
        check_equals_oracle(r, mask, x1, x2, K, ref, thre=prm["ransac_thre"], tag=(kw, k))
        assert r["iters"] <= prm["max_iters"]
    if "max_iters" in kw:
        assert max(int(r["iters"]) for _, r in got) == kw["max_iters"]          # the cap binds on at least one scene
    if "cheirality_dist" in kw:
        full, _ = _run_edges(tctx, sc)
        assert any(int(r["n_good"]) < int(f["n_good"]) for (_, r), (_, f) in zip(got, full))     # the distance cuts some points


def test_random_rate_edges_equal_oracle(tctx, edge_scenes):
    """getDepthFast's every-random_rate-th inlier, at rates around the inlier count and far above it: only the depth changes."""
    base, prm = _run_edges(tctx, edge_scenes[:N_EASY])
    for k, (K, x1, x2) in enumerate(edge_scenes[:N_EASY]):
        ref = _oracle(K, x1, x2, k, prm)
        mask, r = base[k]
        check_equals_oracle(r, mask, x1, x2, K, ref, tag=k)
        n_inl = int(r["n_inliers"])
        assert n_inl > 128                                             # (the inlier numbering carries across blocks of 128 matches)
        for rate in (1, 2, 7, 20, n_inl - 1, n_inl, n_inl + 1, 10 ** 6):
            m2, r2 = _run_edges(tctx, [(K, x1, x2)], first=k, random_rate=rate)[0][0]
            assert m2.tobytes() == mask.tobytes()
            for f in ("E", "R", "t", "n_inliers", "n_good", "iters", "ok"):
                assert np.array_equal(r2[f], r[f]), (k, rate, f)
            d = tvo.mean_depth(r2["R"], r2["t"], x1, x2, K, m2, rate)
            np.testing.assert_allclose(r2["depth"], d, rtol=1e-6, err_msg=str((k, rate)))
            if rate >= n_inl:                                          # only inlier 0
                first = np.flatnonzero(m2)[:1]
                np.testing.assert_allclose(r2["depth"], tvo.mean_depth(r2["R"], r2["t"], x1[first], x2[first], K, [1], 1), rtol=1e-6)


# --------------------------------------------------------------------------------------------------------------------------------------
# d. degenerate scenes
# --------------------------------------------------------------------------------------------------------------------------------------
def dlt_error_bound(R, t, n1, n2):
    """Per match: the unit DLT solution Q of the oracle and a bound on how far the GPU's may lie from it.  The GPU takes the smallest
    eigenvector of A^T A by Jacobi rotations; its rounding error is at most ~eps * ||A^T A|| / (lambda_3 - lambda_4) = eps * s1^2 / (s3^2 - s4^2)
    (s_i the singular values of the 4 x 4 DLT system), taken here with a factor 64.  Points triangulated with w ~ 0 (parallel rays:
    pure rotation, tiny baselines, x1 == x2) have s3 ~ s4 and no useful bound; well-conditioned points have one near 1e-13."""
    P1, P2 = np.eye(3, 4), np.c_[R, t]
    Q = np.empty((len(n1), 4))
    bound = np.empty(len(n1))
    for i in range(len(n1)):
        a, b = n1[i], n2[i]
        A = np.stack([a[0] * P1[2] - P1[0], a[1] * P1[2] - P1[1], b[0] * P2[2] - P2[0], b[1] * P2[2] - P2[1]])
        _, s, vt = np.linalg.svd(A)
        Q[i] = vt[3]
        gap = s[2] ** 2 - s[3] ** 2
        bound[i] = 64.0 * EPS * s[0] ** 2 / gap if gap > 0 else np.inf
    return Q, bound


def cheirality_intervals(E, x1, x2, K, mask, dist):
    """For each of recoverPose's four candidates: the oracle's count and the number of masked matches whose test the rounding bound of
    dlt_error_bound cannot decide (a sign or a comparison with `dist` within the error)."""
    cands, goods, _ = tvo.cheirality_counts(E, x1, x2, K, mask, dist)
    n1, n2 = tvo.normalise(x1, K), tvo.normalise(x2, K)
    sel = mask.astype(bool)
    unsure = []
    for R, t in cands:
        Q, bq = dlt_error_bound(R, t, n1[sel], n2[sel])
        with np.errstate(divide="ignore", invalid="ignore"):
            X = Q[:, :3] / Q[:, 3:4]
            ex = bq * (1.0 + np.linalg.norm(X, axis=1)) / np.abs(Q[:, 3])          # error of X
            z2 = X @ R[2] + t[2]
            u = ((np.abs(Q[:, 2]) <= bq) | (np.abs(Q[:, 3]) <= bq) | (np.abs(X[:, 2] - dist) <= 4 * ex) | (np.abs(z2) <= 4 * ex)
                 | (np.abs(z2 - dist) <= 4 * ex) | ~np.isfinite(ex))
        unsure.append(int(u.sum()))
    return cands, goods, unsure


def check_self_consistent(r, mask, x1, x2, K, prm, tag):
    """An `ok` pair must be what the oracle's deterministic stages make of the GPU's own E: its mask, the iteration bound of the stopping
    rule, recoverPose's choice and count, getDepthFast's depth."""
    m = len(x1)
    for f in ("E", "R", "t", "depth"):
        assert np.isfinite(r[f]).all(), (tag, f)
    if not r["ok"]:
        assert not mask.any() and r["n_inliers"] == 0, tag
        return
    E = r["E"]
    t2 = _t2(K, prm["ransac_thre"])
    n1, n2 = tvo.normalise(x1, K), tvo.normalise(x2, K)
    err = tvo.sampson_errors(E, n1, n2)
    diff = mask.astype(bool) != (err <= t2)
    assert np.all(np.abs(err[diff] - t2) <= 1e-6 * t2), tag
    n_inl = int(r["n_inliers"])
    assert n_inl == int(mask.sum()) > 4, tag
    assert tvo.ransac_update_num_iters(prm["ransac_prob"], 1.0 - n_inl / m, 5, prm["max_iters"]) <= r["iters"] <= prm["max_iters"], tag
    cands, goods, unsure = cheirality_intervals(E, x1, x2, K, mask, prm["cheirality_dist"])
    lo = [g - u for g, u in zip(goods, unsure)]
    hi = [g + u for g, u in zip(goods, unsure)]
    w = int(np.argmax(lo))
    if all(lo[w] > hi[c] for c in range(4) if c != w):                # the winning count is unique whatever the rounding
        np.testing.assert_allclose(r["R"], cands[w][0], atol=1e-6, err_msg=str(tag))
        np.testing.assert_allclose(r["t"], cands[w][1], atol=1e-6, err_msg=str(tag))
        assert lo[w] <= r["n_good"] <= hi[w], tag
    else:                                                             # a tie: the SVD signs of the two sides may pick different candidates
        assert max(lo) <= r["n_good"] <= max(hi), tag
    # getDepthFast with the GPU's pose; the tolerance grows past rtol 1e-6 only by the rounding bound of the selected points
    sel = np.flatnonzero(mask)[::prm["random_rate"]]
    d = tvo.mean_depth(r["R"], r["t"], x1, x2, K, mask, prm["random_rate"])
    Q, bq = dlt_error_bound(r["R"], r["t"], n1[sel], n2[sel])
    with np.errstate(divide="ignore", invalid="ignore"):
        X = Q[:, :3] / Q[:, 3:4]
        cond = float(np.mean(bq * (1.0 + np.linalg.norm(X, axis=1)) / np.abs(Q[:, 3])))
    if np.isfinite(cond):
        assert abs(r["depth"] - d) <= 1e-6 * abs(d) + cond, (tag, r["depth"], d, cond)


DEGEN_PRM = dict(ransac_thre=1.0, ransac_prob=0.99, max_iters=1000, random_rate=20, cheirality_dist=50.0)


def test_degenerate_scenes(tctx):
    rng = np.random.default_rng(17)
    items = []
    for kind in DEGENERATE:
        for noise in (0.0, 0.3):
            K = random_K(rng)
            _, x1, x2, _, _, _ = degenerate_scene(kind, 90 if kind == "repeated" else 240, noise, 40 + len(items), K)
            items.append((kind, noise, K, x1, x2))
    off, p1, p2 = _concat([(x1, x2) for *_, x1, x2 in items])
    Ks = np.stack([it[2] for it in items])
    mask, res = tctx.two_view_batch(off, p1, p2, Ks, seed=3, first_pair=41, **DEGEN_PRM)
    n_ok = 0
    for k, (kind, noise, K, x1, x2) in enumerate(items):
        mk, r = mask[off[k]:off[k + 1]], res[k]
        tag = (kind, noise)
        if kind in ("planar", "collinear"):                          # both minimal solvers agree here: the strict comparison holds
            ref = tvo.estimate_two_view(x1, x2, K, DEGEN_PRM["ransac_prob"], DEGEN_PRM["ransac_thre"], DEGEN_PRM["max_iters"], seed=3,
                                        pair=41 + k, random_rate=DEGEN_PRM["random_rate"])
            check_equals_oracle(r, mk, x1, x2, K, ref, tag=tag)
        check_self_consistent(r, mk, x1, x2, K, DEGEN_PRM, tag)
        n_ok += int(r["ok"])
    assert n_ok >= 10


# --------------------------------------------------------------------------------------------------------------------------------------
# e. esfm_two_view_depth on its own
# --------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 127, 128, 129, 5000])
def test_depth_every_rate(tctx, n):
    """Every random_rate-th match from match 0, n_used = ceil(n / random_rate), for rates up to INT_MAX (a 32-bit start or stride would
    wrap there)."""
    rng = np.random.default_rng(n)
    K = random_K(rng)
    _, x1, x2, R, t = scene(n, 0.3, 0.0, 900 + n, K=K)
    for rate in (1, 2, 20, 127, 128, 129, n - 1, n, n + 1, 2 ** 24, 2 ** 30, 2 ** 31 - 1):
        if rate < 1:
            continue
        d, used = tctx.two_view_depth(x1, x2, K, R, t, rate, return_used=True)
        assert used == -(-n // rate), (n, rate, used)
        np.testing.assert_allclose(d, tvo.mean_depth(R, t, x1, x2, K, np.ones(n, np.uint8), rate), rtol=1e-6, err_msg=str((n, rate)))
    with pytest.raises(capi.EsfmError):
        tctx.two_view_depth(x1, x2, K, R, t, 0)
