"""SURVEY 8f rank 1 -- two-view geometric verification (estimate_motion.cpp:27-97, :234-283).

CPU (`-m "not gpu"`): the numpy oracle (oracle/two_view_oracle.py) pinned against cv2 where cv2 is deterministic -- every solution of the minimal
solver on exactly five points, recoverPose, triangulatePoints -- and statistically for whole RANSAC runs (OpenCV's sample sequence cannot be
restated); the committed fixtures tests/golden/two_view.npz (cv2 4.13.0 outputs, tests/golden/make_golden.py); and the product's own float64
math compiled for the host (tests/host/two_view_host.cpp) against the oracle.
GPU: esfm_two_view_batch through the C ABI against the oracle, hypothesis sequence for hypothesis sequence."""
import ctypes

import numpy as np
import pytest

from oracle import two_view_oracle as tvo
from golden_util import load
from two_view_util import DEGENERATE, degenerate_scene, dir_angle_deg, dptr, host_lib, project, random_K, rot_angle_deg, scene


def _same_up_to_sign(E, F, tol):
    return min(np.abs(E - F).max(), np.abs(E + F).max()) <= tol


# --------------------------------------------------------------------------------------------------------------------------------------
# oracle vs cv2
# --------------------------------------------------------------------------------------------------------------------------------------
def test_oracle_minimal_solver_equals_cv2_on_five_points():
    """cv2.findEssentialMat on exactly five points returns every solution of OpenCV's minimal solver (3k x 3): each must be among the
    oracle's, and the counts must agree."""
    import cv2
    total = tight = 0
    for s in range(40):
        K, x1, x2, _, _ = scene(5, 0.3, 0.0, s)
        Ecv, _ = cv2.findEssentialMat(x1, x2, K, cv2.RANSAC, 0.99, 1.0)
        if Ecv is None:
            continue
        Ecv = Ecv.reshape(-1, 3, 3)
        mine = tvo.five_point(tvo.normalise(x1, K), tvo.normalise(x2, K))
        assert len(mine) == len(Ecv), s
        for E in Ecv:
            E = E / np.linalg.norm(E)
            # (a nearly double root is ill-conditioned: OpenCV's degree-10 polynomial and the action matrix then differ in the 5th digit)
            assert any(_same_up_to_sign(E, M, 1e-3) for M in mine), s
            tight += any(_same_up_to_sign(E, M, 1e-8) for M in mine)
            total += 1
    assert total > 100 and tight >= 0.97 * total


def test_oracle_fixtures():
    """The same pins without cv2: committed cv2 outputs (minimal-solver solutions, recoverPose, triangulatePoints, a whole RANSAC run)."""
    z = load("two_view.npz")
    K = z["K"]
    total = tight = 0
    for k in range(int(z["n_five"])):
        mine = tvo.five_point(tvo.normalise(z[f"five_x1_{k}"], K), tvo.normalise(z[f"five_x2_{k}"], K))
        Ecv = z[f"five_E_{k}"].reshape(-1, 3, 3)
        assert len(mine) == len(Ecv)
        for E in Ecv:
            assert any(_same_up_to_sign(E / np.linalg.norm(E), M, 1e-3) for M in mine)
            tight += any(_same_up_to_sign(E / np.linalg.norm(E), M, 1e-8) for M in mine)
            total += 1
    assert total > 60 and tight >= 0.97 * total
    for k in range(int(z["n_scene"])):
        x1, x2, E, mask = z[f"sc_x1_{k}"], z[f"sc_x2_{k}"], z[f"sc_E_{k}"], z[f"sc_mask_{k}"]
        R, t, good, _ = tvo.recover_pose(E, x1, x2, K, mask)
        np.testing.assert_allclose(R, z[f"sc_R_{k}"], atol=1e-9)
        np.testing.assert_allclose(t, z[f"sc_t_{k}"], atol=1e-9)
        assert good == int(z[f"sc_good_{k}"])
        # cv2's inlier mask is the oracle's Sampson test of cv2's own E (float32 error array in OpenCV: borderline points may differ)
        n1, n2 = tvo.normalise(x1, K), tvo.normalise(x2, K)
        err = tvo.sampson_errors(E / np.linalg.norm(E), n1, n2)
        t2 = (1.0 / ((K[0, 0] + K[1, 1]) / 2)) ** 2
        diff = (err <= t2) != mask.astype(bool)
        assert np.all(np.abs(err[diff] - t2) <= 1e-5 * t2)
        np.testing.assert_allclose(tvo.mean_depth(R, t, x1, x2, K, mask), float(z[f"sc_depth_{k}"]), rtol=1e-7)


def test_oracle_ransac_statistics_vs_cv2():
    """Whole RANSAC runs cannot agree match by match (different samples); they must agree as estimators: similar inlier counts, poses as
    close to the truth as cv2's."""
    import cv2
    for s, (noise, outl) in enumerate([(0.3, 0.2), (0.5, 0.4), (0.2, 0.6)]):
        K, x1, x2, R, t = scene(500, noise, outl, 100 + s)
        r = tvo.estimate_two_view(x1, x2, K, 0.99, 1.0, 1000, seed=7, pair=s)
        Ecv, mcv = cv2.findEssentialMat(x1, x2, K, cv2.RANSAC, 0.99, 1.0)
        _, Rcv, tcv, _ = cv2.recoverPose(Ecv, x1, x2, K, mask=mcv.copy())
        assert r["E"] is not None
        assert abs(r["n_inliers"] - int(mcv.sum())) <= 0.25 * int(mcv.sum())
        assert rot_angle_deg(r["R"], R) <= max(2.0, 3.0 * rot_angle_deg(Rcv, R))
        assert dir_angle_deg(r["t"], t) <= max(6.0, 3.0 * dir_angle_deg(tcv, t))      # (raw RANSAC models, no refinement: degrees, not arc minutes)
        inl_true = np.arange(len(x1)) >= int(outl * len(x1))
        assert (r["mask"].astype(bool) & ~inl_true).sum() <= 0.05 * r["n_inliers"] + 3      # few gross outliers accepted


def test_oracle_cheirality_distance_argument():
    """estimate_two_view's `dist` reaches recoverPose: its pose, count and depth are recover_pose's with that threshold, and a threshold
    inside the scene's depth range (4 .. 9) drops points that the default keeps."""
    K, x1, x2, _, _ = scene(300, 0.3, 0.2, 61)
    full = tvo.estimate_two_view(x1, x2, K, 0.99, 1.0, 1000, seed=2, pair=9, random_rate=3)
    near = tvo.estimate_two_view(x1, x2, K, 0.99, 1.0, 1000, seed=2, pair=9, random_rate=3, dist=8.0)
    for r, d in ((full, 50.0), (near, 8.0)):
        R, t, good, _ = tvo.recover_pose(r["E"], x1, x2, K, r["mask"], d)
        assert np.array_equal(r["R"], R) and np.array_equal(r["t"], t) and r["n_good"] == good
        assert r["depth"] == tvo.mean_depth(R, t, x1, x2, K, r["mask"], 3)
    assert np.array_equal(near["E"], full["E"]) and np.array_equal(near["mask"], full["mask"])
    assert 0 < near["n_good"] < full["n_good"]


@pytest.mark.parametrize("noise", [0.0, 0.3])
def test_degenerate_generators(noise):
    """Each degenerate scene is the geometry it claims: points on a plane or a line, t = 0, |t| = 1e-6, depth x 1e4, every correspondence
    2 or 3 times, one correspondence n times, x1 == x2; without noise the pixels are the projections of X."""
    for s, kind in enumerate(DEGENERATE):
        K, x1, x2, R, t, X = degenerate_scene(kind, 200, noise, 70 + s, random_K(np.random.default_rng(s)))
        assert x1.shape == x2.shape == (len(X), 2) and x1.dtype == np.float32
        assert np.all(X[:, 2] > 0) and np.all((X @ R.T + t)[:, 2] > 0)
        if noise == 0.0:
            scale = max(1.0, np.abs(project(K, X)).max())
            np.testing.assert_allclose(x1, project(K, X), atol=1e-6 * scale)
            np.testing.assert_allclose(x2, project(K, X @ R.T + t), atol=1e-6 * scale)
        sv = np.linalg.svd(X - X.mean(0), compute_uv=False)
        if kind == "planar":
            assert sv[2] <= 1e-12 * sv[0] and sv[1] > 0.1 * sv[0]
            np.testing.assert_allclose(X[:, 2], 6.0 + 0.4 * X[:, 0] - 0.3 * X[:, 1], atol=1e-12)
        if kind == "collinear":
            assert sv[1] <= 1e-12 * sv[0]
        if kind in ("rotation", "same"):
            assert np.array_equal(t, np.zeros(3))
        if kind == "baseline":
            assert abs(np.linalg.norm(t) - 1e-6) <= 1e-18
        if kind == "far":
            assert X[:, 2].min() >= 4e4 and X[:, 2].max() <= 9e4 and abs(np.linalg.norm(t) - 1.0) < 1e-12
        if kind == "repeated":
            rows, inv, counts = np.unique(np.c_[x1, x2], axis=0, return_inverse=True, return_counts=True)
            assert len(rows) == 200 and set(counts.tolist()) == {2, 3} and len(x1) == counts.sum()
            assert not np.all(np.diff(inv.ravel()) >= 0)                        # shuffled, not in runs
        if kind == "identical":
            assert len(np.unique(np.c_[x1, x2], axis=0)) == 1 and len(x1) == 200
        if kind == "same":
            assert np.array_equal(x1, x2) and np.array_equal(R, np.eye(3))
        if kind not in ("repeated", "identical"):
            assert len(np.unique(np.c_[x1, x2], axis=0)) == len(x1)


# --------------------------------------------------------------------------------------------------------------------------------------
# the product's float64 math, compiled for the host, vs the oracle
# --------------------------------------------------------------------------------------------------------------------------------------
def test_host_math_equals_oracle():
    L = host_lib()
    for (seed, pair, hyp, m) in [(0, 0, 0, 5), (7, 3, 11, 600), (123456789, 499499, 999, 8000), (2 ** 63 + 5, 12, 0, 6)]:
        out = (ctypes.c_int * 5)()
        L.tvh_sample(ctypes.c_ulonglong(seed), ctypes.c_ulonglong(pair), ctypes.c_ulonglong(hyp), m, out)
        assert list(out) == tvo.sample_indices(seed, pair, hyp, m)
    rng = np.random.default_rng(1)
    n_sol = 0
    for s in range(150):
        K, x1, x2, R, t = scene(5, 0.5, 0.0, 1000 + s)
        q1, q2 = np.ascontiguousarray(tvo.normalise(x1, K)), np.ascontiguousarray(tvo.normalise(x2, K))
        ref = tvo.five_point(q1, q2)
        out = np.zeros(90)
        k = L.tvh_five_point(dptr(q1), dptr(q2), dptr(out))
        mine = out[:9 * k].reshape(k, 3, 3)
        assert k == len(ref)
        for a, b in zip(ref, mine):                      # same order (ascending eigenvalue), same matrices
            assert _same_up_to_sign(a, b, 1e-7)
            n_sol += 1
        # pose pieces on the true essential matrix
        tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
        E = tx @ R
        E = np.ascontiguousarray(E / np.linalg.norm(E) + rng.normal(0, 1e-4, (3, 3)))
        R1, R2, tt = np.zeros(9), np.zeros(9), np.zeros(3)
        L.tvh_decompose(dptr(E), dptr(R1), dptr(R2), dptr(tt))
        o1, o2, ot = tvo.decompose_essential(E)
        got = {tuple(np.round(R1, 9)), tuple(np.round(R2, 9))}
        assert got == {tuple(np.round(o1.ravel(), 9)), tuple(np.round(o2.ravel(), 9))}
        assert min(np.abs(tt - ot).max(), np.abs(tt + ot).max()) < 1e-9
        Q = np.zeros(4)
        Rc, tc = np.ascontiguousarray(R.ravel()), np.ascontiguousarray(t)
        a, b = q1[0], q2[0]
        L.tvh_triangulate(dptr(Rc), dptr(tc), ctypes.c_double(a[0]), ctypes.c_double(a[1]), ctypes.c_double(b[0]), ctypes.c_double(b[1]), dptr(Q))
        ref_q = tvo.triangulate_dlt(np.eye(3, 4), np.c_[R, t], a[None], b[None])[0]
        np.testing.assert_allclose(Q[:3] / Q[3], ref_q[:3] / ref_q[3], rtol=1e-8, atol=1e-10)
    assert n_sol > 400
    for (p, ep, mx) in [(0.99, 0.5, 1000), (0.99, 0.0, 1000), (0.99, 1.0, 1000), (0.999, 0.9, 1000), (0.5, 0.3, 7)]:
        assert L.tvh_update_iters(ctypes.c_double(p), ctypes.c_double(ep), 5, mx) == tvo.ransac_update_num_iters(p, ep, 5, mx)


# --------------------------------------------------------------------------------------------------------------------------------------
# GPU vs oracle
# --------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_two_view_batch_equals_oracle(ctx):
    """One esfm_two_view_batch call over pairs of very different kinds (clean, noisy, outlier-ridden, tiny, hopeless): every pair must take the
    oracle's path -- same number of hypotheses, same best model, same inliers except matches whose Sampson error sits on the threshold, same
    (R, t) and mean depth."""
    cfgs = [(400, 0.3, 0.2), (700, 0.5, 0.4), (250, 1.0, 0.3), (900, 0.2, 0.6), (5, 0.0, 0.0), (3, 0.0, 0.0), (0, 0.0, 0.0), (60, 0.3, 0.0),
            (300, 0.5, 0.97), (1500, 0.4, 0.25)]
    scenes = [scene(n, noise, outl, 300 + k) for k, (n, noise, outl) in enumerate(cfgs)]
    K = scenes[0][0]
    off = np.cumsum([0] + [len(s[1]) for s in scenes]).astype(np.int64)
    p1 = np.concatenate([s[1].reshape(-1, 2) for s in scenes])
    p2 = np.concatenate([s[2].reshape(-1, 2) for s in scenes])
    mask, res = ctx.two_view_batch(off, p1, p2, K, 1.0, 0.99, max_iters=1000, seed=11, first_pair=5)
    t2 = (1.0 / ((K[0, 0] + K[1, 1]) / 2)) ** 2
    for k, sc in enumerate(scenes):
        ref = tvo.estimate_two_view(sc[1], sc[2], K, 0.99, 1.0, 1000, seed=11, pair=5 + k)
        got = res[k]
        assert bool(got["ok"]) == (ref["E"] is not None), k
        assert got["n_matches"] == len(sc[1])
        if ref["E"] is None:
            assert not mask[off[k]:off[k + 1]].any()
            continue
        assert got["iters"] == ref["iters"], (k, got["iters"], ref["iters"])
        assert _same_up_to_sign(got["E"], ref["E"], 1e-6), k
        err = tvo.sampson_errors(ref["E"], tvo.normalise(sc[1], K), tvo.normalise(sc[2], K))
        diff = mask[off[k]:off[k + 1]].astype(bool) != ref["mask"].astype(bool)
        assert np.all(np.abs(err[diff] - t2) <= 1e-6 * t2), k
        if diff.any():
            continue                                                  # (a borderline match moves the counts below)
        assert got["n_inliers"] == ref["n_inliers"]
        np.testing.assert_allclose(got["R"], ref["R"], atol=1e-6)
        np.testing.assert_allclose(got["t"], ref["t"], atol=1e-6)
        assert abs(int(got["n_good"]) - ref["n_good"]) <= 1
        np.testing.assert_allclose(got["depth"], ref["depth"], rtol=1e-6)
    # the estimator is right, not just self-consistent: poses near the truth on the well-posed pairs
    for k in (0, 1, 3, 9):
        assert rot_angle_deg(res[k]["R"], scenes[k][3]) < 1.5 and dir_angle_deg(res[k]["t"], scenes[k][4]) < 4.0
    # per-pair cameras, several chunks' worth of keys: results do not depend on how the job is split into calls
    Ks = np.stack([K] * len(scenes))
    mask2, res2 = ctx.two_view_batch(off[3:] - off[3], p1[off[3]:], p2[off[3]:], Ks[3:], 1.0, 0.99, max_iters=1000, seed=11, first_pair=8)
    assert mask2.tobytes() == mask[off[3]:].tobytes() and res2.tobytes() == res[3:].tobytes()


@pytest.mark.gpu
def test_motion_estimator_mirror(ctx):
    """The Python mirror of MotionEstimator::estimate2D2D_E5P_RANSAC on matches in DMatch form (indices into keypoint arrays)."""
    import easysfm_b200 as esfm
    K, x1, x2, R, t = scene(500, 0.4, 0.3, 77)
    rng = np.random.default_rng(3)
    perm1, perm2 = rng.permutation(500), rng.permutation(500)
    kp1, kp2 = np.zeros((500, 2), np.float32), np.zeros((500, 2), np.float32)
    kp1[perm1], kp2[perm2] = x1, x2
    m = np.zeros(500, esfm.DMATCH_DTYPE)
    m["queryIdx"], m["trainIdx"] = perm1, perm2
    me = esfm.MotionEstimator(ctx, seed=5)
    ok, inl, T = me.estimate2D2D_E5P_RANSAC(kp1, kp2, m, K, 1.0, 0.99)
    assert ok and 250 < len(inl) <= 500 and T.shape == (4, 4) and T.dtype == np.float32
    assert rot_angle_deg(T[:3, :3].astype(np.float64), R) < 1.5 and dir_angle_deg(T[:3, 3], t) < 4.0
    ref = tvo.estimate_two_view(x1, x2, K, 0.99, 1.0, 1000, seed=5, pair=0)
    assert len(inl) == ref["n_inliers"] or abs(len(inl) - ref["n_inliers"]) <= 2
