"""CPU restatement (numpy, float64) of the reference's two-view geometric verification -- TEST INFRASTRUCTURE ONLY (SURVEY 8f rank 1).

Reference: p3dv::MotionEstimator::estimate2D2D_E5P_RANSAC, cpp_code/src/estimate_motion.cpp:27-97 (called at cpp_code/test/sfm.cpp:165):
    cv::findEssentialMat(pts1, pts2, K, RANSAC, prob, thre, mask)   :48-49   -> inlier_matches = matches with mask set   :54-60
    cv::recoverPose(E, pts1, pts2, K, R, t, mask)                   :65      -> T = [R t; 0 1]                            :72-82
and MotionEstimator::getDepthFast, :234-283 (sfm.cpp:166): triangulate every random_rate-th inlier with [I|0], T_21, mean point norm.

The arithmetic lives in OpenCV (calib3d: five-point.cpp, ptsetreg.cpp, triangulate.cpp), which is not vendored under /root/reference; its
PUBLISHED algorithm is restated here:
  * normalisation by K, threshold / ((fx + fy) / 2);
  * minimal solver: Nister's five-point problem solved with the action-matrix method (null space of the 5 x 9 epipolar system, the ten cubic
    constraints det E = 0 and 2 E E^T E - tr(E E^T) E = 0 in the three null-space coordinates, Gauss-Jordan on the 10 x 20 coefficient
    matrix, eigenvectors of the 10 x 10 multiplication matrix);
  * model error = Sampson distance (x2^T E x1)^2 / (|E x1|_xy^2 + |E^T x2|_xy^2), inlier iff error <= threshold^2;
  * RANSAC with OpenCV's adaptive stopping rule (RANSACUpdateNumIters), the best model = most inliers, first found wins ties;
  * recoverPose: the four (R, t) of the SVD, triangulation of all points, points in front of both cameras and nearer than 50, masked by the
    inliers; OpenCV's preference order on ties;
  * triangulation: homogeneous DLT (smallest singular vector of the 4 x 4 system).
What cannot be restated is OpenCV's random SAMPLE SEQUENCE (cv::RNG state shared across calls): RANSAC here draws its 5-subsets from a
counter-based generator (sample_indices) that the CUDA implementation reproduces bit for bit, so the CUDA path is compared with this oracle
hypothesis by hypothesis, and this oracle is pinned against cv2 where cv2 is deterministic (every solution of the minimal solver on exactly
five points; recoverPose; triangulatePoints) and statistically where it is not (inlier sets and poses of whole RANSAC runs).  Parity of the
full RANSAC against the reference is therefore 'pinned up to the sample sequence' -- see tests/test_two_view.py.
"""
from __future__ import annotations

import numpy as np

MASK64 = (1 << 64) - 1


def splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & MASK64
    z = x
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK64
    return z ^ (z >> 31)


def sample_indices(seed: int, pair: int, hyp: int, m: int):
    """Five distinct match indices in [0, m) for hypothesis `hyp` of pair `pair`: a stream of splitmix64 values keyed by (seed, pair, hyp),
    each reduced with the high product (v * m) >> 64, duplicates skipped."""
    out = []
    key = splitmix64((seed ^ splitmix64(pair & MASK64)) & MASK64)
    key = splitmix64((key ^ (hyp * 0xD6E8FEB86659FD93)) & MASK64)
    c = 0
    while len(out) < 5:
        v = splitmix64((key + c) & MASK64)
        c += 1
        i = (v * m) >> 64
        if i not in out:
            out.append(int(i))
    return out


# ---- polynomials in (x, y, z) of total degree <= 3 as 4 x 4 x 4 coefficient arrays ----------------------------------------------------
def _pmul(a, b):
    out = np.zeros((4, 4, 4))
    ia = np.argwhere(a != 0)
    for i, j, k in ia:
        ib = np.argwhere(b != 0)
        for p, q, r in ib:
            if i + p < 4 and j + q < 4 and k + r < 4:
                out[i + p, j + q, k + r] += a[i, j, k] * b[p, q, r]
    return out


# monomial order of the 10 x 20 system: the ten cubics first, then x^2, xy, xz, y^2, yz, z^2, x, y, z, 1
MONOMIALS = [(3, 0, 0), (2, 1, 0), (2, 0, 1), (1, 2, 0), (1, 1, 1), (1, 0, 2), (0, 3, 0), (0, 2, 1), (0, 1, 2), (0, 0, 3),
             (2, 0, 0), (1, 1, 0), (1, 0, 1), (0, 2, 0), (0, 1, 1), (0, 0, 2), (1, 0, 0), (0, 1, 0), (0, 0, 1), (0, 0, 0)]


def five_point(q1, q2):
    """All real essential matrices (each scaled to unit Frobenius norm) through five correspondences in NORMALISED coordinates:
    q2_h^T E q1_h = 0.  Returns an array (n, 3, 3), n <= 10."""
    q1 = np.asarray(q1, np.float64)
    q2 = np.asarray(q2, np.float64)
    A = np.stack([np.kron([q2[i, 0], q2[i, 1], 1.0], [q1[i, 0], q1[i, 1], 1.0]) for i in range(5)])
    _, _, vt = np.linalg.svd(A)
    B = vt[5:9].reshape(4, 3, 3)                      # E = x B0 + y B1 + z B2 + B3
    E = np.empty((3, 3), object)
    for r in range(3):
        for c in range(3):
            p = np.zeros((4, 4, 4))
            p[1, 0, 0], p[0, 1, 0], p[0, 0, 1], p[0, 0, 0] = B[0, r, c], B[1, r, c], B[2, r, c], B[3, r, c]
            E[r, c] = p
    EEt = np.empty((3, 3), object)
    for r in range(3):
        for c in range(3):
            EEt[r, c] = sum(_pmul(E[r, k], E[c, k]) for k in range(3))
    tr = EEt[0, 0] + EEt[1, 1] + EEt[2, 2]
    eqs = []
    for r in range(3):
        for c in range(3):
            eqs.append(2.0 * sum(_pmul(EEt[r, k], E[k, c]) for k in range(3)) - _pmul(tr, E[r, c]))
    det = (_pmul(E[0, 0], _pmul(E[1, 1], E[2, 2]) - _pmul(E[1, 2], E[2, 1]))
           - _pmul(E[0, 1], _pmul(E[1, 0], E[2, 2]) - _pmul(E[1, 2], E[2, 0]))
           + _pmul(E[0, 2], _pmul(E[1, 0], E[2, 1]) - _pmul(E[1, 1], E[2, 0])))
    eqs.append(det)
    M = np.array([[e[m] for m in MONOMIALS] for e in eqs])          # 10 x 20
    try:
        Bm = np.linalg.solve(M[:, :10], M[:, 10:])                 # cubic_i = - sum_j Bm[i, j] basis_j
    except np.linalg.LinAlgError:
        return np.zeros((0, 3, 3))
    Ax = np.zeros((10, 10))                                          # multiplication by x in the basis (x^2, xy, xz, y^2, yz, z^2, x, y, z, 1)
    Ax[0:6] = -Bm[0:6]                                               # x*x^2 = x^3, x*xy = x^2 y, x*xz = x^2 z, x*y^2 = x y^2, x*yz = xyz, x*z^2 = x z^2
    Ax[6, 0] = Ax[7, 1] = Ax[8, 2] = Ax[9, 6] = 1.0                  # x*x = x^2, x*y = xy, x*z = xz, x*1 = x
    w, V = np.linalg.eig(Ax)
    sols = []
    for k in range(10):
        if abs(w[k].imag) > 1e-9 * max(1.0, abs(w[k].real)):
            continue
        v = V[:, k].real
        if abs(v[9]) < 1e-14:
            continue
        v = v / v[9]
        Ek = v[6] * B[0] + v[7] * B[1] + v[8] * B[2] + B[3]
        n = np.linalg.norm(Ek)
        if n > 0 and np.isfinite(n):
            sols.append(Ek / n)
    # a canonical order that depends on neither the null-space basis nor the sign of E: ascending leading 2 x 2 minor
    sols.sort(key=lambda M: M[0, 0] * M[1, 1] - M[0, 1] * M[1, 0])
    return np.array(sols).reshape(-1, 3, 3)


def sampson_errors(E, n1, n2):
    """(x2^T E x1)^2 / (|E x1|_xy^2 + |E^T x2|_xy^2) for every correspondence (normalised coordinates, float64)."""
    x1 = np.c_[n1, np.ones(len(n1))]
    x2 = np.c_[n2, np.ones(len(n2))]
    Ex1 = x1 @ E.T
    Etx2 = x2 @ E
    num = np.einsum("ij,ij->i", x2, Ex1) ** 2
    return num / (Ex1[:, 0] ** 2 + Ex1[:, 1] ** 2 + Etx2[:, 0] ** 2 + Etx2[:, 1] ** 2)


def ransac_update_num_iters(p, ep, model_points, max_iters):
    p = min(max(p, 0.0), 1.0)
    ep = min(max(ep, 0.0), 1.0)
    num = max(1.0 - p, np.finfo(np.float64).tiny)
    denom = 1.0 - (1.0 - ep) ** model_points
    if denom < np.finfo(np.float64).tiny:
        return 0
    num, denom = np.log(num), np.log(denom)
    if denom >= 0 or -num >= max_iters * (-denom):
        return max_iters
    return int(np.floor(num / denom + 0.5))


def normalise(pts, K):
    pts = np.asarray(pts, np.float64)
    return np.c_[(pts[:, 0] - K[0, 2]) / K[0, 0], (pts[:, 1] - K[1, 2]) / K[1, 1]]


def find_essential_ransac(pts1, pts2, K, prob=0.99, thre=1.0, max_iters=1000, seed=0, pair=0):
    """findEssentialMat(RANSAC) with this module's sample sequence.  Returns (E, mask uint8[m], hypotheses evaluated)."""
    K = np.asarray(K, np.float64)
    n1, n2 = normalise(pts1, K), normalise(pts2, K)
    m = len(n1)
    mask = np.zeros(m, np.uint8)
    if m < 5:
        return None, mask, 0
    t2 = (thre / ((K[0, 0] + K[1, 1]) / 2.0)) ** 2
    best_count, best_E, niters, it = 4, None, max_iters, 0
    while it < niters:
        idx = sample_indices(seed, pair, it, m)
        for E in five_point(n1[idx], n2[idx]):
            cnt = int((sampson_errors(E, n1, n2) <= t2).sum())
            if cnt > best_count:
                best_count, best_E = cnt, E
                niters = ransac_update_num_iters(prob, (m - cnt) / m, 5, niters)
        it += 1
    if best_E is None:
        return None, mask, it
    mask[:] = sampson_errors(best_E, n1, n2) <= t2
    return best_E, mask, it


def triangulate_dlt(P1, P2, a, b):
    """cv::triangulatePoints: per correspondence the smallest right singular vector of [a_x P1_3 - P1_1; a_y P1_3 - P1_2; b_x P2_3 - P2_1; ...]."""
    out = np.empty((len(a), 4))
    for i in range(len(a)):
        A = np.stack([a[i, 0] * P1[2] - P1[0], a[i, 1] * P1[2] - P1[1], b[i, 0] * P2[2] - P2[0], b[i, 1] * P2[2] - P2[1]])
        out[i] = np.linalg.svd(A)[2][3]
    return out


def decompose_essential(E):
    U, _, Vt = np.linalg.svd(E)
    if np.linalg.det(U) < 0:
        U = -U
    if np.linalg.det(Vt) < 0:
        Vt = -Vt
    W = np.array([[0.0, 1.0, 0.0], [-1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    return U @ W @ Vt, U @ W.T @ Vt, U[:, 2].copy()


def cheirality_counts(E, pts1, pts2, K, mask, dist=50.0):
    """recoverPose's four candidates (R1, t), (R2, t), (R1, -t), (R2, -t) and, for each, the masked matches triangulated in front of both
    cameras and nearer than `dist`: returns (candidates, counts, per-match uint8 masks)."""
    K = np.asarray(K, np.float64)
    n1, n2 = normalise(pts1, K), normalise(pts2, K)
    R1, R2, t = decompose_essential(E)
    P0 = np.eye(3, 4)
    cands = [(R1, t), (R2, t), (R1, -t), (R2, -t)]
    goods, masks = [], []
    for R, tt in cands:
        P = np.c_[R, tt]
        Q = triangulate_dlt(P0, P, n1, n2)
        ok = Q[:, 2] * Q[:, 3] > 0
        X = Q[:, :3] / Q[:, 3:4]
        ok &= X[:, 2] < dist
        X2 = X @ R.T + tt
        ok &= (X2[:, 2] > 0) & (X2[:, 2] < dist)
        ok &= mask.astype(bool)
        goods.append(int(ok.sum()))
        masks.append(ok.astype(np.uint8))
    return cands, goods, masks


def recover_pose(E, pts1, pts2, K, mask, dist=50.0):
    """cv::recoverPose(E, pts1, pts2, K, R, t, mask) (calib3d five-point.cpp): returns (R, t, n_good, mask_out)."""
    cands, goods, masks = cheirality_counts(E, pts1, pts2, K, mask, dist)
    g1, g2, g3, g4 = goods
    if g1 >= g2 and g1 >= g3 and g1 >= g4:
        k = 0
    elif g2 >= g1 and g2 >= g3 and g2 >= g4:
        k = 1
    elif g3 >= g1 and g3 >= g2 and g3 >= g4:
        k = 2
    else:
        k = 3
    return cands[k][0], cands[k][1], goods[k], masks[k]


def mean_depth(R, t, pts1, pts2, K, mask, random_rate=1):
    """getDepthFast (estimate_motion.cpp:234-283) on the inlier matches: every random_rate-th inlier triangulated with [I|0] and [R|t],
    mean Euclidean norm of the points."""
    K = np.asarray(K, np.float64)
    sel = np.flatnonzero(mask)[::random_rate]
    if len(sel) == 0:
        return float("nan")
    n1, n2 = normalise(np.asarray(pts1)[sel], K), normalise(np.asarray(pts2)[sel], K)
    Q = triangulate_dlt(np.eye(3, 4), np.c_[R, t], n1, n2)
    X = Q[:, :3] / Q[:, 3:4]
    return float(np.linalg.norm(X, axis=1).mean())


def estimate_two_view(pts1, pts2, K, prob=0.99, thre=1.0, max_iters=1000, seed=0, pair=0, random_rate=1, dist=50.0):
    """The whole of estimate2D2D_E5P_RANSAC + getDepthFast for one image pair; `dist` is recoverPose's distance threshold.  Returns a dict."""
    E, mask, iters = find_essential_ransac(pts1, pts2, K, prob, thre, max_iters, seed, pair)
    out = {"E": E, "mask": mask, "iters": iters, "n_inliers": int(mask.sum()), "R": None, "t": None, "n_good": 0, "depth": float("nan")}
    if E is None:
        return out
    R, t, good, pmask = recover_pose(E, pts1, pts2, K, mask, dist)
    out.update(R=R, t=t, n_good=good, depth=mean_depth(R, t, pts1, pts2, K, mask, random_rate))
    return out
