"""Shared checkers for the parity tests.

Tolerance (BASELINE.json north_star): Hamming -- bit-exact.  L2 -- distances within 1e-5 relative of the
reference's; indices identical except where the reference's competing distances lie within that tolerance.
`justify_l2` implements the second clause with float64 ground-truth distances.
"""
from __future__ import annotations

import numpy as np

REL_TOL = 1e-5  # stated by north_star for SURF distances


def dist64(Q, T):
    """float64 ground-truth L2 distance matrix (direct form)."""
    Q = Q.astype(np.float64)
    T = T.astype(np.float64)
    out = np.empty((Q.shape[0], T.shape[0]), np.float64)
    for a in range(0, Q.shape[0], 512):
        d = Q[a:a + 512, None, :] - T[None, :, :]
        out[a:a + 512] = np.sqrt(np.einsum("qtk,qtk->qt", d, d))
    return out


class LazyDist64:
    """float64 ground-truth distances of a big pair, evaluated row by row / column by column on demand (an 8000 x 8000
    float64 matrix is 512 MB and seconds of work; justify_l2 only ever looks at the few rows and columns that differ)."""

    def __init__(self, Q, T):
        self.Q = Q.astype(np.float64)
        self.T = T.astype(np.float64)
        self.shape = (Q.shape[0], T.shape[0])
        self._rows, self._cols = {}, {}

    def __getitem__(self, key):
        if isinstance(key, tuple):          # D[:, t]
            sl, t = key
            assert sl == slice(None)
            t = int(t)
            if t not in self._cols:
                d = self.Q - self.T[t]
                self._cols[t] = np.sqrt(np.einsum("qk,qk->q", d, d))
            return self._cols[t]
        q = int(key)                        # D[q]
        if q not in self._rows:
            d = self.T - self.Q[q]
            self._rows[q] = np.sqrt(np.einsum("tk,tk->t", d, d))
        return self._rows[q]


def assert_matches_equal(got, ref, exact_distance=True):
    assert len(got) == len(ref), f"match count {len(got)} != {len(ref)}"
    np.testing.assert_array_equal(got["queryIdx"], ref["queryIdx"])
    np.testing.assert_array_equal(got["trainIdx"], ref["trainIdx"])
    assert (got["imgIdx"] == 0).all()
    if exact_distance:
        np.testing.assert_array_equal(got["distance"], ref["distance"])
    else:
        np.testing.assert_allclose(got["distance"], ref["distance"], rtol=REL_TOL, atol=0)


def near(a, b, tol=REL_TOL):
    if not (np.isfinite(a) and np.isfinite(b)):
        return a == b            # (inf - finite = inf would pass the relative test: a missing third neighbour is no near-tie)
    return abs(a - b) <= tol * max(abs(a), abs(b), 1e-30)


def justify_l2(Q, T, ratio, cross_check, got, ref, D=None, tol=REL_TOL):
    """Every difference between `got` and `ref` (DMATCH arrays) must be explained by a near-tie in the
    float64 distances.  Returns the number of differing queries; raises AssertionError on an unexplained one."""
    if D is None:
        D = dist64(Q, T)
    g = {int(m["queryIdx"]): m for m in got}
    r = {int(m["queryIdx"]): m for m in ref}
    diffs = 0
    for q in sorted(set(g) | set(r)):
        mg, mr = g.get(q), r.get(q)
        if mg is not None and mr is not None and mg["trainIdx"] == mr["trainIdx"]:
            assert near(float(mg["distance"]), float(mr["distance"]), tol), (q, mg, mr)
            continue
        diffs += 1
        row = D[q]
        srt = np.sort(row)
        d1, d2 = srt[0], srt[1]
        d3 = srt[2] if len(srt) > 2 else np.inf
        reasons = []
        if near(d1, d2, tol):
            reasons.append("nn1~nn2")
        if near(d2, d3, tol):
            reasons.append("nn2~nn3")
        if near(d1, ratio * d2, 4 * tol):
            reasons.append("ratio-borderline")
        if cross_check:
            for m in (mg, mr):
                if m is not None:
                    col = np.sort(D[:, int(m["trainIdx"])])
                    if len(col) > 1 and near(col[0], col[1], tol):
                        reasons.append("col-tie")
            t1 = int(np.argmin(row))
            col = np.sort(D[:, t1])
            if len(col) > 1 and near(col[0], col[1], tol):
                reasons.append("col-tie")
        assert reasons, f"unexplained difference at query {q}: got={mg} ref={mr} d1={d1} d2={d2} d3={d3}"
    return diffs


def check_knn_l2(Q, T, idx, dist, D=None, tol=REL_TOL):
    """GPU knn-2 (idx, dist) against float64 truth: distances within tol; index swaps only at near-ties."""
    if D is None:
        D = dist64(Q, T)
    nq, nt = D.shape
    order = np.argsort(D, axis=1, kind="stable")
    swaps = 0
    for r in range(min(2, nt)):
        ref_idx = order[:, r]
        ref_d = D[np.arange(nq), ref_idx]
        got_idx = idx[:, r]
        assert (got_idx >= 0).all()
        got_true = D[np.arange(nq), got_idx]
        # reported distance must be the true distance of the reported index
        np.testing.assert_allclose(dist[:, r], got_true, rtol=tol, atol=1e-12)
        bad = got_idx != ref_idx
        swaps += int(bad.sum())
        if bad.any():
            assert np.all(np.abs(got_true[bad] - ref_d[bad]) <= tol * np.maximum(ref_d[bad], 1e-30)), \
                f"rank {r}: index differs from truth beyond tolerance at {np.nonzero(bad)[0][:5]}"
    return swaps
