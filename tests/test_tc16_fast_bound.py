"""The error bound of the SURF tc16 FAST sweep (sweep_win.cu, 9 MMA slots per tile) and the classification built on it, modelled in
numpy against float64 (no GPU).

The fast sweep ranks by v' = a_q.(a_t + b_t) - 1/2|q|^2 - 1/2|t|^2 (a = fp16(x), b = fp16(x - a)); esfm_internal.cuh win_fast_eps bounds
|v' + 1/2 d^2| per query row from |q - a_q|_2 and the frames' largest norms, and win_ratio_class / win_classify_kernel decide from the
sweep's values alone which rows pass or fail the ratio test for certain and which go to the exact fallback sweep.  The model below
restates both in float32 operation by operation (the device code uses non-contracted _rn arithmetic) and checks:
  * the bound holds on adversarial rows: norms x1/16 .. x16, components in fp16's subnormal range, exact duplicates;
  * every row the classification settles is settled correctly (same verdict, same nearest column as float64);
  * on bench-like synthetic frames (synth.surf_like, 8000 x 8000) no row needs the fallback.
"""
import numpy as np

from easysfm_b200 import synth

F32 = np.float32


def f16(x):
    return x.astype(np.float16).astype(np.float32)          # round to nearest even, subnormals kept: cvt.rn.f16.f32


def row_eps(X):
    """pack_tch_kernel: |x - fp16(x)|_2 per row, rounded up."""
    d = (X - f16(X)).astype(np.float64)
    return (np.sqrt((d * d).sum(1)) * (1 + 2.0 ** -16)).astype(F32)


def frame_norm(X):
    x = X.astype(np.float64)
    return F32(np.sqrt((x * x).sum(1)).max() * (1 + 2.0 ** -16))


def win_fast_eps(e_q, n_q, n_t):
    """esfm_internal.cuh win_fast_eps, same float32 operations in the same order."""
    e_q, n_q, n_t = F32(e_q), F32(n_q), F32(n_t)
    m = F32(0.5) * (n_q * n_q + n_t * n_t) + n_q * n_t
    r = (n_q + e_q) * (F32(2.0 ** -22) * (n_t + F32(1)))
    return ((e_q * n_t + r) + F32(2.0 ** -15) * m) * F32(1.001)


def win_ratio_class(s1, s2, e, r2):
    """esfm_internal.cuh win_ratio_class, vectorised: 0 = certain fail, 1 = certain pass, 2 = decide exactly."""
    s1, s2, e, r2 = F32(s1), F32(s2), F32(e), F32(r2)
    fail = (s1 - e) > (r2 * (s2 + e)) * F32(1.001) + F32(4e-6)
    pas = ((s1 + e) < (r2 * (s2 - e)) * F32(0.999) - F32(4e-6)) & ((e == 0) | ((s2 - s1) > F32(2) * e))
    return np.where(fail, 0, np.where(pas, 1, 2))


def half_d2(Q, T):
    """(exact 1/2 d^2, fast-sweep 1/2 d^2 without the fp32 accumulation rounding) in float64."""
    q, t = Q.astype(np.float64), T.astype(np.float64)
    hq, ht = 0.5 * (q * q).sum(1), 0.5 * (t * t).sum(1)
    exact = hq[:, None] + ht[None, :] - q @ t.T
    at = f16(T).astype(np.float64)
    bt = f16(T - f16(T)).astype(np.float64)
    fast = hq[:, None] + ht[None, :] - f16(Q).astype(np.float64) @ (at + bt).T
    return exact, fast


def check_bound(Q, T):
    exact, fast = half_d2(Q, T)
    n_q, n_t = frame_norm(Q), frame_norm(T)
    e_q = row_eps(Q)
    eps = np.array([win_fast_eps(e, n_q, n_t) for e in e_q], np.float64)
    err = np.abs(fast - exact).max(axis=1)
    # the representation part alone (what the model computes exactly) already lies within the bound, with the accumulation term to spare
    rep = e_q.astype(np.float64) * n_t + (float(n_q) + e_q) * 2.0 ** -22 * (float(n_t) + 1)
    assert (err <= rep).all(), float((err - rep).max())
    assert (err <= eps).all()
    return err, eps


def adversarial_rows(rng, n):
    X = rng.standard_normal((n, 64)).astype(F32)
    X /= np.linalg.norm(X, axis=1, keepdims=True)
    X *= (2.0 ** rng.uniform(-4, 4, n)).astype(F32)[:, None]                  # norms x1/16 .. x16
    sub = rng.random((n, 64)) < 0.25                                           # fp16 subnormals: |x| < 2^-14
    X[sub] = (rng.uniform(-1, 1, int(sub.sum())) * 2.0 ** rng.integers(-30, -13, int(sub.sum()))).astype(F32)
    return X


def test_bound_adversarial_rows():
    rng = np.random.default_rng(5)
    for scale_q, scale_t in ((1, 1), (1 / 16, 16), (16, 1 / 16), (1, 1 / 4)):
        Q = adversarial_rows(rng, 300) * F32(scale_q)
        T = adversarial_rows(rng, 400) * F32(scale_t)
        T[:50] = T[50:100]                                                     # exact duplicates among the train rows ...
        Q[:40] = T[:40] * F32(scale_q / scale_t)                               # ... and query rows on top of train rows
        Q[40:60] = T[40:60] + F32(2.0 ** -20) * T[60:80]                       # within fp16's rounding of a train row
        err, eps = check_bound(Q, T)
        assert (err > 0).any()


def test_bound_tiny_rows():
    """Rows entirely in fp16's subnormal range (b = fp16(x - a) underflows to 0): the bound is on |x - a|, not on |b|."""
    rng = np.random.default_rng(6)
    Q = (rng.standard_normal((200, 64)) * 2.0 ** -18).astype(F32)
    T = (rng.standard_normal((300, 64)) * 2.0 ** -18).astype(F32)
    assert (f16(Q - f16(Q)) == 0).mean() > 0.5
    check_bound(Q, T)


def top2(v):
    """indices and values of the two smallest entries of every row."""
    i = np.argpartition(v, 1, axis=1)[:, :2]
    vv = np.take_along_axis(v, i, 1)
    o = np.argsort(vv, axis=1, kind="stable")
    return np.take_along_axis(i, o, 1), np.take_along_axis(vv, o, 1)


def classify(Q, T, ratio):
    """-> (class per row as finalize sees it after win_classify, exact verdict, exact nearest column, fast nearest column)."""
    exact, fast = half_d2(Q, T)
    e = np.array([win_fast_eps(x, frame_norm(Q), frame_norm(T)) for x in row_eps(Q)], F32)
    fi, fv = top2(fast)
    ei, ev = top2(exact)
    cls = win_ratio_class(fv[:, 0], fv[:, 1], e, ratio * ratio)
    exact_pass = ev[:, 0] < ratio * ratio * ev[:, 1]
    return cls, exact_pass, ei[:, 0], fi[:, 0]


def test_classification_sound_and_no_fallback_on_bench_like_frames():
    frames = synth.surf_like(4, 8000, seed=4)
    flagged = 0
    for a, b in ((0, 1), (2, 3), (1, 2)):
        cls, exact_pass, e_best, f_best = classify(frames[a], frames[b], 0.8)
        assert (exact_pass[cls == 1]).all() and not (exact_pass[cls == 0]).any()
        assert (e_best[cls == 1] == f_best[cls == 1]).all()                  # the best slice holds the nearest column
        assert (cls == 1).sum() > 1000                                          # real matches exist
        flagged += int((cls == 2).sum())
    assert flagged == 0


def test_classification_flags_near_ties():
    """Query rows nearly equidistant from two train rows at the ratio boundary, or exact duplicates: the fast values cannot settle
    them, so they are flagged (and settled correctly wherever they are not)."""
    rng = np.random.default_rng(8)
    T = rng.standard_normal((500, 64)).astype(F32)
    T /= np.linalg.norm(T, axis=1, keepdims=True)
    Q = rng.standard_normal((300, 64)).astype(F32)
    Q /= np.linalg.norm(Q, axis=1, keepdims=True)
    for k in range(100):                          # q between t1 and t2 with d1 / d2 = 0.8 +- 1e-4
        t1, t2 = T[2 * k], T[2 * k + 1]
        s = 0.8 * (1 + rng.uniform(-1e-4, 1e-4))
        w = s / (1 + s)
        Q[k] = (1 - w) * t1 + w * t2
    Q[100:120] = T[300:320]
    T[320:340] = T[300:320]                       # duplicated train rows: ties at d = 0
    cls, exact_pass, e_best, f_best = classify(Q, T, 0.8)
    assert (exact_pass[cls == 1]).all() and not (exact_pass[cls == 0]).any()
    assert (e_best[cls == 1] == f_best[cls == 1]).all()
    assert (cls[:100] == 2).sum() > 50 and (cls[100:120] == 2).all()
