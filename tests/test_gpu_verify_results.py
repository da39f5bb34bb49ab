"""GPU: esfm_two_view_results / esfm_multi_two_view_results -- a whole match batch verified on the device (Results.verify).

The scenes are multi-view: landmarks with 3-D positions and 256-bit descriptors seen by frames with their own poses and cameras; key points
are projections plus 0.5 px noise next to distractors, descriptors the landmark's with ~8 % of the bits flipped.  Matching the bank on the
GPU gives real match batches whose indices name the key points.  esfm_two_view_batch is pinned against the oracle
(tests/test_gpu_two_view_batch.py), so byte equality with it, pair by pair, is the parity check here."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from easysfm_b200 import capi
from two_view_util import project, random_K, rodrigues

CHUNK = 4096
SEED = 0xC0FFEE
RATIO = 0.8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def multiview_scene(n_frames, n_landmarks, seed, visible=0.6, distractors=60, flip_p=0.08):
    """-> (key points float32[n_f, 2] per frame, descriptors uint8[n_f, 32] per frame, K [n_frames, 3, 3])."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.uniform(-4, 4, n_landmarks), rng.uniform(-3, 3, n_landmarks), rng.uniform(8, 16, n_landmarks)]
    world = rng.integers(0, 256, (n_landmarks, 32), dtype=np.uint8)
    kps, descs, Ks = [], [], []
    for _ in range(n_frames):
        K = random_K(rng)
        R = rodrigues(rng.normal(0, 0.08, 3))
        c = rng.uniform(-1.5, 1.5, 3)
        seen = np.flatnonzero(rng.random(n_landmarks) < visible)
        xy = project(K, (X[seen] - c) @ R.T) + 0.5 * rng.standard_normal((len(seen), 2))
        d = world[seen] ^ np.packbits(rng.random((len(seen), 256)) < flip_p, axis=1)
        nd = int(distractors)
        xy = np.r_[xy, np.c_[rng.uniform(0, 800, nd), rng.uniform(0, 600, nd)]]
        d = np.r_[d, rng.integers(0, 256, (nd, 32), dtype=np.uint8)]
        order = rng.permutation(len(xy))
        kps.append(np.ascontiguousarray(xy[order], np.float32))
        descs.append(np.ascontiguousarray(d[order]))
        Ks.append(K)
    return kps, descs, np.stack(Ks)


def pairs_of(n):
    return [(i, j) for i in range(n) for j in range(i)]


def batch_reference(ctx, kps, Ks, i, j, m, random_rate=20, seed=SEED):
    """esfm_two_view_batch on host-gathered points of pair (i, j) alone, keyed (i << 32) | j: (inlier records, result record)."""
    mask, r = ctx.two_view_batch(np.array([0, len(m)], np.int64), kps[i][m["queryIdx"]], kps[j][m["trainIdx"]], Ks[i], 1.0, 0.99, max_iters=1000,
                                 seed=seed, first_pair=(i << 32) | j, random_rate=random_rate)
    return m[mask.astype(bool)], r[0]


def per_pair(res, tv):
    """{(query, train): (inlier bytes, result bytes)} of a verified batch (first occurrence of a pair)."""
    out = {}
    for k in range(res.n_pairs):
        q, t, m = res.pair_at(k)
        out.setdefault((q, t), (m.tobytes(), tv[k].tobytes()))
    return out


@pytest.fixture(scope="module")
def vctx():
    """Verification does not depend on the matching engine: one context for the module."""
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def small(vctx):
    kps, descs, Ks = multiview_scene(8, 500, seed=3)
    res = vctx.bank_from_frames(descs).match_all_pairs(RATIO)
    inl, tv = res.verify(vctx, kps, Ks, seed=SEED)
    return dict(kps=kps, descs=descs, Ks=Ks, res=res, inl=inl, tv=tv)


@pytest.fixture(scope="module")
def big(vctx):
    """92 frames: 4186 pairs in loop order, across the 4096-pair chunk edge."""
    kps, descs, Ks = multiview_scene(92, 240, seed=11, visible=0.5, distractors=30)
    bank = vctx.bank_from_frames(descs)
    res = bank.match_all_pairs(RATIO)
    assert res.n_pairs == 4186
    inl, tv = res.verify(vctx, kps, Ks, seed=SEED)
    return dict(kps=kps, Ks=Ks, bank=bank, res=res, inl=inl, tv=tv, ref=per_pair(inl, tv))


# 1. every pair equals esfm_two_view_batch on host-gathered points with the frame-id key -------------------------------------------------
@pytest.mark.gpu
def test_equals_batch_call_pair_by_pair(vctx, small):
    kps, Ks, res, inl, tv = small["kps"], small["Ks"], small["res"], small["inl"], small["tv"]
    assert inl.n_pairs == res.n_pairs == 28 and len(tv) == 28
    n_ok = 0
    for k in range(res.n_pairs):
        i, j, m = res.pair_at(k)
        qi, tj, got = inl.pair_at(k)
        assert (qi, tj) == (i, j)
        assert tv[k]["n_matches"] == len(m)
        if len(m) <= 20:
            assert tv[k]["ok"] == 0 and tv[k]["iters"] == 0 and len(got) == 0, k
            continue
        want, r = batch_reference(vctx, kps, Ks, i, j, m)
        assert got.tobytes() == want.tobytes(), k
        assert tv[k].tobytes() == r.tobytes(), k
        assert tv[k]["n_inliers"] == len(got)
        n_ok += int(tv[k]["ok"])
    assert n_ok >= 20
    assert inl.params() == res.params()
    assert np.array_equal(inl.frame_rows(), res.frame_rows())


@pytest.mark.gpu
def test_equals_batch_call_at_the_chunk_edge(vctx, big):
    kps, Ks, res, inl, tv = big["kps"], big["Ks"], big["res"], big["inl"], big["tv"]
    for k in [0, 1, CHUNK - 2, CHUNK - 1, CHUNK, CHUNK + 1, res.n_pairs - 1] + list(range(1000, 4000, 311)):
        i, j, m = res.pair_at(k)
        if len(m) <= 20:
            assert tv[k]["ok"] == 0 and tv[k]["iters"] == 0 and inl.pair_at(k)[2].size == 0
            continue
        want, r = batch_reference(vctx, kps, Ks, i, j, m)
        assert inl.pair_at(k)[2].tobytes() == want.tobytes(), k
        assert tv[k].tobytes() == r.tobytes(), k
    assert int(tv["ok"].sum()) > res.n_pairs // 2
    assert inl.n_matches == int(tv["n_inliers"].sum())


# 2. order, duplicates, splits and chunk position do not change a pair's bytes --------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("how", ["shuffled", "duplicated", "split", "tail_alone", "reversed"])
def test_order_and_chunk_independence(vctx, big, how):
    rng = np.random.default_rng(7)
    allp = pairs_of(92)
    if how == "shuffled":
        lists = [[allp[k] for k in rng.permutation(len(allp))]]
    elif how == "duplicated":
        extra = [allp[k] for k in rng.choice(len(allp), 300, replace=False)]
        lists = [allp[:2000] + extra + allp[2000:]]
    elif how == "split":
        lists = [allp[:1500], allp[1500:]]
    elif how == "tail_alone":
        lists = [allp[CHUNK - 10:]]               # the second chunk's pairs in chunk 0
    else:
        lists = [allp[::-1]]
    for pl in lists:
        res = big["bank"].match_pairs(pl, RATIO)
        inl, tv = res.verify(vctx, big["kps"], big["Ks"], seed=SEED)
        assert inl.n_pairs == len(pl)
        for k in range(inl.n_pairs):
            q, t, m = inl.pair_at(k)
            assert (q, t) == tuple(pl[k])
            assert (m.tobytes(), tv[k].tobytes()) == big["ref"][(q, t)], (how, k)


# 3. min_pair_matches edges, on a hand-built match file -----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def edge_file(small, tmp_path_factory):
    """Pairs cut to 0, 4, 5, 20 and 21 of their own matches, and one whole pair, in a version-2 match file."""
    res, descs = small["res"], small["descs"]
    cuts = [((1, 0), 0), ((2, 0), 4), ((2, 1), 5), ((3, 0), 20), ((3, 1), 21), ((4, 0), None)]
    pairs, per = [], []
    for (i, j), n in cuts:
        m = res.pair(i, j)
        assert len(m) > 21, (i, j, len(m))
        pairs.append((i, j))
        per.append(m if n is None else m[:n])
    path = str(tmp_path_factory.mktemp("edges") / "edges.matches")
    capi.write_match_file(path, pairs, per, capi.KIND_B256, RATIO, False, frame_rows=[len(d) for d in descs])
    return path, pairs, per


@pytest.mark.gpu
@pytest.mark.parametrize("threshold", [20, 0, -1])
def test_min_pair_matches_edges(vctx, small, edge_file, threshold):
    path, pairs, per = edge_file
    loaded = capi.load_results(path)
    inl, tv = loaded.verify(vctx, small["kps"], small["Ks"], min_pair_matches=threshold, seed=SEED)
    for k, ((i, j), m) in enumerate(zip(pairs, per)):
        got = inl.pair_at(k)[2]
        assert tv[k]["n_matches"] == len(m)
        if len(m) <= max(threshold, 4):
            assert tv[k]["ok"] == 0 and tv[k]["iters"] == 0 and tv[k]["n_inliers"] == 0 and len(got) == 0, (threshold, k)
            assert not tv[k]["E"].any()
        else:
            want, r = batch_reference(vctx, small["kps"], small["Ks"], i, j, m)
            assert got.tobytes() == want.tobytes() and tv[k].tobytes() == r.tobytes(), (threshold, k)
            assert tv[k]["iters"] > 0


# 4. tracks: the reference's loop sfm.cpp:163-217 ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_tracks_from_verified_batch(small):
    import oracle
    kps, res, inl = small["kps"], small["res"], small["inl"]
    rows = [len(k) for k in kps]
    t = capi.Tracks(rows)
    t.build(inl, min_pair_matches=0)
    feed = [inl.pair_at(k)[2] if len(res.pair_at(k)[2]) > 20 else np.zeros(0, capi.DMATCH_DTYPE) for k in range(res.n_pairs)]
    ids_ref, has_ref, _, npts = oracle.tracks_build(rows, feed)
    assert t.counts() == (len(rows), npts)
    for f in range(len(rows)):
        ids, has = t.frame(f)
        assert np.array_equal(ids, ids_ref[f]) and np.array_equal(has, has_ref[f])


# 5. persistence -----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_verified_batch_save_load_and_loaded_input(vctx, small, tmp_path):
    inl, tv, res = small["inl"], small["tv"], small["res"]
    p = str(tmp_path / "inliers.matches")
    inl.save(p)
    back = capi.load_results(p)
    assert back.n_pairs == inl.n_pairs and back.n_matches == inl.n_matches
    assert np.array_equal(back.pair_counts(), inl.pair_counts())
    assert back.all_matches()[0].tobytes() == inl.all_matches()[0].tobytes()
    assert np.array_equal(back.frame_rows(), res.frame_rows())
    back.validate([len(k) for k in small["kps"]])
    q = str(tmp_path / "matches.matches")
    res.save(q)
    inl2, tv2 = capi.load_results(q).verify(vctx, small["kps"], small["Ks"], seed=SEED)
    assert tv2.tobytes() == tv.tobytes()
    assert inl2.all_matches()[0].tobytes() == inl.all_matches()[0].tobytes()


# 6. refusals, before any output -------------------------------------------------------------------------------------------------------------
def raw_verify(lib, ctx_h, res_h, kps, K, first_pair=0, null=None):
    """The C call with every argument explicit; `null` names one argument to pass as NULL.  -> (rc, message, inliers handle, out)."""
    kp_off = np.zeros(len(kps) + 1, np.int64)
    kp_off[1:] = np.cumsum([len(k) for k in kps])
    xy = np.concatenate(kps + [np.zeros((1, 2), np.float32)]).astype(np.float32)
    K = np.ascontiguousarray(K, np.float64)
    prm = capi.TwoViewParams()
    lib.esfm_two_view_default_params(ctypes.byref(prm))
    prm.first_pair = first_pair
    n = capi.c_int64()
    lib.esfm_results_counts(res_h, ctypes.byref(n), None)
    out = np.zeros(max(n.value, 1), capi.TWO_VIEW_DTYPE)
    h = capi.c_void_p(12345)
    args = dict(ctx=ctx_h, matches=res_h, kp_off=kp_off.ctypes.data, kp_xy=xy.ctypes.data, K=K.ctypes.data, params=ctypes.byref(prm),
                inliers=ctypes.byref(h), out=out.ctypes.data)
    if null:
        args[null] = None
    rc = lib.esfm_two_view_results(args["ctx"], args["matches"], len(kps), args["kp_off"], args["kp_xy"], args["K"], int(K.ndim == 3),
                                   args["params"], 20, args["inliers"], args["out"])
    return rc, lib.esfm_last_error().decode(), h.value, out


@pytest.mark.gpu
def test_refuses_digest_and_device_resident_batches(vctx, small):
    bank = vctx.bank_from_frames(small["descs"])
    for res in (bank.match_pairs(pairs_of(8), RATIO, keep=capi.KEEP_DIGESTS), bank.match_pairs(pairs_of(8), RATIO, device_resident=True)):
        with pytest.raises(capi.EsfmError) as e:
            res.verify(vctx, small["kps"], small["Ks"])
        assert e.value.code == 3
        rc, _, h, out = raw_verify(capi.load_library(), vctx._h, res._h, small["kps"], small["Ks"])
        assert rc == 3 and h is None and not out.view(np.uint8).any()


@pytest.mark.gpu
def test_refuses_bad_input(vctx, small, tmp_path):
    lib = capi.load_library()
    kps, Ks, res = small["kps"], small["Ks"], small["res"]
    # one out-of-range trainIdx in one pair of many, in a file (no stored frame rows: the device check is what catches it)
    per = [res.pair_at(k)[2].copy() for k in range(res.n_pairs)]
    bad_k = 17
    q, t = res.pair_at(bad_k)[:2]
    per[bad_k]["trainIdx"][len(per[bad_k]) // 2] = len(kps[t])
    path = str(tmp_path / "bad.matches")
    capi.write_match_file(path, pairs_of(8), per, capi.KIND_B256, RATIO, False)
    loaded = capi.load_results(path)
    rc, msg, h, out = raw_verify(lib, vctx._h, loaded._h, kps, Ks)
    assert rc == 1 and f"pair {bad_k} = ({q},{t})" in msg and h is None and not out.view(np.uint8).any(), msg
    # key-point counts different from the stored frame rows
    short = [k[:-1] if f == 3 else k for f, k in enumerate(kps)]
    rc, msg, h, out = raw_verify(lib, vctx._h, res._h, short, Ks)
    assert rc == 1 and "frame 3" in msg and h is None and not out.view(np.uint8).any(), msg
    # a nonzero first_pair
    rc, msg, h, out = raw_verify(lib, vctx._h, res._h, kps, Ks, first_pair=5)
    assert rc == 1 and "first_pair" in msg and h is None and not out.view(np.uint8).any()
    # NULL arguments
    for null in ("ctx", "matches", "kp_off", "kp_xy", "K", "params", "inliers", "out"):
        rc, msg, h, out = raw_verify(lib, vctx._h, res._h, kps, Ks, null=null)
        assert rc == 1, null
        assert not out.view(np.uint8).any() or null == "out", null
        assert h is None or null == "inliers", null
    # too few frames for the batch's pairs
    with pytest.raises(capi.EsfmError) as e:
        res.verify(vctx, kps[:5], Ks[:5])
    assert e.value.code == 1


# 7. several devices -------------------------------------------------------------------------------------------------------------------------
def _multi_equals_single(devices, big):
    with capi.MultiContext(devices) as multi:
        inl, tv = big["res"].verify(multi, big["kps"], big["Ks"], seed=SEED)
        assert tv.tobytes() == big["tv"].tobytes()
        assert inl.all_matches()[0].tobytes() == big["inl"].all_matches()[0].tobytes()
        assert np.array_equal(inl.pair_counts(), big["inl"].pair_counts())
        assert np.array_equal(inl.digests(), big["inl"].digests())


@pytest.mark.gpu
def test_multi_device_listed_twice_equals_one_device(big):
    _multi_equals_single([0, 0], big)


@pytest.mark.gpu
def test_multi_two_devices_equal_one_device(big):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _multi_equals_single(2, big)


# 8. the C++ drop-in: esfm_prepare_all_pairs -> esfm_verify_all_pairs -> the reference's loop over estimate2D2D_E5P_RANSAC --------------------
def build_verify_shim(tmp):
    exe = os.path.join(tmp, "verify_main")
    libdir = os.path.join(ROOT, "easysfm_b200", "lib")
    shim = os.path.join(ROOT, "easysfm_b200", "shim")
    cmd = ["g++", "-std=c++14", "-O1", "-Wall", "-I", os.path.join(ROOT, "tests", "shim"), "-I", os.path.join(ROOT, "include"),
           os.path.join(shim, "feature_matching_gpu.cpp"), os.path.join(shim, "estimate_motion_gpu.cpp"), os.path.join(ROOT, "tests", "shim", "verify_main.cpp"),
           "-L", libdir, "-lesfm_match", f"-Wl,-rpath,{libdir}", "-o", exe]
    subprocess.check_call(cmd)
    return exe


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", ["1", "2"])
def test_verify_shim_lookups_equal_per_call(tmp_path, gpus):
    """After esfm_verify_all_pairs every estimate2D2D_E5P_RANSAC call with a pair's batch matches is a lookup whose inliers and T equal the
    per-call answer; with a match dropped the call is computed and equals its own per-call answer.  ESFM_GPUS=2 verifies on two GPUs."""
    if gpus == "2":
        import torch
        if torch.cuda.device_count() < 2:
            pytest.skip("needs 2 GPUs")
    kps, descs, Ks = multiview_scene(7, 400, seed=21)
    exe = build_verify_shim(str(tmp_path))
    inp = os.path.join(str(tmp_path), "in.bin")
    with open(inp, "wb") as f:
        f.write(np.int32(len(kps)).tobytes())
        for K, k, d in zip(Ks, kps, descs):
            f.write(np.ascontiguousarray(K, np.float64).tobytes())
            f.write(np.int32(len(k)).tobytes())
            f.write(k.tobytes())
            f.write(d.tobytes())
    out = os.path.join(str(tmp_path), "out.bin")
    run = subprocess.run([exe, inp, out], stdout=subprocess.PIPE, env=dict(os.environ, ESFM_GPUS=gpus), check=True)
    rec = np.frombuffer(open(out, "rb").read(), np.int32).reshape(-1, 5)
    assert len(rec) >= 15 and (rec[:, 2] > 20).all()
    assert (rec[:, 3] == 1).all(), rec
    assert (rec[:, 4] == 1).all(), rec
    assert run.stdout.decode().count("(verified batch)") == len(rec)


def test_verify_shim_compiles_and_links(tmp_path):
    assert os.path.exists(build_verify_shim(str(tmp_path)))
