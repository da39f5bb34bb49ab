"""Verification of a whole match batch on the device (esfm_two_view_results / esfm_multi_two_view_results), measured.

1. One GPU, 2048 pairs x 2000 matches (0.5 px noise, 30 % gross outliers: the shape of DESIGN 5.6).  The pairs are (Q, j) for j < 2048 -- one
   query frame against 2048 others -- so that the host recipe of INTEGRATION 7 (gather on the host -> esfm_two_view_batch -> compact on the
   host) can key every pair by its frame ids in ONE call (first_pair = Q << 32) and its output can be compared byte for byte with
   esfm_two_view_results on the same batch.  Both paths start from the same loaded results batch and end with the inlier records on the host.
2. Several GPUs: esfm_multi_two_view_results on a 200-frame all-pairs batch (19,900 pairs, 2000 matches each) at N = 1, 2, 4, 8 devices:
   wall time, slowest / fastest device, and the digest of the verified batch.  N larger than the box's GPU count runs with device 0 listed N
   times (the digest check only: such a run says nothing about scaling) and is marked so.

usage: python tools/verify_bench.py [--out FILE] [--reps R]; prints the JSON and writes it to FILE.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from easysfm_b200 import capi                      # noqa: E402
from two_view_util import project, random_K, rodrigues   # noqa: E402

N_MATCH = 2000
OUTLIERS = 0.3
NOISE = 0.5


def frames(n_frames, seed):
    """n_frames views of N_MATCH landmarks by one camera (the reference's setting: a pair is verified with one K), every landmark seen by every
    frame: key points (shuffled), where landmark k sits in each frame, K."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.uniform(-4, 4, N_MATCH), rng.uniform(-3, 3, N_MATCH), rng.uniform(8, 16, N_MATCH)]
    K = random_K(rng)
    kps, pos = [], []
    for _ in range(n_frames):
        R = rodrigues(rng.normal(0, 0.08, 3))
        c = rng.uniform(-1.5, 1.5, 3)
        xy = project(K, (X - c) @ R.T) + NOISE * rng.standard_normal((N_MATCH, 2))
        order = rng.permutation(N_MATCH)
        kps.append(np.ascontiguousarray(xy[order], np.float32))
        p = np.empty(N_MATCH, np.int64)
        p[order] = np.arange(N_MATCH)
        pos.append(p)
    return kps, pos, K, rng


def match_records(pos_q, pos_t, rng):
    """Ground-truth correspondences with OUTLIERS of them given a random trainIdx, in ascending queryIdx (as the matcher returns them)."""
    m = np.zeros(N_MATCH, capi.DMATCH_DTYPE)
    m["queryIdx"], m["trainIdx"] = pos_q, pos_t
    bad = rng.random(N_MATCH) < OUTLIERS
    m["trainIdx"][bad] = rng.integers(0, N_MATCH, int(bad.sum()))
    m["distance"] = rng.uniform(10, 60, N_MATCH).astype(np.float32)
    return m[np.argsort(m["queryIdx"], kind="stable")]


def loaded_batch(tmp, name, pairs, per, rows):
    path = os.path.join(tmp, name)
    capi.write_match_file(path, pairs, per, capi.KIND_B256, 0.8, False, frame_rows=rows)
    return capi.load_results(path)


def timed(fn, reps):
    fn()                                            # warm-up: module load, pool allocations
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), [round(t, 4) for t in ts], out


def verified_digest(inl, tv):
    return hashlib.sha1(inl.digests().tobytes() + tv.tobytes()).hexdigest()


def single_gpu(tmp, reps):
    n_pairs = 2048
    kps, pos, K, rng = frames(n_pairs + 1, seed=1)
    Q = n_pairs
    pairs = [(Q, j) for j in range(n_pairs)]
    per = [match_records(pos[Q], pos[j], rng) for j in range(n_pairs)]
    res = loaded_batch(tmp, "single.matches", pairs, per, [len(k) for k in kps])
    ctx = capi.Context(0)
    kp_off = np.concatenate([[0], np.cumsum([len(k) for k in kps])])
    xy = np.concatenate(kps)

    def recipe():
        m, off = res.all_matches()
        q_frame = np.repeat(np.array([p[0] for p in pairs]), np.diff(off))
        t_frame = np.repeat(np.array([p[1] for p in pairs]), np.diff(off))
        p1 = xy[kp_off[q_frame] + m["queryIdx"]]
        p2 = xy[kp_off[t_frame] + m["trainIdx"]]
        mask, tv = ctx.two_view_batch(off, p1, p2, K, 1.0, 0.99, max_iters=1000, seed=0, first_pair=Q << 32, random_rate=20)
        keep = mask.astype(bool)
        return [m[off[k]:off[k + 1]][keep[off[k]:off[k + 1]]] for k in range(n_pairs)], tv

    def device():
        inl, tv = res.verify(ctx, kps, K, seed=0)
        return inl, tv

    t_recipe, ts_recipe, (inl_r, tv_r) = timed(recipe, reps)
    t_dev, ts_dev, (inl_d, tv_d) = timed(device, reps)
    equal = tv_r.tobytes() == tv_d.tobytes() and all(inl_r[k].tobytes() == inl_d.pair_at(k)[2].tobytes() for k in range(n_pairs))
    out = dict(pairs=n_pairs, matches_per_pair=N_MATCH, noise_px=NOISE, outliers=OUTLIERS, shape="query frame Q against frames 0..2047",
               recipe_s=round(t_recipe, 4), recipe_runs_s=ts_recipe, recipe_pairs_per_s=round(n_pairs / t_recipe),
               results_s=round(t_dev, 4), results_runs_s=ts_dev, results_pairs_per_s=round(n_pairs / t_dev),
               byte_equal=bool(equal), ok_pairs=int(tv_d["ok"].sum()), inliers_mean=float(tv_d["n_inliers"].mean()),
               hypotheses_mean=float(tv_d["iters"].mean()), digest=verified_digest(inl_d, tv_d))
    ctx.close()
    return out


def multi_gpu(tmp, reps, n_list):
    import torch
    n_gpus = torch.cuda.device_count()
    n_frames = 200
    kps, pos, K, rng = frames(n_frames, seed=2)
    pairs = [(i, j) for i in range(n_frames) for j in range(i)]
    per = [match_records(pos[i], pos[j], rng) for i, j in pairs]
    res = loaded_batch(tmp, "multi.matches", pairs, per, [len(k) for k in kps])
    del per
    rows = []
    for n in n_list:
        devices = list(range(n)) if n <= n_gpus else [0] * n
        with capi.MultiContext(devices) as multi:
            def run():
                inl, tv = res.verify(multi, kps, K, seed=0)
                return inl, tv, multi.timing()
            t, ts, (inl, tv, tm) = timed(run, reps)
            rows.append(dict(N=n, devices=devices, distinct_gpus=n <= n_gpus, wall_s=round(t, 4), runs_s=ts,
                             device_ms_max=round(tm["device_ms_max"], 2), device_ms_min=round(tm["device_ms_min"], 2),
                             work_imbalance=round(tm["work_imbalance"], 4), pairs_per_s=round(len(pairs) / t),
                             digest=verified_digest(inl, tv), inliers_mean=float(tv["n_inliers"].mean()),
                             hypotheses_mean=float(tv["iters"].mean())))
    return dict(frames=n_frames, pairs=len(pairs), matches_per_pair=N_MATCH, gpus_on_box=n_gpus, runs=rows,
                digests_equal=len({r["digest"] for r in rows}) == 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--n", default="1,2,4,8")
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    with tempfile.TemporaryDirectory() as tmp:
        single = single_gpu(tmp, a.reps)
        multi = multi_gpu(tmp, a.reps, [int(x) for x in a.n.split(",")])
    out = dict(gpus=smi.splitlines(), single_gpu=single, multi_gpu=multi,
               timing="host clock around calls that end in a device synchronise; median of the runs after one warm-up run")
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
