"""Latency of the UNMODIFIED caller's shape (sfm.cpp:153,156: one matchFeaturesX call per image pair = esfm_match_descriptors):
config 1, the 11 bundled fountain images as ORB(8000) descriptors (tests/golden/fountain_orb.part*.npz), 55 pairs in loop order, against
one esfm_match_all_pairs over the same frames.  usage: python tools/per_pair_latency.py  -> one JSON line"""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import easysfm_b200 as esfm
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from golden_util import load, frames_of

frames = frames_of(load("fountain_orb.npz"))
ctx = esfm.Context(0)
pairs = [(i, j) for i in range(len(frames)) for j in range(i)]
out = {}
for name, fr, ratio in (("orb", frames, 0.8),):
    for rep in range(3):
        lat = []
        for (i, j) in pairs:
            t0 = time.perf_counter()
            m = ctx.match_descriptors(fr[i], fr[j], ratio, False)
            lat.append(time.perf_counter() - t0)
    t0 = time.perf_counter()
    bank = ctx.bank_from_frames(fr)
    res = bank.match_all_pairs(ratio, False)
    t_all = time.perf_counter() - t0
    out[name] = {"pairs": len(pairs), "rows": [int(f.shape[0]) for f in fr], "per_call_ms_median": 1e3 * float(np.median(lat)), "per_call_ms_max": 1e3 * float(np.max(lat)),
                 "per_call_total_ms": 1e3 * float(np.sum(lat)), "all_pairs_one_call_ms": 1e3 * t_all, "matches": int(res.n_matches)}
print(json.dumps(out))
