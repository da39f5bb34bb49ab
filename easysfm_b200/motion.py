"""Python mirror of the reference's MotionEstimator for the two-view step (cpp_code/include/estimate_motion.h:17-20, :33-34;
cpp_code/src/estimate_motion.cpp:27-97, :234-283), on the GPU through esfm_two_view_batch.  Same names and argument meaning as the reference;
the batch form serves the all-pairs loop of cpp_code/test/sfm.cpp:140-166 in one call.  For a match batch (capi.Results) the same step runs
without gathering on the host: Results.verify returns the inlier matches as a new batch plus a pose per pair, keyed like this class's per-pair
calls when pair_id = (frame_1 << 32) | frame_2."""
from __future__ import annotations

import numpy as np

from .capi import Context, DMATCH_DTYPE


class MotionEstimator:
    def __init__(self, ctx: Context, seed: int = 0):
        self.ctx = ctx
        self.seed = seed

    def estimate2D2D_E5P_RANSAC(self, keypoints_1, keypoints_2, matches, K, ransac_thre: float = 1.0, ransac_prob: float = 0.99, pair_id: int = 0):
        """keypoints_*: float32[n, 2] pixel coordinates (frame_t::keypoints[k].pt); matches: DMATCH array (queryIdx into keypoints_1, trainIdx into
        keypoints_2).  Returns (ok, inlier_matches, T) with T the 4 x 4 float32 transform [R t; 0 1] of estimate_motion.cpp:72-82."""
        ok, inl, T, _ = self.estimate_pairs([(keypoints_1, keypoints_2, matches)], K, ransac_thre, ransac_prob, first_pair=pair_id)[0]
        return ok, inl, T

    def estimate_pairs(self, items, K, ransac_thre: float = 1.0, ransac_prob: float = 0.99, first_pair: int = 0, random_rate: int = 1):
        """items: sequence of (keypoints_1, keypoints_2, matches).  One esfm_two_view_batch call; returns per pair
        (ok, inlier_matches, T float32 4 x 4, relative_depth) -- what estimate2D2D_E5P_RANSAC + getDepthFast give at sfm.cpp:165-166."""
        off = [0]
        p1, p2 = [], []
        for kp1, kp2, m in items:
            m = np.asarray(m, DMATCH_DTYPE)
            p1.append(np.asarray(kp1, np.float32).reshape(-1, 2)[m["queryIdx"]])
            p2.append(np.asarray(kp2, np.float32).reshape(-1, 2)[m["trainIdx"]])
            off.append(off[-1] + len(m))
        cat = lambda xs: np.concatenate(xs) if xs else np.zeros((0, 2), np.float32)
        mask, res = self.ctx.two_view_batch(np.asarray(off, np.int64), cat(p1), cat(p2), K, ransac_thre, ransac_prob, seed=self.seed,
                                            first_pair=first_pair, random_rate=random_rate)
        out = []
        for k, (kp1, kp2, m) in enumerate(items):
            m = np.asarray(m, DMATCH_DTYPE)
            T = np.eye(4, dtype=np.float32)
            T[:3, :3] = res[k]["R"]
            T[:3, 3] = res[k]["t"]
            out.append((bool(res[k]["ok"]), m[mask[off[k]:off[k + 1]].astype(bool)], T, float(res[k]["depth"])))
        return out
