"""Generates the committed golden fixtures by running the REFERENCE's matcher calls (cv2.BFMatcher, exactly as
python_code/feature_match.py:24-39 and cpp_code/src/feature_matching.cpp:74-92 issue them) in the build container.

    python tests/golden/make_golden.py            # needs cv2 4.13.0; reads /root/reference/test_data for the fountain set

Outputs (all small, all committed):
  kat_cases.npz       hand-built known-answer cases: ties, duplicates, rows < 2, ragged sizes, d = 0, ratio edge (F5)
  synth_surf.npz      4 SURF-like frames (seeded), cv2 matches for ratio {0.5, 0.8} x cross_check {0, 1}, all 6 pairs
  synth_orb.npz       4 ORB-like frames (seeded), same grid
  fountain_orb.npz    BASELINE configs[0] stand-in: ORB_create(8000) descriptors of the 11 bundled fountain images
                      (SURF is not in this image's OpenCV, SURVEY.md F9) + cv2 matches of all 55 pairs, cross_check 0/1;
                      about 2 MB, so stored as fountain_orb.part<k>.npz (save_parts) and loaded as one by golden_util.load
The fixtures store descriptors AND expected matches, so the tests need neither cv2 nor /root/reference.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from easysfm_b200 import synth  # noqa: E402
from oracle import cv2_oracle  # noqa: E402


def pack_matches(m):
    return np.stack([m["queryIdx"], m["trainIdx"]], axis=1).astype(np.int32), m["distance"].astype(np.float32)


def all_pairs_expected(frames, ratios, out, prefix):
    n = len(frames)
    for ratio in ratios:
        for cc in (0, 1):
            for i in range(n):
                for j in range(i):
                    m = cv2_oracle.match(frames[i], frames[j], ratio, bool(cc))
                    ij, d = pack_matches(m)
                    out[f"{prefix}_r{int(ratio * 100)}_c{cc}_{i}_{j}_idx"] = ij
                    out[f"{prefix}_r{int(ratio * 100)}_c{cc}_{i}_{j}_dist"] = d


PART_BYTES = 900_000


def save_parts(stem, arrays):
    """Writes `arrays` as stem.part0.npz, stem.part1.npz, ... (compressed, in insertion order), each holding at most PART_BYTES of
    array data so every committed file stays under 1 MB; tests/golden_util.load(stem + ".npz") merges them back."""
    parts, size = [{}], 0
    for k, a in arrays.items():
        if parts[-1] and size + a.nbytes > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = a
        size += a.nbytes
    for n, p in enumerate(parts):
        np.savez_compressed(f"{stem}.part{n}.npz", **p)


def kat_cases():
    rng = np.random.default_rng(1234)
    cases = {}
    # 1. query equal to three identical train rows (SURVEY A1), float
    T = rng.standard_normal((9, 64)).astype(np.float32)
    T /= np.linalg.norm(T, axis=1, keepdims=True)
    T[4] = T[1]; T[5] = T[1]
    Q = np.stack([T[1], T[7], T[2] * 0.999])
    cases["f32_triple_dup"] = (Q.astype(np.float32), T)
    # 2. Hamming duplicate train rows, second neighbour must be the LOWER index
    Tb = rng.integers(0, 256, (40, 32), dtype=np.uint8)
    Tb[3] = Tb[0]; Tb[17] = Tb[0]
    Qb = Tb[[3, 9, 17]].copy(); Qb[0, 0] ^= 0x80; Qb[1, 5] ^= 0x01
    cases["b256_dup_rows"] = (Qb, Tb)
    # 3. ratio edge case evaluated in double (F5): d1 = 44, d2 = 55, 0.8 * 55 == 44
    T3 = np.zeros((2, 32), np.uint8); Q3 = np.zeros((1, 32), np.uint8)
    T3[0, :5] = 0xFF; T3[0, 5] = 0x0F; T3[1, :6] = 0xFF; T3[1, 6] = 0x7F
    cases["b256_ratio_edge"] = (Q3, T3)
    # 4. rows < 2 on the train side, and a single query row
    cases["f32_train_one_row"] = (synth.surf_like(1, 7, seed=5)[0], synth.surf_like(1, 1, seed=6)[0])
    cases["b256_one_query"] = (synth.orb_like(1, 1, seed=7)[0], synth.orb_like(1, 33, seed=8)[0])
    # 5. ragged, non-multiple-of-tile sizes
    cases["f32_ragged"] = tuple(synth.surf_like(2, [129, 257], seed=9))
    cases["b256_ragged"] = tuple(synth.orb_like(2, [255, 1025], seed=10))
    # 6. duplicate queries (cross-check keeps only the lower index), A2
    Q6, T6 = synth.surf_like(2, [40, 60], seed=11)
    Q6[9] = Q6[4]; Q6[4] = T6[12]; Q6[9] = T6[12]
    cases["f32_dup_queries"] = (Q6, T6)
    out = {}
    for name, (Q, T) in cases.items():
        out[f"{name}_Q"] = Q
        out[f"{name}_T"] = T
        for ratio in (0.5, 0.8):
            for cc in (0, 1):
                ij, d = pack_matches(cv2_oracle.match(Q, T, ratio, bool(cc)))
                out[f"{name}_r{int(ratio * 100)}_c{cc}_idx"] = ij
                out[f"{name}_r{int(ratio * 100)}_c{cc}_dist"] = d
        idx, dist = cv2_oracle.knn2(Q, T)
        out[f"{name}_knn_idx"] = idx
        out[f"{name}_knn_dist"] = dist
        ij, d = pack_matches(cv2_oracle.mutual_nn(Q, T))
        out[f"{name}_mutual_idx"] = ij
        out[f"{name}_mutual_dist"] = d
    out["names"] = np.array(sorted(cases.keys()))
    return out


def main():
    import cv2
    print("cv2", cv2.__version__)
    np.savez_compressed(os.path.join(HERE, "kat_cases.npz"), **kat_cases())

    for kind, gen, rows in (("surf", synth.surf_like, [300, 257, 128, 411]), ("orb", synth.orb_like, [500, 256, 333, 1025])):
        frames = gen(len(rows), rows, seed=21)
        out = {f"frame_{i}": f for i, f in enumerate(frames)}
        all_pairs_expected(frames, (0.5, 0.8), out, "m")
        np.savez_compressed(os.path.join(HERE, f"synth_{kind}.npz"), **out)

    data_dir = "/root/reference/test_data"
    names = [l.strip() for l in open(os.path.join(data_dir, "image_list.txt")) if l.strip()]
    orb = cv2.ORB_create(8000)   # cpp_code/src/feature_matching.cpp:16-22 with max_num = 8000
    frames = []
    for n in names:
        img = cv2.imread(os.path.join(data_dir, "images_25", os.path.basename(n)))
        if img is None:
            img = cv2.imread(os.path.join(data_dir, n))
        gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
        _, desc = orb.detectAndCompute(gray, None)
        frames.append(np.ascontiguousarray(desc))
    out = {f"frame_{i}": f for i, f in enumerate(frames)}
    all_pairs_expected(frames, (0.8,), out, "m")
    save_parts(os.path.join(HERE, "fountain_orb"), out)
    print("fountain frames:", [f.shape[0] for f in frames])
    for f in os.listdir(HERE):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
