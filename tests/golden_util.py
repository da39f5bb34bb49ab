import os

import numpy as np

from oracle import DMATCH_DTYPE

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class _Arrays(dict):
    @property
    def files(self):
        return list(self)


def load(name):
    """A fixture by name; one that make_golden.save_parts split into name.part<k>.npz comes back as the merged arrays."""
    path = os.path.join(GOLDEN, name)
    if os.path.exists(path):
        return np.load(path)
    stem = path[: -len(".npz")]
    out = _Arrays()
    k = 0
    while os.path.exists(f"{stem}.part{k}.npz"):
        with np.load(f"{stem}.part{k}.npz") as z:
            out.update((f, z[f]) for f in z.files)
        k += 1
    if not out:
        raise FileNotFoundError(path)
    return out


def as_matches(idx, dist):
    out = np.zeros(len(idx), DMATCH_DTYPE)
    if len(idx):
        out["queryIdx"] = idx[:, 0]
        out["trainIdx"] = idx[:, 1]
        out["distance"] = dist
    return out


def frames_of(z):
    n = len([k for k in z.files if k.startswith("frame_")])
    return [z[f"frame_{i}"] for i in range(n)]
