"""Synthetic two-view scenes for the geometric-verification tests (known pose, pixel noise, gross outliers) and the host build of the
product's float64 math (easysfm_b200/csrc/two_view_math.cuh compiled with g++: tests/host/two_view_host.cpp)."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def rodrigues(r):
    r = np.asarray(r, np.float64)
    th = np.linalg.norm(r)
    if th < 1e-15:
        return np.eye(3)
    k = r / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx


def scene(n, noise=0.0, outliers=0.0, seed=0, K=None):
    """n matches between two views of a random point cloud: returns (K, pts1, pts2 float32 pixels, R, t unit)."""
    rng = np.random.default_rng(seed)
    if K is None:
        K = np.array([[800.0, 0, 384], [0, 820.0, 256], [0, 0, 1]])
    X = np.c_[rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(4, 9, n)]
    R = rodrigues(rng.normal(0, 0.12, 3))
    t = rng.normal(0, 1, 3)
    t /= np.linalg.norm(t)
    x1 = (K @ X.T).T
    x1 = x1[:, :2] / x1[:, 2:]
    X2 = X @ R.T + t
    x2 = (K @ X2.T).T
    x2 = x2[:, :2] / x2[:, 2:]
    x1 = x1 + noise * rng.standard_normal(x1.shape)
    x2 = x2 + noise * rng.standard_normal(x2.shape)
    no = int(outliers * n)
    x2[:no] = np.c_[rng.uniform(0, 768, no), rng.uniform(0, 512, no)]
    return K, x1.astype(np.float32), x2.astype(np.float32), R, t


def random_K(rng):
    """A pinhole camera with fx in [400, 1600], fy = fx * (1 +- 2..10 %) and a principal point that moves around the image centre."""
    fx = rng.uniform(400.0, 1600.0)
    fy = fx * (1.0 + rng.choice([-1.0, 1.0]) * rng.uniform(0.02, 0.1))
    return np.array([[fx, 0.0, rng.uniform(250.0, 550.0)], [0.0, fy, rng.uniform(180.0, 380.0)], [0.0, 0.0, 1.0]])


def project(K, X):
    x = X @ K.T
    return x[:, :2] / x[:, 2:]


DEGENERATE = ("planar", "collinear", "rotation", "baseline", "far", "repeated", "identical", "same")


def degenerate_scene(kind, n, noise=0.0, seed=0, K=None):
    """Two views of a configuration on which the essential matrix is ill-posed or not unique.  Returns (K, pts1, pts2 float32 pixels, R, t,
    X): X holds the 3-D point of every match in camera 1 (noise-free); pts1 ~ K X, pts2 ~ K (R X + t) plus `noise` px.
      planar      points on the plane z = 6 + 0.4 x - 0.3 y
      collinear   points on one 3-D line
      rotation    pure rotation, t = 0
      baseline    |t| = 1e-6
      far         the cloud of `scene` with every coordinate times 1e4 (depth 4e4 .. 9e4), unit baseline
      repeated    n distinct correspondences, each repeated 2 or 3 times, in shuffled order (noise drawn once per distinct one)
      identical   one correspondence n times
      same        pts2 == pts1 (R = I, t = 0; noise drawn once)"""
    assert kind in DEGENERATE, kind
    rng = np.random.default_rng(seed)
    if K is None:
        K = np.array([[800.0, 0, 384], [0, 820.0, 256], [0, 0, 1]])
    X = np.c_[rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(4, 9, n)]
    R = rodrigues(rng.normal(0, 0.12, 3))
    t = rng.normal(0, 1, 3)
    t /= np.linalg.norm(t)
    if kind == "planar":
        X[:, 2] = 6.0 + 0.4 * X[:, 0] - 0.3 * X[:, 1]
    elif kind == "collinear":
        X = np.array([-1.5, -1.0, 5.0]) + rng.uniform(0, 1, (n, 1)) * np.array([3.0, 2.0, 3.0])
    elif kind == "rotation":
        t = np.zeros(3)
    elif kind == "baseline":
        t = t * 1e-6
    elif kind == "far":
        X = X * 1e4
    elif kind == "identical":
        X = np.repeat(X[:1], n, axis=0)
    elif kind == "same":
        R, t = np.eye(3), np.zeros(3)
    x1 = project(K, X) + noise * rng.standard_normal((n, 2))
    x2 = x1.copy() if kind == "same" else project(K, X @ R.T + t) + noise * rng.standard_normal((n, 2))
    if kind == "identical":
        x1[:], x2[:] = x1[0], x2[0]
    if kind == "repeated":
        idx = rng.permutation(np.repeat(np.arange(n), rng.integers(2, 4, n)))
        x1, x2, X = x1[idx], x2[idx], X[idx]
    return K, x1.astype(np.float32), x2.astype(np.float32), R, t, X


def rot_angle_deg(A, B):
    return float(np.degrees(np.arccos(np.clip((np.trace(A.T @ B) - 1) / 2, -1, 1))))


def dir_angle_deg(a, b):
    a, b = np.ravel(a), np.ravel(b)
    return float(np.degrees(np.arccos(np.clip(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)), -1, 1))))


_lib = None


def host_lib():
    """tests/host/two_view_host.cpp -> tests/_build/libtvhost.so (g++), loaded once."""
    global _lib
    if _lib is None:
        out = os.path.join(HERE, "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libtvhost.so")
        src = os.path.join(HERE, "host", "two_view_host.cpp")
        hdr = os.path.join(HERE, "..", "easysfm_b200", "csrc", "two_view_math.cuh")
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src])
        _lib = ctypes.CDLL(so)
        _lib.tvh_five_point.restype = ctypes.c_int
        _lib.tvh_sampson.restype = ctypes.c_double
        _lib.tvh_update_iters.restype = ctypes.c_int
        _lib.tvh_cheirality.restype = ctypes.c_int
    return _lib


def dptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
