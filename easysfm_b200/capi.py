"""ctypes binding of include/esfm_match.h (libesfm_match.so).

Thin by design: every function maps 1:1 onto a C entry point; numpy arrays are passed as raw
pointers + sizes.  Loading fails loudly if the library has not been built -- there is no fallback.
"""
from __future__ import annotations

import ctypes
import os
import weakref
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

KIND_F32X64 = 0
KIND_B256 = 1

DMATCH_DTYPE = np.dtype([("queryIdx", "<i4"), ("trainIdx", "<i4"), ("imgIdx", "<i4"), ("distance", "<f4")])
PAIR_DTYPE = np.dtype([("query", "<i4"), ("train", "<i4")])


L2_ENGINE_FFMA = 0
L2_ENGINE_TC = 1
L2_ENGINE_TC16 = 2
HAMMING_ENGINE_POPC = 0
HAMMING_ENGINE_TC = 1
HAMMING_ENGINE_TC16 = 2
KEEP_MATCHES = 0
KEEP_DIGESTS = 1


class EsfmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"esfm error {code}: {msg}")
        self.code = code


class Stats(ctypes.Structure):
    _fields_ = [
        ("kernel_launches", c_uint64),
        ("h2d_bytes", c_uint64),
        ("d2h_bytes", c_uint64),
        ("comparisons", c_uint64),
        ("pairs", c_uint64),
        ("last_sweep_ms", c_double),
        ("last_finalize_ms", c_double),
        ("sweep_ms_total", c_double),
        ("sweep_launches", c_uint64),
        ("fallback_rows", c_uint64),
        ("verified_rows", c_uint64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class MultiTiming(ctypes.Structure):
    _fields_ = [
        ("broadcast_ms", c_double),
        ("commit_ms", c_double),
        ("match_ms", c_double),
        ("device_ms_max", c_double),
        ("device_ms_min", c_double),
        ("work_imbalance", c_double),
        ("used_nccl", c_int),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class TwoViewParams(ctypes.Structure):
    _fields_ = [("ransac_thre", c_double), ("ransac_prob", c_double), ("cheirality_dist", c_double), ("seed", c_uint64), ("first_pair", c_uint64),
                ("max_iters", c_int32), ("random_rate", c_int32)]


class TwoView(ctypes.Structure):
    _fields_ = [("E", c_double * 9), ("R", c_double * 9), ("t", c_double * 3), ("depth", c_double), ("n_matches", c_int32), ("n_inliers", c_int32),
                ("n_good", c_int32), ("iters", c_int32), ("ok", c_int32), ("reserved", c_int32)]


TWO_VIEW_DTYPE = np.dtype([("E", "<f8", (3, 3)), ("R", "<f8", (3, 3)), ("t", "<f8", (3,)), ("depth", "<f8"), ("n_matches", "<i4"), ("n_inliers", "<i4"),
                           ("n_good", "<i4"), ("iters", "<i4"), ("ok", "<i4"), ("reserved", "<i4")])
assert TWO_VIEW_DTYPE.itemsize == ctypes.sizeof(TwoView)

# esfm_keypoint_t: the cv::KeyPoint fields the reference reads (class_id is always -1)
KEYPOINT_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"), ("octave", "<i4")])
ERR_CAPACITY = 5

# name -> (restype, argtypes); kept in one table so tests can check it against the header.
SIGNATURES = {
    "esfm_abi_version": (c_int, []),
    "esfm_last_error": (c_char_p, []),
    "esfm_init": (c_int, [c_int, c_void_p, POINTER(c_void_p)]),
    "esfm_destroy": (c_int, [c_void_p]),
    "esfm_synchronize": (c_int, [c_void_p]),
    "esfm_get_stats": (c_int, [c_void_p, POINTER(Stats)]),
    "esfm_set_profiling": (c_int, [c_void_p, c_int]),
    "esfm_device_sm_count": (c_int, [c_void_p, POINTER(c_int)]),
    "esfm_set_l2_engine": (c_int, [c_void_p, c_int]),
    "esfm_get_l2_engine": (c_int, [c_void_p, POINTER(c_int)]),
    "esfm_set_hamming_engine": (c_int, [c_void_p, c_int]),
    "esfm_get_hamming_engine": (c_int, [c_void_p, POINTER(c_int)]),
    "esfm_bank_create": (c_int, [c_void_p, c_int, c_int, POINTER(c_void_p)]),
    "esfm_bank_set_frame": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_size_t]),
    "esfm_bank_set_frame_pinned": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_size_t]),
    "esfm_bank_set_frame_rows": (c_int, [c_void_p, c_int, c_int]),
    "esfm_bank_commit": (c_int, [c_void_p]),
    "esfm_bank_alloc_device": (c_int, [c_void_p]),
    "esfm_bank_device_rows": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_size_t)]),
    "esfm_bank_commit_device": (c_int, [c_void_p]),
    "esfm_bank_n_frames": (c_int, [c_void_p, POINTER(c_int)]),
    "esfm_bank_frame_rows": (c_int, [c_void_p, c_int, POINTER(c_int)]),
    "esfm_bank_device_bytes": (c_int, [c_void_p, POINTER(c_size_t)]),
    "esfm_bank_destroy": (c_int, [c_void_p]),
    "esfm_match_all_pairs": (c_int, [c_void_p, c_double, c_int, POINTER(c_void_p)]),
    "esfm_match_pairs": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_int, POINTER(c_void_p)]),
    "esfm_match_pairs_device": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_int, POINTER(c_void_p)]),
    "esfm_results_fetch": (c_int, [c_void_p]),
    "esfm_bank_chunk_pairs": (c_int, [c_void_p, POINTER(c_int64)]),
    "esfm_match_pair": (c_int, [c_void_p, c_int, c_int, c_double, c_int, c_void_p, c_int, POINTER(c_int)]),
    "esfm_match_descriptors": (c_int, [c_void_p, c_int, c_void_p, c_int, c_size_t, c_void_p, c_int, c_size_t, c_int,
                                       c_double, c_int, c_void_p, c_int, POINTER(c_int)]),
    "esfm_knn2_pair": (c_int, [c_void_p, c_int, c_int, POINTER(c_int32), POINTER(c_float)]),
    "esfm_results_counts": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64)]),
    "esfm_results_pair_at": (c_int, [c_void_p, c_int64, POINTER(c_int), POINTER(c_int), POINTER(c_void_p), POINTER(c_int)]),
    "esfm_results_pair": (c_int, [c_void_p, c_int, c_int, POINTER(c_void_p), POINTER(c_int)]),
    "esfm_results_pair_counts": (c_int, [c_void_p, POINTER(c_int32)]),
    "esfm_results_destroy": (c_int, [c_void_p]),
    "esfm_results_save": (c_int, [c_void_p, c_char_p]),
    "esfm_results_load": (c_int, [c_char_p, POINTER(c_void_p)]),
    "esfm_results_params": (c_int, [c_void_p, POINTER(c_int), POINTER(ctypes.c_double), POINTER(c_int)]),
    "esfm_results_frame_rows": (c_int, [c_void_p, POINTER(c_int32), c_int, POINTER(c_int)]),
    "esfm_results_validate": (c_int, [c_void_p, c_int, POINTER(c_int32)]),
    "esfm_match_pairs_keep": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_int, c_int, POINTER(c_void_p)]),
    "esfm_results_copy_all": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_int64)]),
    "esfm_results_digests": (c_int, [c_void_p, POINTER(c_uint64)]),
    "esfm_results_segment_count": (c_int, [c_void_p, POINTER(c_int)]),
    "esfm_two_view_default_params": (c_int, [POINTER(TwoViewParams)]),
    "esfm_two_view_batch": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, POINTER(TwoViewParams), c_void_p, c_void_p]),
    "esfm_two_view_depth": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, POINTER(c_double), POINTER(c_int32)]),
    "esfm_two_view_results": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, POINTER(TwoViewParams), c_int, POINTER(c_void_p),
                                      c_void_p]),
    "esfm_multi_two_view_results": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, POINTER(TwoViewParams), c_int,
                                            POINTER(c_void_p), c_void_p]),
    "esfm_orb_extract": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_size_t, c_int, c_void_p, c_void_p, c_int, POINTER(c_int)]),
    "esfm_bank_set_frame_from_image": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_size_t, c_int, c_void_p, c_void_p, c_int, POINTER(c_int)]),
    "esfm_orb_last_timing": (c_int, [c_void_p, POINTER(c_double), POINTER(c_int)]),
    "esfm_orb_debug_level": (c_int, [c_void_p, c_int, c_int, c_void_p, c_size_t, POINTER(c_int), POINTER(c_int)]),
    "esfm_results_segment_at": (c_int, [c_void_p, c_int, POINTER(c_void_p), POINTER(c_int64)]),
    "esfm_results_pair_layout": (c_int, [c_void_p, POINTER(c_int32), POINTER(c_int64)]),
    "esfm_results_device_matches": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_int64)]),
    "esfm_results_device_layout": (c_int, [c_void_p, POINTER(c_int64)]),
    "esfm_tracks_create": (c_int, [c_int, POINTER(c_int32), POINTER(c_void_p)]),
    "esfm_tracks_destroy": (c_int, [c_void_p]),
    "esfm_tracks_add_pair": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int]),
    "esfm_tracks_finish_frame": (c_int, [c_void_p, c_int]),
    "esfm_tracks_build": (c_int, [c_void_p, c_void_p, c_int]),
    "esfm_tracks_frame": (c_int, [c_void_p, c_int, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int)]),
    "esfm_tracks_counts": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int64)]),
    "esfm_tracks_pair_scores": (c_int, [c_void_p, c_void_p, POINTER(c_int64), POINTER(c_double)]),
    "esfm_tracks_find_init_pair": (c_int, [c_void_p, c_void_p, POINTER(c_double), c_int, c_double, POINTER(c_int), POINTER(c_int),
                                           POINTER(c_double), POINTER(c_int64), POINTER(c_int)]),
    "esfm_tracks_find_next_frame": (c_int, [c_void_p, ctypes.POINTER(ctypes.c_uint8), POINTER(c_int32), c_int64, POINTER(c_int), POINTER(c_int)]),
    "esfm_multi_init": (c_int, [c_int, POINTER(c_int), POINTER(c_void_p)]),
    "esfm_multi_destroy": (c_int, [c_void_p]),
    "esfm_multi_device_count": (c_int, [c_void_p, POINTER(c_int)]),
    "esfm_multi_ctx": (c_int, [c_void_p, c_int, POINTER(c_void_p)]),
    "esfm_multi_timing": (c_int, [c_void_p, POINTER(MultiTiming)]),
    "esfm_multi_bank_create": (c_int, [c_void_p, c_int, c_int, POINTER(c_void_p)]),
    "esfm_multi_bank_set_frame": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_size_t]),
    "esfm_multi_bank_primary": (c_int, [c_void_p, POINTER(c_void_p)]),
    "esfm_multi_bank_commit": (c_int, [c_void_p]),
    "esfm_multi_bank_destroy": (c_int, [c_void_p]),
    "esfm_multi_match_all_pairs": (c_int, [c_void_p, c_double, c_int, c_int, POINTER(c_void_p)]),
    "esfm_multi_match_pairs": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_int, c_int, POINTER(c_void_p)]),
}

_LIB = None


def library_path() -> str:
    # ESFM_LIBRARY lets kernel experiments load an alternative build of the SAME C ABI (never a CPU path)
    return os.environ.get("ESFM_LIBRARY") or os.path.join(_HERE, "lib", "libesfm_match.so")


def load_library():
    """dlopen libesfm_match.so; raises if it was not built (python __graft_entry__.py build, or make -C easysfm_b200/csrc)."""
    global _LIB
    if _LIB is None:
        path = library_path()
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"{path} is missing: build it with `make -C easysfm_b200/csrc` (nvcc, sm_100a). "
                "easysfm_b200 has no CPU fallback.")
        lib = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = lib
    return _LIB


def _check(rc: int):
    if rc != 0:
        msg = load_library().esfm_last_error()
        raise EsfmError(rc, msg.decode("utf-8", "replace") if msg else "")


def _as_image(image):
    img = np.asarray(image)
    if img.dtype != np.uint8 or img.ndim not in (2, 3) or (img.ndim == 3 and img.shape[2] not in (1, 3)):
        raise TypeError("image must be uint8 [rows, cols] (gray) or [rows, cols, 3] (BGR)")
    ch = 1 if img.ndim == 2 else img.shape[2]
    if img.strides[-1] != 1 or (img.ndim == 3 and img.strides[1] != ch):
        img = np.ascontiguousarray(img)
    return img, img.shape[0], img.shape[1], ch


def _as_desc(arr, kind=None):
    arr = np.asarray(arr)
    if arr.ndim != 2:
        raise ValueError("descriptor matrix must be 2-D (rows x cols)")
    if arr.dtype == np.float32:
        k = KIND_F32X64
    elif arr.dtype == np.uint8:
        k = KIND_B256
    else:
        raise TypeError(f"descriptors must be float32 (SURF) or uint8 (ORB), got {arr.dtype}")
    if kind is not None and k != kind:
        raise TypeError("descriptor dtype does not match the bank kind")
    if arr.shape[0] and arr.strides[1] != arr.itemsize:
        arr = np.ascontiguousarray(arr)
    return arr, k


class Context:
    """One CUDA device + stream (esfm_ctx_t)."""

    def __init__(self, device: int = 0, stream: int | None = None, _borrowed=None):
        self._lib = load_library()
        self._owned = _borrowed is None
        if _borrowed is None:
            h = c_void_p()
            _check(self._lib.esfm_init(int(device), c_void_p(stream) if stream else None, ctypes.byref(h)))
        else:
            h = _borrowed            # a per-device context of a MultiContext: destroyed by esfm_multi_destroy
        self._h = h
        self.device = int(device)
        # banks and result batches borrow the context's stream, scratch and pinned pool: they must go first
        self._children = weakref.WeakSet()

    def close(self):
        if getattr(self, "_h", None):
            for child in list(getattr(self, "_children", ())):
                child.close()
            if self._owned:
                self._lib.esfm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def synchronize(self):
        _check(self._lib.esfm_synchronize(self._h))

    def stats(self) -> dict:
        s = Stats()
        _check(self._lib.esfm_get_stats(self._h, ctypes.byref(s)))
        return s.as_dict()

    def set_profiling(self, on: bool):
        _check(self._lib.esfm_set_profiling(self._h, int(bool(on))))

    @property
    def sm_count(self) -> int:
        n = c_int()
        _check(self._lib.esfm_device_sm_count(self._h, ctypes.byref(n)))
        return n.value

    def set_l2_engine(self, engine):
        """'ffma' (exact-FP32 FMA pipe), 'tc' (3xTF32 on the tcgen05 tensor cores) or 'tc16' (two-term FP16 split, slice keys) for the SURF / L2 sweep."""
        code = {"ffma": L2_ENGINE_FFMA, "tc": L2_ENGINE_TC, "tc16": L2_ENGINE_TC16}.get(engine, engine)
        _check(self._lib.esfm_set_l2_engine(self._h, int(code)))

    def l2_engine(self) -> str:
        e = c_int(0)
        _check(self._lib.esfm_get_l2_engine(self._h, ctypes.byref(e)))
        return {L2_ENGINE_FFMA: "ffma", L2_ENGINE_TC: "tc", L2_ENGINE_TC16: "tc16"}[e.value]

    def set_hamming_engine(self, engine):
        """'popc' (XOR + POPC on the integer pipes), 'tc' (exact FP8 dot product on the tensor cores, packed keys) or 'tc16' (FP8 dot product
        with FP16 accumulators, packed-half epilogue, slice keys) for the ORB sweep."""
        code = {"popc": HAMMING_ENGINE_POPC, "tc": HAMMING_ENGINE_TC, "tc16": HAMMING_ENGINE_TC16}.get(engine, engine)
        _check(self._lib.esfm_set_hamming_engine(self._h, int(code)))

    def hamming_engine(self) -> str:
        e = c_int(0)
        _check(self._lib.esfm_get_hamming_engine(self._h, ctypes.byref(e)))
        return {HAMMING_ENGINE_POPC: "popc", HAMMING_ENGINE_TC: "tc", HAMMING_ENGINE_TC16: "tc16"}[e.value]

    def bank(self, kind: int, n_frames: int) -> "Bank":
        return Bank(self, kind, n_frames)

    def two_view_batch(self, pair_off, pts1, pts2, K, ransac_thre=1.0, ransac_prob=0.99, max_iters=1000, seed=0, first_pair=0, random_rate=1,
                       cheirality_dist=50.0):
        """esfm_two_view_batch: the reference's estimate2D2D_E5P_RANSAC + getDepthFast for a batch of image pairs.
        pair_off: int64[n_pairs + 1]; pts1 / pts2: float32[total, 2] matched pixel coordinates (query / train keypoints of every match, all
        pairs back to back); K: 3 x 3 (one camera) or n_pairs x 3 x 3.  Returns (inlier mask uint8[total], per-pair structured array)."""
        pair_off = np.ascontiguousarray(pair_off, np.int64)
        n_pairs = len(pair_off) - 1
        pts1 = np.ascontiguousarray(pts1, np.float32).reshape(-1, 2)
        pts2 = np.ascontiguousarray(pts2, np.float32).reshape(-1, 2)
        K = np.ascontiguousarray(K, np.float64)
        k_per_pair = 1 if K.ndim == 3 else 0
        if k_per_pair and K.shape[0] != n_pairs:
            raise ValueError("K must be 3 x 3 or n_pairs x 3 x 3")
        total = int(pair_off[-1]) if n_pairs >= 0 and len(pair_off) else 0
        if len(pts1) != total or len(pts2) != total:
            raise ValueError("pts1 / pts2 must have pair_off[-1] rows")
        prm = TwoViewParams()
        _check(self._lib.esfm_two_view_default_params(ctypes.byref(prm)))
        prm.ransac_thre, prm.ransac_prob, prm.cheirality_dist = float(ransac_thre), float(ransac_prob), float(cheirality_dist)
        prm.seed, prm.first_pair, prm.max_iters, prm.random_rate = int(seed), int(first_pair), int(max_iters), int(random_rate)
        mask = np.zeros(max(total, 1), np.uint8)
        out = np.zeros(max(n_pairs, 1), TWO_VIEW_DTYPE)
        _check(self._lib.esfm_two_view_batch(self._h, n_pairs, pair_off.ctypes.data, pts1.ctypes.data, pts2.ctypes.data, K.ctypes.data, k_per_pair,
                                             ctypes.byref(prm), mask.ctypes.data, out.ctypes.data))
        return mask[:total], out[:n_pairs]

    def two_view_depth(self, pts1, pts2, K, R, t, random_rate=20, return_used=False):
        """esfm_two_view_depth: MotionEstimator::getDepthFast for one pair (every random_rate-th match, [I|0] and [R|t]).  Returns the mean
        depth, or (mean depth, number of matches triangulated) with return_used=True."""
        pts1 = np.ascontiguousarray(pts1, np.float32).reshape(-1, 2)
        pts2 = np.ascontiguousarray(pts2, np.float32).reshape(-1, 2)
        K, R, t = (np.ascontiguousarray(a, np.float64) for a in (K, R, t))
        depth, used = c_double(0.0), c_int32(0)
        _check(self._lib.esfm_two_view_depth(self._h, len(pts1), pts1.ctypes.data, pts2.ctypes.data, K.ctypes.data, R.ctypes.data, t.ctypes.data,
                                             int(random_rate), ctypes.byref(depth), ctypes.byref(used)))
        return (depth.value, used.value) if return_used else depth.value

    def orb_extract(self, image, max_features: int = 5000, want_descriptors: bool = True):
        """esfm_orb_extract: FeatureMatching::detectFeaturesORB (feature_matching.cpp:14-41) for one image -- uint8 [rows, cols] (gray) or
        [rows, cols, 3] (BGR).  Returns (key points as KEYPOINT_DTYPE records in cv2's order, uint8 [n, 32] descriptors)."""
        img, rows, cols, ch = _as_image(image)
        cap = int(max_features) + 256
        while True:
            kps = np.zeros(cap, KEYPOINT_DTYPE)
            desc = np.zeros((cap, 32), np.uint8) if want_descriptors else None
            n = c_int(0)
            rc = self._lib.esfm_orb_extract(self._h, img.ctypes.data, rows, cols, ch, img.strides[0], int(max_features), kps.ctypes.data,
                                            desc.ctypes.data if want_descriptors else None, cap, ctypes.byref(n))
            if rc == ERR_CAPACITY and n.value > cap:
                cap = n.value
                continue
            _check(rc)
            return kps[:n.value].copy(), (desc[:n.value].copy() if want_descriptors else None)

    def orb_last_timing(self) -> dict:
        """Host wall-clock phases of the last orb_extract / set_frame_from_image on this context (esfm_orb_last_timing)."""
        ms, corners = (c_double * 5)(), c_int(0)
        _check(self._lib.esfm_orb_last_timing(self._h, ms, ctypes.byref(corners)))
        return {"front_end_ms": ms[0], "corner_records_ms": ms[1], "host_selection_ms": ms[2], "descriptors_ms": ms[3], "total_ms": ms[4],
                "corners": corners.value}

    def orb_debug_level(self, level: int, blurred: bool = False) -> np.ndarray:
        """Pyramid level of the last orb_extract call on this context, as resized or after the 7 x 7 blur (tests)."""
        r, c = c_int(0), c_int(0)
        _check(self._lib.esfm_orb_debug_level(self._h, int(level), int(blurred), None, 0, ctypes.byref(r), ctypes.byref(c)))
        out = np.zeros((r.value, c.value), np.uint8)
        _check(self._lib.esfm_orb_debug_level(self._h, int(level), int(blurred), out.ctypes.data, out.nbytes, ctypes.byref(r), ctypes.byref(c)))
        return out

    def bank_from_frames(self, frames) -> "Bank":
        """frames: sequence of 2-D numpy arrays (all float32 x64 or all uint8 x32)."""
        frames = list(frames)
        if not frames:
            raise ValueError("no frames")
        _, kind = _as_desc(frames[0])
        b = Bank(self, kind, len(frames))
        for i, f in enumerate(frames):
            b.set_frame(i, f)
        b.commit()
        return b

    def match_descriptors(self, query, train, ratio: float, cross_check: bool = False) -> np.ndarray:
        """Two host matrices in, matches out (esfm_match_descriptors)."""
        q, kind = _as_desc(query)
        t, _ = _as_desc(train, kind)
        cols = q.shape[1] if q.shape[0] else (t.shape[1] if t.shape[0] else (64 if kind == KIND_F32X64 else 32))
        out = np.zeros(max(q.shape[0], 1), DMATCH_DTYPE)
        n = c_int(0)
        _check(self._lib.esfm_match_descriptors(
            self._h, kind, q.ctypes.data, q.shape[0], q.strides[0] if q.shape[0] else 0,
            t.ctypes.data, t.shape[0], t.strides[0] if t.shape[0] else 0, cols, float(ratio), int(bool(cross_check)),
            out.ctypes.data, out.shape[0], ctypes.byref(n)))
        return out[: n.value].copy()


class Bank:
    """Device-resident descriptor bank (esfm_bank_t)."""

    def __init__(self, ctx: Context, kind: int, n_frames: int, _borrowed=None):
        self._lib = ctx._lib
        self.ctx = ctx
        self.kind = int(kind)
        self._owned = _borrowed is None
        if _borrowed is None:
            h = c_void_p()
            _check(self._lib.esfm_bank_create(ctx._h, int(kind), int(n_frames), ctypes.byref(h)))
        else:
            h = _borrowed            # the primary replica of a MultiBank: destroyed by esfm_multi_bank_destroy
        self._h = h
        self.n_frames = int(n_frames)
        ctx._children.add(self)

    def close(self):
        if getattr(self, "_h", None):
            if self._owned:
                self._lib.esfm_bank_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_frame(self, frame_id: int, desc):
        a, _ = _as_desc(desc, self.kind)
        _check(self._lib.esfm_bank_set_frame(self._h, int(frame_id), a.ctypes.data, a.shape[0], a.shape[1],
                                             a.strides[0] if a.shape[0] else a.shape[1] * a.itemsize))

    def set_frame_from_image(self, frame_id: int, image, max_features: int = 5000, want_descriptors: bool = False):
        """esfm_bank_set_frame_from_image: ORB-extract `image` on the device and make the descriptors frame `frame_id` of this (B256) bank
        without a round trip through the host.  Returns the key points (and the descriptors when asked for)."""
        img, rows, cols, ch = _as_image(image)
        cap = int(max_features) + 256
        while True:
            kps = np.zeros(cap, KEYPOINT_DTYPE)
            desc = np.zeros((cap, 32), np.uint8) if want_descriptors else None
            n = c_int(0)
            rc = self._lib.esfm_bank_set_frame_from_image(self._h, int(frame_id), img.ctypes.data, rows, cols, ch, img.strides[0], int(max_features),
                                                          kps.ctypes.data, desc.ctypes.data if want_descriptors else None, cap, ctypes.byref(n))
            if rc == ERR_CAPACITY and n.value > cap:
                cap = n.value
                continue
            _check(rc)
            return (kps[:n.value].copy(), desc[:n.value].copy()) if want_descriptors else kps[:n.value].copy()

    def set_frame_pinned(self, frame_id: int, desc):
        """No host-side copy: `desc` must be a C-contiguous array in page-locked memory (e.g. a view of a torch
        pin_memory tensor) and must stay alive and unmodified until commit() returns."""
        a = np.asarray(desc)
        b, _ = _as_desc(a, self.kind)
        if b is not a or (a.shape[0] and not a.flags.c_contiguous):
            raise ValueError("set_frame_pinned needs a C-contiguous array (no implicit copy)")
        self._pinned_refs = getattr(self, "_pinned_refs", [])
        self._pinned_refs.append(a)
        _check(self._lib.esfm_bank_set_frame_pinned(self._h, int(frame_id), a.ctypes.data, a.shape[0], a.shape[1],
                                                    a.shape[1] * a.itemsize))

    def set_frame_rows(self, frame_id: int, rows: int):
        _check(self._lib.esfm_bank_set_frame_rows(self._h, int(frame_id), int(rows)))

    def commit(self):
        _check(self._lib.esfm_bank_commit(self._h))
        self._pinned_refs = []

    def alloc_device(self):
        _check(self._lib.esfm_bank_alloc_device(self._h))

    def device_rows(self):
        """(device pointer, bytes) of the raw row-major bank, e.g. to wrap as a torch tensor for a broadcast."""
        p, n = c_void_p(), c_size_t()
        _check(self._lib.esfm_bank_device_rows(self._h, ctypes.byref(p), ctypes.byref(n)))
        return p.value, n.value

    def commit_device(self):
        _check(self._lib.esfm_bank_commit_device(self._h))

    def frame_rows(self, frame_id: int) -> int:
        r = c_int()
        _check(self._lib.esfm_bank_frame_rows(self._h, int(frame_id), ctypes.byref(r)))
        return r.value

    def chunk_pairs(self) -> int:
        """Largest batch the library processes as one chunk (a device-resident batch must not exceed it)."""
        n = c_int64()
        _check(self._lib.esfm_bank_chunk_pairs(self._h, ctypes.byref(n)))
        return n.value

    def device_bytes(self) -> int:
        n = c_size_t()
        _check(self._lib.esfm_bank_device_bytes(self._h, ctypes.byref(n)))
        return n.value

    # ---- matching ----
    def match_all_pairs(self, ratio: float, cross_check: bool = False) -> "Results":
        h = c_void_p()
        _check(self._lib.esfm_match_all_pairs(self._h, float(ratio), int(bool(cross_check)), ctypes.byref(h)))
        return Results(self._lib, h, self.ctx)

    def match_pairs(self, pairs, ratio: float, cross_check: bool = False, device_resident: bool = False,
                    keep: int = KEEP_MATCHES) -> "Results":
        p = np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))
        h = c_void_p()
        if device_resident:
            _check(self._lib.esfm_match_pairs_device(self._h, p.ctypes.data, p.shape[0], float(ratio), int(bool(cross_check)), ctypes.byref(h)))
        else:
            _check(self._lib.esfm_match_pairs_keep(self._h, p.ctypes.data, p.shape[0], float(ratio), int(bool(cross_check)), int(keep),
                                                   ctypes.byref(h)))
        return Results(self._lib, h, self.ctx)

    def match_pair(self, query_frame: int, train_frame: int, ratio: float, cross_check: bool = False) -> np.ndarray:
        cap = max(self.frame_rows(query_frame), 1)
        out = np.zeros(cap, DMATCH_DTYPE)
        n = c_int(0)
        _check(self._lib.esfm_match_pair(self._h, int(query_frame), int(train_frame), float(ratio), int(bool(cross_check)),
                                         out.ctypes.data, cap, ctypes.byref(n)))
        return out[: n.value].copy()

    def knn2_pair(self, query_frame: int, train_frame: int):
        fq = self.frame_rows(query_frame)
        idx = np.full((fq, 2), -1, np.int32)
        dist = np.full((fq, 2), np.inf, np.float32)
        _check(self._lib.esfm_knn2_pair(self._h, int(query_frame), int(train_frame),
                                        idx.ctypes.data_as(POINTER(c_int32)), dist.ctypes.data_as(POINTER(c_float))))
        return idx, dist


MATCH_FILE_HEADER = np.dtype([("magic", "S8"), ("version", "<u4"), ("dmatch_bytes", "<u4"), ("n_pairs", "<i8"), ("n_matches", "<i8"),
                              ("kind", "<i4"), ("cross_check", "<i4"), ("ratio", "<f8")])


def load_results(path: str) -> "Results":
    """esfm_results_load: a saved batch back as a Results object; needs no device."""
    lib = load_library()
    h = c_void_p()
    _check(lib.esfm_results_load(os.fsencode(path), ctypes.byref(h)))
    return Results(lib, h)


def write_match_file(path: str, pairs, matches_per_pair, kind: int, ratio: float, cross_check: bool, frame_rows=None):
    """The match-file format written with numpy (tools and tests; the library's writer is esfm_results_save).
    frame_rows given -> version 2 (row counts of the bank's frames stored), else version 1."""
    pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
    counts = np.array([len(m) for m in matches_per_pair], np.int32)
    hdr = np.zeros(1, MATCH_FILE_HEADER)
    hdr["magic"], hdr["version"], hdr["dmatch_bytes"] = b"ESFMMTCH", 1 if frame_rows is None else 2, DMATCH_DTYPE.itemsize
    hdr["n_pairs"], hdr["n_matches"] = len(pairs), int(counts.sum())
    hdr["kind"], hdr["cross_check"], hdr["ratio"] = kind, int(bool(cross_check)), ratio
    with open(path, "wb") as f:
        f.write(hdr.tobytes())
        if frame_rows is not None:
            f.write(np.array([len(frame_rows), 0], np.int32).tobytes())
            f.write(np.asarray(frame_rows, np.int32).tobytes())
        f.write(pairs.tobytes())
        f.write(counts.tobytes())
        for m in matches_per_pair:
            f.write(np.ascontiguousarray(m, dtype=DMATCH_DTYPE).tobytes())


def read_match_file(path: str):
    """-> (header record, pairs [n,2] int32, counts [n] int32, matches [n_matches] DMATCH_DTYPE)."""
    with open(path, "rb") as f:
        hdr = np.frombuffer(f.read(MATCH_FILE_HEADER.itemsize), MATCH_FILE_HEADER)[0]
        if int(hdr["version"]) == 2:
            nf = int(np.frombuffer(f.read(8), np.int32)[0])
            f.read(4 * nf)
        n = int(hdr["n_pairs"])
        pairs = np.frombuffer(f.read(8 * n), np.int32).reshape(n, 2)
        counts = np.frombuffer(f.read(4 * n), np.int32)
        matches = np.frombuffer(f.read(), DMATCH_DTYPE)
    return hdr, pairs, counts, matches


class Results:
    """Host-resident compacted matches of a batch of pairs (esfm_results_t)."""

    def __init__(self, lib, handle, ctx=None):
        self._lib = lib
        self._h = handle
        if ctx is not None:      # (a batch loaded from a match file has no context)
            ctx._children.add(self)
        n_pairs, n_matches = c_int64(), c_int64()
        _check(lib.esfm_results_counts(handle, ctypes.byref(n_pairs), ctypes.byref(n_matches)))
        self.n_pairs = n_pairs.value
        self.n_matches = n_matches.value

    def close(self):
        if getattr(self, "_h", None):
            self._lib.esfm_results_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def fetch(self):
        _check(self._lib.esfm_results_fetch(self._h))

    def pair_counts(self) -> np.ndarray:
        out = np.zeros(self.n_pairs, np.int32)
        if self.n_pairs:
            _check(self._lib.esfm_results_pair_counts(self._h, out.ctypes.data_as(POINTER(c_int32))))
        return out

    def save(self, path: str):
        """Write the (fetched) batch to a match file (include/esfm_match.h: persistence)."""
        _check(self._lib.esfm_results_save(self._h, os.fsencode(path)))

    def frame_rows(self):
        """Row counts of the frames the batch was matched on (empty array: unknown, a version-1 file)."""
        n = c_int()
        _check(self._lib.esfm_results_frame_rows(self._h, None, 0, ctypes.byref(n)))
        rows = np.zeros(n.value, np.int32)
        if n.value:
            _check(self._lib.esfm_results_frame_rows(self._h, rows.ctypes.data_as(POINTER(c_int32)), n.value, ctypes.byref(n)))
        return rows

    def validate(self, frame_rows):
        """Raises EsfmError unless the batch fits frames with these row counts (stored counts, pair ids, every match index)."""
        rows = np.ascontiguousarray(frame_rows, dtype=np.int32)
        _check(self._lib.esfm_results_validate(self._h, len(rows), rows.ctypes.data_as(POINTER(c_int32))))

    def params(self):
        """(kind, ratio, cross_check) the batch was matched with."""
        k, r, c = c_int(), ctypes.c_double(), c_int()
        _check(self._lib.esfm_results_params(self._h, ctypes.byref(k), ctypes.byref(r), ctypes.byref(c)))
        return k.value, r.value, bool(c.value)

    def _view(self, ptr, n):
        if n == 0 or not ptr:
            return np.zeros(0, DMATCH_DTYPE)
        buf = (ctypes.c_char * (n * DMATCH_DTYPE.itemsize)).from_address(ptr)
        return np.frombuffer(buf, dtype=DMATCH_DTYPE, count=n).copy()

    def all_matches(self):
        """Every pair's matches back to back in batch order, in one call: (matches, offsets[n_pairs + 1])."""
        out = np.zeros(max(self.n_matches, 1), DMATCH_DTYPE)
        off = np.zeros(self.n_pairs + 1, np.int64)
        _check(self._lib.esfm_results_copy_all(self._h, out.ctypes.data, self.n_matches, off.ctypes.data_as(POINTER(c_int64))))
        return out[: self.n_matches], off

    def segments(self):
        """Zero-copy views: ([segment arrays], segment index per pair, offset per pair).  The arrays alias library memory and
        are valid until close()."""
        n = c_int()
        _check(self._lib.esfm_results_segment_count(self._h, ctypes.byref(n)))
        segs = []
        for s in range(n.value):
            p, m = c_void_p(), c_int64()
            _check(self._lib.esfm_results_segment_at(self._h, s, ctypes.byref(p), ctypes.byref(m)))
            if m.value == 0 or not p.value:
                segs.append(np.zeros(0, DMATCH_DTYPE))
            else:
                buf = (ctypes.c_char * (m.value * DMATCH_DTYPE.itemsize)).from_address(p.value)
                segs.append(np.frombuffer(buf, dtype=DMATCH_DTYPE, count=m.value))
        seg = np.zeros(self.n_pairs, np.int32)
        off = np.zeros(self.n_pairs, np.int64)
        if self.n_pairs:
            _check(self._lib.esfm_results_pair_layout(self._h, seg.ctypes.data_as(POINTER(c_int32)), off.ctypes.data_as(POINTER(c_int64))))
        return segs, seg, off

    def digests(self) -> np.ndarray:
        """64-bit digest per pair (count, indices and distance bits of its matches, in order)."""
        out = np.zeros(self.n_pairs, np.uint64)
        if self.n_pairs:
            _check(self._lib.esfm_results_digests(self._h, out.ctypes.data_as(POINTER(c_uint64))))
        return out

    def device_matches(self):
        """(device pointer, n_matches, per-pair offsets) of a device-resident batch's match arena."""
        p, n = c_void_p(), c_int64()
        _check(self._lib.esfm_results_device_matches(self._h, ctypes.byref(p), ctypes.byref(n)))
        off = np.zeros(self.n_pairs, np.int64)
        if self.n_pairs:
            _check(self._lib.esfm_results_device_layout(self._h, off.ctypes.data_as(POINTER(c_int64))))
        return p.value, n.value, off

    def pair_at(self, k: int):
        q, t, n, p = c_int(), c_int(), c_int(), c_void_p()
        _check(self._lib.esfm_results_pair_at(self._h, int(k), ctypes.byref(q), ctypes.byref(t), ctypes.byref(p), ctypes.byref(n)))
        return q.value, t.value, self._view(p.value, n.value)

    def pair(self, query_frame: int, train_frame: int) -> np.ndarray:
        n, p = c_int(), c_void_p()
        _check(self._lib.esfm_results_pair(self._h, int(query_frame), int(train_frame), ctypes.byref(p), ctypes.byref(n)))
        return self._view(p.value, n.value)

    def __iter__(self):
        for k in range(self.n_pairs):
            yield self.pair_at(k)

    def verify(self, ctx_or_multi, keypoints, K, ransac_thre=1.0, ransac_prob=0.99, min_pair_matches=20, random_rate=20, seed=0, max_iters=1000):
        """esfm_two_view_results (a Context) or esfm_multi_two_view_results (a MultiContext): the reference's estimate2D2D_E5P_RANSAC +
        getDepthFast for every pair of this batch with more than min_pair_matches matches (sfm.cpp:163-166), on the device.
        keypoints: one float32[n_f, 2] array of pixel coordinates per frame (frame_t::keypoints[k].pt); K: 3 x 3 (every frame) or
        n_frames x 3 x 3 (a pair uses its query frame's).  Pair (i, j) draws its hypotheses from the key (i << 32) | j.
        Returns (the inlier matches as a new Results in the same pair order, TWO_VIEW_DTYPE[n_pairs])."""
        kps = [np.ascontiguousarray(k, np.float32).reshape(-1, 2) for k in keypoints]
        kp_off = np.zeros(len(kps) + 1, np.int64)
        kp_off[1:] = np.cumsum([len(k) for k in kps])
        xy = np.concatenate(kps + [np.zeros((1, 2), np.float32)])
        K = np.ascontiguousarray(K, np.float64)
        k_per_frame = 1 if K.ndim == 3 else 0
        if K.shape[-2:] != (3, 3) or (k_per_frame and K.shape[0] != len(kps)):
            raise ValueError("K must be 3 x 3 or n_frames x 3 x 3")
        prm = TwoViewParams()
        _check(self._lib.esfm_two_view_default_params(ctypes.byref(prm)))
        prm.ransac_thre, prm.ransac_prob, prm.seed = float(ransac_thre), float(ransac_prob), int(seed)
        prm.max_iters, prm.random_rate = int(max_iters), int(random_rate)
        out = np.zeros(max(self.n_pairs, 1), TWO_VIEW_DTYPE)
        h = c_void_p()
        fn = self._lib.esfm_multi_two_view_results if isinstance(ctx_or_multi, MultiContext) else self._lib.esfm_two_view_results
        _check(fn(ctx_or_multi._h, self._h, len(kps), kp_off.ctypes.data, xy.ctypes.data, K.ctypes.data, k_per_frame, ctypes.byref(prm),
                  int(min_pair_matches), ctypes.byref(h), out.ctypes.data))
        return Results(self._lib, h), out[:self.n_pairs]


class MultiContext:
    """Several GPUs of one box driven by this one process (esfm_multi_t): one worker thread + stream per device inside the
    library, bank replicated with one ncclBroadcast, matches merged into one Results in the caller's pair order."""

    def __init__(self, devices):
        self._lib = load_library()
        devs = list(range(devices)) if isinstance(devices, int) else [int(d) for d in devices]
        arr = (c_int * len(devs))(*devs)
        h = c_void_p()
        _check(self._lib.esfm_multi_init(len(devs), arr, ctypes.byref(h)))
        self._h = h
        self.devices = devs
        self._children = weakref.WeakSet()
        self.contexts = []
        for k, d in enumerate(devs):
            c = c_void_p()
            _check(self._lib.esfm_multi_ctx(self._h, k, ctypes.byref(c)))
            self.contexts.append(Context(d, _borrowed=c))

    def close(self):
        if getattr(self, "_h", None):
            for child in list(getattr(self, "_children", ())):
                child.close()
            for c in self.contexts:
                c.close()
            self._lib.esfm_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_engines(self, l2=None, hamming=None):
        for c in self.contexts:
            if l2:
                c.set_l2_engine(l2)
            if hamming:
                c.set_hamming_engine(hamming)

    def timing(self) -> dict:
        t = MultiTiming()
        _check(self._lib.esfm_multi_timing(self._h, ctypes.byref(t)))
        return t.as_dict()

    def stats(self):
        return [c.stats() for c in self.contexts]

    def bank(self, kind: int, n_frames: int) -> "MultiBank":
        return MultiBank(self, kind, n_frames)

    def bank_from_frames(self, frames) -> "MultiBank":
        frames = list(frames)
        _, kind = _as_desc(frames[0])
        b = MultiBank(self, kind, len(frames))
        for i, f in enumerate(frames):
            b.set_frame(i, f)
        b.commit()
        return b


class MultiBank:
    """A descriptor bank replicated on every device of a MultiContext (esfm_multi_bank_t)."""

    def __init__(self, multi: MultiContext, kind: int, n_frames: int):
        self._lib = multi._lib
        self.multi = multi
        self.kind = int(kind)
        self.n_frames = int(n_frames)
        h = c_void_p()
        _check(self._lib.esfm_multi_bank_create(multi._h, int(kind), int(n_frames), ctypes.byref(h)))
        self._h = h
        multi._children.add(self)
        p = c_void_p()
        _check(self._lib.esfm_multi_bank_primary(self._h, ctypes.byref(p)))
        self.primary = Bank(multi.contexts[0], kind, n_frames, _borrowed=p)   # device-0 replica: set_frame_pinned / device fill

    def close(self):
        if getattr(self, "_h", None):
            self.primary.close()
            self._lib.esfm_multi_bank_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_frame(self, frame_id: int, desc):
        a, _ = _as_desc(desc, self.kind)
        _check(self._lib.esfm_multi_bank_set_frame(self._h, int(frame_id), a.ctypes.data, a.shape[0], a.shape[1],
                                                   a.strides[0] if a.shape[0] else a.shape[1] * a.itemsize))

    def commit(self):
        _check(self._lib.esfm_multi_bank_commit(self._h))

    def match_all_pairs(self, ratio: float, cross_check: bool = False, keep: int = KEEP_MATCHES) -> "Results":
        h = c_void_p()
        _check(self._lib.esfm_multi_match_all_pairs(self._h, float(ratio), int(bool(cross_check)), int(keep), ctypes.byref(h)))
        return Results(self._lib, h, self.multi)

    def match_pairs(self, pairs, ratio: float, cross_check: bool = False, keep: int = KEEP_MATCHES) -> "Results":
        p = np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))
        h = c_void_p()
        _check(self._lib.esfm_multi_match_pairs(self._h, p.ctypes.data, p.shape[0], float(ratio), int(bool(cross_check)), int(keep),
                                                ctypes.byref(h)))
        return Results(self._lib, h, self.multi)


class Tracks:
    """Unique point ids of every keypoint + co-visibility scoring (esfm_tracks_t; reference: sfm.cpp:140-217,
    feature_matching.cpp:160-268).  Building the tracks is host work and needs no device."""

    def __init__(self, keypoints_per_frame):
        self._lib = load_library()
        kp = np.ascontiguousarray(keypoints_per_frame, dtype=np.int32)
        self.keypoints = kp
        self.n_frames = len(kp)
        h = c_void_p()
        _check(self._lib.esfm_tracks_create(len(kp), kp.ctypes.data_as(POINTER(c_int32)), ctypes.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.esfm_tracks_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add_pair(self, frame_i: int, frame_j: int, inlier_matches):
        m = np.ascontiguousarray(inlier_matches, dtype=DMATCH_DTYPE)
        _check(self._lib.esfm_tracks_add_pair(self._h, int(frame_i), int(frame_j), m.ctypes.data if len(m) else None, len(m)))

    def finish_frame(self, frame_i: int):
        _check(self._lib.esfm_tracks_finish_frame(self._h, int(frame_i)))

    def build(self, results: "Results", min_pair_matches: int = 20):
        _check(self._lib.esfm_tracks_build(self._h, results._h, int(min_pair_matches)))

    def frame(self, f: int):
        """(unique_pixel_ids int32 [n], unique_pixel_has_match uint8 [n]) of frame f (copies)."""
        pi, ph, n = c_void_p(), c_void_p(), c_int()
        _check(self._lib.esfm_tracks_frame(self._h, int(f), ctypes.byref(pi), ctypes.byref(ph), ctypes.byref(n)))
        if n.value == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.uint8)
        ids = np.frombuffer((ctypes.c_char * (4 * n.value)).from_address(pi.value), np.int32, n.value).copy()
        has = np.frombuffer((ctypes.c_char * n.value).from_address(ph.value), np.uint8, n.value).copy()
        return ids, has

    def counts(self):
        """(frames finished, unique points so far)."""
        d, p = c_int(), c_int64()
        _check(self._lib.esfm_tracks_counts(self._h, ctypes.byref(d), ctypes.byref(p)))
        return d.value, p.value

    def pair_scores(self, ctx: Context):
        """Co-visibility score of every pair in loop order (device kernel) -> (int64 [n_pairs], kernel ms)."""
        n = self.n_frames * (self.n_frames - 1) // 2
        out = np.zeros(max(n, 1), np.int64)
        ms = c_double()
        _check(self._lib.esfm_tracks_pair_scores(ctx._h, self._h, out.ctypes.data_as(POINTER(c_int64)), ctypes.byref(ms)))
        return out[:n], ms.value

    def find_init_pair(self, ctx: Context, appro_depth=None, min_track_num_init: int = 100, max_depth_baseline_ratio_init: float = 50.0):
        """findInitializeFramePair -> (found, frame_1, frame_2, depth_init, best_score)."""
        d = None if appro_depth is None else np.ascontiguousarray(appro_depth, dtype=np.float64)
        f1, f2, di, best, found = c_int(), c_int(), c_double(), c_int64(), c_int()
        _check(self._lib.esfm_tracks_find_init_pair(ctx._h, self._h, None if d is None else d.ctypes.data_as(POINTER(c_double)),
                                                    int(min_track_num_init), float(max_depth_baseline_ratio_init), ctypes.byref(f1),
                                                    ctypes.byref(f2), ctypes.byref(di), ctypes.byref(best), ctypes.byref(found)))
        return bool(found.value), f1.value, f2.value, di.value, best.value

    def find_next_frame(self, frames_to_process, point_ids, next_frame: int = -1):
        """findNextFrame -> (next_frame, common points)."""
        tp = np.ascontiguousarray(frames_to_process, dtype=np.uint8)
        pid = np.ascontiguousarray(point_ids, dtype=np.int32)
        nf, common = c_int(int(next_frame)), c_int()
        _check(self._lib.esfm_tracks_find_next_frame(self._h, tp.ctypes.data_as(POINTER(ctypes.c_uint8)),
                                                     pid.ctypes.data_as(POINTER(c_int32)) if len(pid) else None, len(pid),
                                                     ctypes.byref(nf), ctypes.byref(common)))
        return nf.value, common.value
