"""ctypes front-end of oracle/of_oracle.c (CPU ORACLE, test infrastructure, NOT product code).

Restates OpenCV's pyrDown / cornerMinEigenVal / goodFeaturesToTrack / calcOpticalFlowPyrLK as
called by the reference (velocity_measurment_node:120,133,163; evaluate_exp.py:66,98,106;
of_module.py:44,86,88). Pinned against cv2 4.13.0 in tests/test_oracle_vs_cv2.py.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libof_oracle.so")
_lib = None


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = ctypes.CDLL(_SO)
        u8p = ctypes.POINTER(ctypes.c_uint8)
        f32p = ctypes.POINTER(ctypes.c_float)
        L.orc_bgr2gray.argtypes = [u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, u8p, ctypes.c_int]
        L.orc_bgr2gray.restype = None
        L.orc_pyr_down.argtypes = [u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, u8p, ctypes.c_int]
        L.orc_pyr_down.restype = None
        L.orc_min_eig_map.argtypes = [u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, f32p]
        L.orc_min_eig_map.restype = None
        L.orc_min_eig_map_fp32sum.argtypes = L.orc_min_eig_map.argtypes
        L.orc_min_eig_map_fp32sum.restype = None
        L.orc_select_features.argtypes = [f32p, ctypes.c_int, ctypes.c_int, u8p, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_double, ctypes.c_double, f32p, ctypes.c_int]
        L.orc_select_features.restype = ctypes.c_int
        L.orc_good_features.argtypes = [u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, u8p, ctypes.c_int,
                                        ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_int,
                                        f32p, ctypes.c_int]
        L.orc_good_features.restype = ctypes.c_int
        L.orc_pyrlk.argtypes = [u8p, u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, f32p, ctypes.c_int,
                                ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                ctypes.c_int, ctypes.c_double, f32p, u8p, f32p]
        L.orc_pyrlk.restype = ctypes.c_int
        _lib = L
    return _lib


def _u8(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))


def _f32(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def bgr2gray(bgr):
    bgr = np.ascontiguousarray(bgr, dtype=np.uint8)
    h, w, _ = bgr.shape
    out = np.empty((h, w), np.uint8)
    lib().orc_bgr2gray(_u8(bgr), w, h, 3 * w, _u8(out), w)
    return out


def pyr_down(img):
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w = img.shape
    out = np.empty(((h + 1) // 2, (w + 1) // 2), np.uint8)
    lib().orc_pyr_down(_u8(img), w, h, w, _u8(out), out.shape[1])
    return out


def build_pyramid(img, max_level):
    levels = [np.ascontiguousarray(img, dtype=np.uint8)]
    for _ in range(max_level):
        levels.append(pyr_down(levels[-1]))
    return levels


def min_eig_map(img, block_size, fp32_sums=False):
    """cornerMinEigenVal from EXACT integer window sums (default), or with OpenCV-style fp32 accumulation."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w = img.shape
    eig = np.empty((h, w), np.float32)
    fn = lib().orc_min_eig_map_fp32sum if fp32_sums else lib().orc_min_eig_map
    fn(_u8(img), w, h, w, block_size, _f32(eig))
    return eig


def select_features(eig, max_corners, quality, min_distance, mask=None):
    eig = np.ascontiguousarray(eig, dtype=np.float32)
    h, w = eig.shape
    cap = max_corners if max_corners > 0 else w * h
    xy = np.empty((cap, 2), np.float32)
    mp = None
    if mask is not None:
        mask = np.ascontiguousarray(mask, dtype=np.uint8)
        mp = _u8(mask)
    n = lib().orc_select_features(_f32(eig), w, h, mp, w, max_corners, quality, min_distance, _f32(xy), cap)
    return None if n == 0 else xy[:n].reshape(-1, 1, 2).copy()


def good_features(img, max_corners, quality, min_distance, mask=None, block_size=3):
    return select_features(min_eig_map(img, block_size), max_corners, quality, min_distance, mask)


ORC_LK_EXACT_SUMS = 1 << 16


def pyrlk(prev, nxt, prev_pts, win=(21, 21), max_level=3, criteria=(3, 30, 0.01), min_eig_thr=1e-4, exact_sums=False):
    """calcOpticalFlowPyrLK. exact_sums=False: OpenCV's fp32 running sums; True: A, b and the error summed exactly
    in int64 and rounded to fp32 once, the arithmetic of the device kernels. As cv2, a criteria type without
    TERM_CRITERIA_COUNT (1) means 30 iterations and one without TERM_CRITERIA_EPS (2) eps = 0.01."""
    prev = np.ascontiguousarray(prev, dtype=np.uint8)
    nxt = np.ascontiguousarray(nxt, dtype=np.uint8)
    h, w = prev.shape
    p = np.ascontiguousarray(np.asarray(prev_pts, dtype=np.float32).reshape(-1, 2))
    n = len(p)
    out = np.zeros((n, 2), np.float32)
    st = np.zeros(n, np.uint8)
    err = np.zeros(n, np.float32)
    typ, count, eps = criteria
    count = int(count) if int(typ) & 1 else 30
    eps = float(eps) if int(typ) & 2 else 0.01
    lib().orc_pyrlk(_u8(prev), _u8(nxt), w, h, w, _f32(p), n, win[0], win[1], max_level, count,
                    eps, ORC_LK_EXACT_SUMS if exact_sums else 0, min_eig_thr, _f32(out), _u8(st), _f32(err))
    return out.reshape(-1, 1, 2), st.reshape(-1, 1), err.reshape(-1, 1)
