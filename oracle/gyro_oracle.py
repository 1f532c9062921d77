"""CPU ORACLE (test infrastructure, NOT product code) for the gyro prediction of the LK tracks (include/ofb200.h
`ofb_gyro_predict`, `ofb_frame_pairs_gyro`, `ofb_tracker_set_gyro_prediction`):

* predict          the predictor in NumPy fp64: normalise (pinhole or camera_oracle.undistort), rotate (x, y, 1) by
                   exp([w dt]x) (Rodrigues, series below (|w| dt)^2 = 1e-4), divide by z, back to pixels (pinhole or
                   project_points); the point itself where z <= 0 or anything is not finite, and for w = 0
* project_points   cv2.projectPoints of (x, y, 1) with zero rvec / tvec, restated in cvProjectPoints2Internal's operation
                   order (pinned to cv2 4.13 by tests/golden/gyro_golden.npz)
* pyrlk_init       the C oracle's LK with OPTFLOW_USE_INITIAL_FLOW (oracle/lk_init_oracle.c: of_oracle.c's orc_pyrlk
                   started from the guess; compiled on first use into a temporary directory)
* GyroEngine       a tracker_oracle.Engine wrapper whose pyrlk starts from the prediction under the step's gyro rate
                   (set `engine.w` before each TrackerOracle.step), with the forward-backward check of fb_oracle folded
                   in when T > 0 (backward pass seeded with p1 + (p0 - guess))
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from . import camera_oracle as co
from . import fb_oracle
from . import image_oracle as io

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    """libof_oracle's LK with initial flow (oracle/lk_init_oracle.c), built with of_oracle's flags into the temporary
    directory the first time (the source tree may be read-only); the file name carries a hash of both sources."""
    global _lib
    if _lib is None:
        srcs = [os.path.join(_HERE, f) for f in ("lk_init_oracle.c", "of_oracle.c")]
        h = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "ofb_lk_init_oracle_%d_%s.so" % (os.getuid(), h))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-fvisibility=hidden", "-ffp-contract=off", "-shared",
                                   "-I", _HERE, "-o", tmp, srcs[0], "-lm"], stderr=subprocess.DEVNULL)
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        u8p, f32p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_float)
        L.orc_pyrlk_init.argtypes = [u8p, u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, f32p, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, f32p, u8p,
                                     f32p]
        L.orc_pyrlk_init.restype = ctypes.c_int
        _lib = L
    return _lib


def pinhole(cx, cy, pos_scale, flow_scale):
    """The pinhole model of a frame-pair configuration: dt = pos_scale / flow_scale."""
    return ("pinhole", float(cx), float(cy), float(pos_scale), float(pos_scale) / float(flow_scale))


def camera(K, D, rate, iterations):
    """The calibrated model (the velocity paths' camera tuple): dt = 1 / rate."""
    return ("camera", np.asarray(K, np.float64).reshape(3, 3), None if D is None else np.asarray(D, np.float64).ravel(),
            float(rate), int(iterations))


def project_points(xy, K, D):
    """(N,2) normalised coordinates -> (N,2) float64 pixels, cv2.projectPoints(np.c_[xy, 1], 0, 0, K, D)."""
    xy = np.asarray(xy, np.float64).reshape(-1, 2)
    K = np.asarray(K, np.float64).reshape(3, 3)
    k = np.zeros(8)
    if D is not None and len(np.ravel(D)):
        d = np.asarray(D, np.float64).ravel()
        k[:len(d)] = d
    k1, k2, p1, p2, k3, k4, k5, k6 = k
    x, y = xy[:, 0], xy[:, 1]
    r2 = x * x + y * y
    r4 = r2 * r2
    r6 = r4 * r2
    a1 = 2 * x * y
    a2 = r2 + 2 * x * x
    a3 = r2 + 2 * y * y
    cdist = 1 + k1 * r2 + k2 * r4 + k3 * r6
    icdist2 = 1. / (1 + k4 * r2 + k5 * r4 + k6 * r6)
    xd = x * cdist * icdist2 + p1 * a1 + p2 * a2
    yd = y * cdist * icdist2 + p1 * a3 + p2 * a1
    return np.stack([xd * K[0, 0] + K[0, 2], yd * K[1, 1] + K[1, 2]], axis=1)


def rotation_coeffs(r):
    """(a, b) of R X = X + a (r x X) + b r x (r x X) for the rotation vector r (fp64, as the device computes them)."""
    t2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2]
    if t2 < 1e-4:
        return 1.0 - t2 * (1.0 / 6.0 - t2 * (1.0 / 120.0)), 0.5 - t2 * (1.0 / 24.0 - t2 * (1.0 / 720.0))
    t = np.sqrt(t2)
    s = np.sin(0.5 * t)
    return np.sin(t) / t, 2.0 * s * s / t2


def predict(points, w, model):
    """(N,2) / (N,1,2) float32 pixels -> (N,2) float32 guesses under the gyro rate w (3,) for `model` (pinhole(...) or
    camera(...))."""
    p = np.asarray(points, np.float32).reshape(-1, 2)
    w = np.asarray(w, np.float64).reshape(3)
    if not np.any(w):                       # no rotation: the point itself (the lens model's round trip is not exact)
        return p.copy()
    with np.errstate(all="ignore"):
        if model[0] == "pinhole":
            _, cx, cy, ps, dt = model
            x = (p[:, 0].astype(np.float64) - cx) * ps
            y = (p[:, 1].astype(np.float64) - cy) * ps
        else:
            _, K, D, rate, iters = model
            xy = co.undistort(p, K, D, iters)
            x, y = xy[:, 0], xy[:, 1]
            dt = 1.0 / rate
        r = w * dt
        a, b = rotation_coeffs(r)
        c0, c1, c2 = r[1] - r[2] * y, r[2] * x - r[0], r[0] * y - r[1] * x
        d0, d1, d2 = r[1] * c2 - r[2] * c1, r[2] * c0 - r[0] * c2, r[0] * c1 - r[1] * c0
        X, Y, Z = x + a * c0 + b * d0, y + a * c1 + b * d1, 1.0 + a * c2 + b * d2
        xn, yn = X / Z, Y / Z
        if model[0] == "pinhole":
            g = np.stack([cx + xn / ps, cy + yn / ps], axis=1)
        else:
            g = project_points(np.stack([xn, yn], axis=1), K, D)
        g = g.astype(np.float32)
    ok = (Z > 0) & np.isfinite(g).all(axis=1)
    return np.where(ok[:, None], g, p).astype(np.float32)


def pyrlk_init(prev, nxt, prev_pts, guess, win=(21, 21), max_level=3, criteria=(3, 30, 0.01), min_eig_thr=1e-4):
    """image_oracle.pyrlk started from `guess` (OPTFLOW_USE_INITIAL_FLOW)."""
    prev = np.ascontiguousarray(prev, dtype=np.uint8)
    nxt = np.ascontiguousarray(nxt, dtype=np.uint8)
    h, w = prev.shape
    p = np.ascontiguousarray(np.asarray(prev_pts, dtype=np.float32).reshape(-1, 2))
    n = len(p)
    out = np.ascontiguousarray(np.asarray(guess, dtype=np.float32).reshape(-1, 2)).copy()
    st = np.zeros(n, np.uint8)
    err = np.zeros(n, np.float32)
    _, count, eps = criteria
    lib().orc_pyrlk_init(io._u8(prev), io._u8(nxt), w, h, w, io._f32(p), n, win[0], win[1], max_level, int(count),
                         float(eps), min_eig_thr, io._f32(out), io._u8(st), io._f32(err))
    return out.reshape(-1, 1, 2), st.reshape(-1, 1), err.reshape(-1, 1)


def track(prev, nxt, p0, guess, win, max_level, criteria, T=0.0, lk=pyrlk_init):
    """Forward LK from `guess`; with T > 0 the backward LK from p1 + (p0 - guess) and fb_oracle's fold.
    -> (p1 (N,1,2), status (N,1), err (N,1))."""
    p0 = np.asarray(p0, np.float32).reshape(-1, 2)
    g = np.asarray(guess, np.float32).reshape(-1, 2)
    p1, st, err = lk(prev, nxt, p0, g, win, max_level, criteria)
    if T == 0.0:
        return p1, st, err
    p1f = np.asarray(p1, np.float32).reshape(-1, 2)
    p0r, st0, _ = lk(nxt, prev, p1f, p1f + (p0 - g), win, max_level, criteria)
    status, _ = fb_oracle.fb_check(p0, p1, st, p0r, st0, T)
    return p1, status.reshape(np.shape(st)), err


class GyroEngine:
    """Step operators of `inner` with pyrlk started from the gyro prediction (model: pinhole(...) / camera(...)) under
    `self.w`, the gyro rate of the step about to run. T > 0 adds the forward-backward check with the seeded backward
    pass. Every other operator is the inner engine's."""

    def __init__(self, inner, model, T=0.0):
        self.inner, self.model, self.T = inner, model, float(T)
        self.w = np.zeros(3)

    def __getattr__(self, name):
        return getattr(self.inner, name)

    def pyrlk(self, prev, nxt, pts, win, max_level, criteria):
        g = predict(pts, self.w, self.model)
        return track(prev, nxt, pts, g, win, max_level, criteria, self.T)
