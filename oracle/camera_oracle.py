"""CPU ORACLE (test infrastructure, NOT product code) for the calibrated camera (include/ofb200.h `ofb_camera`).

Restates OpenCV's cv2.undistortPoints / cv2.undistortPointsIter with the COUNT criterion (cvUndistortPointsInternal
in modules/calib3d/src/undistort.dispatch.cpp, an un-vendored dependency) in fp64 and in its operation order:

    x0 = (px - cx) * (1/fx), y0 = (py - cy) * (1/fy); x = x0, y = y0
    `iterations` times (none without coefficients):
        r2 = x*x + y*y
        icdist = (1 + ((k6*r2 + k5)*r2 + k4)*r2) / (1 + ((k3*r2 + k2)*r2 + k1)*r2)
        icdist < 0: x = x0, y = y0, stop
        dx = 2*p1*x*y + p2*(r2 + 2*x*x);  dy = p1*(r2 + 2*y*y) + 2*p2*x*y
        x = (x0 - dx)*icdist;  y = (y0 - dy)*icdist
    xx = H0 x + H1 y + H2, yy = H3 x + H4 y + H5, ww = 1/(H6 x + H7 y + H8): (xx*ww, yy*ww),  H = P[:, :3] @ R

NumPy evaluates every elementwise expression above in that order without contraction, so on the same inputs it
reproduces cv2 4.13 bit for bit (pinned by tests/golden/camera_golden.npz, made by tools/make_golden_camera.py).

CameraTrackerOracle is oracle/tracker_oracle.py's TrackerOracle with a calibrated camera in place of the pinhole
(principal, scaling): the r_tilde gate and the solve see x = undistort(p_new), u = (undistort(p_new) -
undistort(p_old)) * rate, static_immobile stays in pixels.

Only tests/, tools/ and __graft_entry__.smoke() may import this.
"""
import numpy as np

from . import tracker_oracle


def rectification(R=None, P=None):
    """H = P[:, :3] @ R as OpenCV forms it (cvMatMul: sums over k in order), or None for the identity."""
    if R is None and P is None:
        return None
    Rm = np.eye(3) if R is None else np.asarray(R, np.float64).reshape(3, 3)
    if P is None:
        return Rm.copy()
    Pm = np.asarray(P, np.float64).reshape(3, -1)[:, :3]
    H = np.zeros((3, 3))
    for i in range(3):
        for j in range(3):
            H[i, j] = Pm[i, 0] * Rm[0, j] + Pm[i, 1] * Rm[1, j] + Pm[i, 2] * Rm[2, j]
    return H


def undistort(pts, K, D, iterations=5, H=None):
    """(N,2) pixels -> (N,2) float64: normalised coordinates, or rectified/projected ones with H."""
    p = np.asarray(pts, np.float64).reshape(-1, 2)
    K = np.asarray(K, np.float64).reshape(3, 3)
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    x0 = (p[:, 0] - cx) * (1.0 / fx)
    y0 = (p[:, 1] - cy) * (1.0 / fy)
    x, y = x0.copy(), y0.copy()
    D = np.zeros(0) if D is None else np.asarray(D, np.float64).ravel()
    if len(D):
        k = np.zeros(8)
        k[:len(D)] = D
        k1, k2, p1, p2, k3, k4, k5, k6 = k
        live = np.ones(len(p), bool)                  # points whose iteration has not stopped at icdist < 0
        for _ in range(int(iterations)):
            r2 = x * x + y * y
            icdist = (1 + ((k6 * r2 + k5) * r2 + k4) * r2) / (1 + ((k3 * r2 + k2) * r2 + k1) * r2)
            stop = live & (icdist < 0)
            x[stop], y[stop] = x0[stop], y0[stop]
            live &= ~stop
            dx = 2 * p1 * x * y + p2 * (r2 + 2 * x * x)
            dy = p1 * (r2 + 2 * y * y) + 2 * p2 * x * y
            x = np.where(live, (x0 - dx) * icdist, x)
            y = np.where(live, (y0 - dy) * icdist, y)
    if H is not None:
        H = np.asarray(H, np.float64).reshape(3, 3)
        xx = H[0, 0] * x + H[0, 1] * y + H[0, 2]
        yy = H[1, 0] * x + H[1, 1] * y + H[1, 2]
        ww = 1. / (H[2, 0] * x + H[2, 1] * y + H[2, 2])
        x, y = xx * ww, yy * ww
    return np.stack([x, y], axis=1)


def calibrate(new, old, camera):
    """The velocity paths' metric inputs for tracks (new, old) (float32 pixels, (N,2)) under camera = (K, D, rate,
    iterations): x = undistort(new), u = (undistort(new) - undistort(old)) * rate."""
    K, D, rate, iterations = camera
    xn = undistort(np.asarray(new, np.float32), K, D, iterations)
    xo = undistort(np.asarray(old, np.float32), K, D, iterations)
    return xn, (xn - xo) * rate


class _CalibratedEngine(tracker_oracle.Engine):
    """Wraps the step operators of a TrackerOracle that runs with the identity pinhole (principal (0, 0), scaling 1, so
    the x it hands to r_tilde and solve are the float32 positions widened). It keeps the (old, new) tracks of the step
    from the LK call and the survivors of each filter, and hands r_tilde and solve the calibrated x, u of those tracks
    instead of the pinhole's."""

    def __init__(self, inner, camera, gate):
        self.inner, self.camera, self.gate = inner, camera, gate
        self.old = self.new = self.keep = None

    def good_features(self, *a, **k):
        return self.inner.good_features(*a, **k)

    def mask(self, *a, **k):
        return self.inner.mask(*a, **k)

    def bgr2gray(self, bgr):
        return self.inner.bgr2gray(bgr)

    def pyrlk(self, prev, nxt, pts, win, max_level, criteria):
        new, st, err = self.inner.pyrlk(prev, nxt, pts, win, max_level, criteria)
        self.old = np.asarray(pts, np.float32).reshape(-1, 2)
        self.new = np.asarray(new, np.float32).reshape(-1, 2)
        self.keep = np.asarray(st).reshape(-1) == 1                    # evaluate_exp.py:99
        return new, st, err

    def static_immobile(self, new, old, maxspeed, distance, dummy):
        m = self.inner.static_immobile(new, old, maxspeed, distance, dummy)
        self.keep = self.keep & np.asarray(m).reshape(-1).astype(bool)
        return m

    def r_tilde(self, x, u, n, v, d):
        assert np.array_equal(x, self.new.astype(np.float64))
        xc, uc = calibrate(self.new, self.old, self.camera)
        r = np.asarray(self.inner.r_tilde(xc, uc, n, v, d))
        self.keep = self.keep & ((r >= self.gate[1]) if self.gate[0] == "ge" else (r <= self.gate[1]))
        return r

    def solve(self, x, u, d, n, w, t, variant):
        kn, kp = self.new[self.keep], self.old[self.keep]
        assert np.array_equal(x, kn.astype(np.float64)), "the kept tracks are not the ones the filters passed"
        xc, uc = calibrate(kn, kp, self.camera)
        return self.inner.solve(xc, uc, d, n, w, t, variant)


class CameraTrackerOracle(tracker_oracle.TrackerOracle):
    """One camera stream, parameters as ofb200.StreamTracker(camera=...): camera = (K, D, rate, iterations); principal /
    scaling, if given, are not used."""

    def __init__(self, width, height, camera, engine=None, **kw):
        kw = {k: v for k, v in kw.items() if k not in ("principal", "scaling")}
        super().__init__(width, height, principal=(0.0, 0.0), scaling=1.0,
                         engine=_CalibratedEngine(engine or tracker_oracle.Engine(), camera, kw.get("gate")), **kw)
        self.camera = camera
