"""CPU ORACLE (test infrastructure, NOT product code) for the forward-backward check of the LK tracks (include/ofb200.h
`ofb_pyrlk_fb`), the check of OpenCV's samples/python/lk_track.py:

    p1, st, err = cv2.calcOpticalFlowPyrLK(img0, img1, p0, None, **lk_params)
    p0r, st0, _ = cv2.calcOpticalFlowPyrLK(img1, img0, p1, None, **lk_params)
    d = abs(p0 - p0r).reshape(-1, 2).max(-1)
    good = d < 1

with one difference: the backward status must be 1 as well (the positions of points that lose status are not pinned
to cv2 anywhere in this project).

* fb_check   the fold of the two passes into (status, fb_err) in NumPy
* FBEngine   a tracker_oracle.Engine wrapper whose pyrlk runs the inner engine forward, backward, and folds: wrapping
             the C oracle's Engine or the cv2 engine of tests/tracker_cases.py gives TrackerOracle with the check, and
             passing it as CameraTrackerOracle's engine= gives it with a calibrated camera as well.
"""
import numpy as np


def fb_check(p0, p1, st1, p0r, st0, T):
    """-> (status (N,) uint8, fb_err (N,) float32). fb_err = max(|x0 - x0r|, |y0 - y0r|) in float32 where both passes
    have status 1, +inf elsewhere; status = 1 iff both passes have status 1 and fb_err < T (compared in float64).
    T == 0: no check (status = st1, fb_err = +inf everywhere). p1 is not used by the fold; it is the caller's forward
    result and stays as it is."""
    T = float(T)
    if not T >= 0.0:
        raise ValueError("T must be >= 0")
    st1 = np.asarray(st1).reshape(-1) == 1
    if T == 0.0:
        return st1.astype(np.uint8), np.full(len(st1), np.inf, np.float32)
    p0 = np.asarray(p0, np.float32).reshape(-1, 2)
    p0r = np.asarray(p0r, np.float32).reshape(-1, 2)
    both = st1 & (np.asarray(st0).reshape(-1) == 1)
    d = np.abs(p0 - p0r).max(-1)
    fb_err = np.where(both, d, np.float32(np.inf)).astype(np.float32)
    return (both & (fb_err.astype(np.float64) < T)).astype(np.uint8), fb_err


class FBEngine:
    """Step operators of `inner` with the forward-backward check folded into pyrlk's status (threshold T px). Every other
    operator is the inner engine's."""

    def __init__(self, inner, T):
        self.inner, self.T = inner, float(T)

    def __getattr__(self, name):
        return getattr(self.inner, name)

    def pyrlk(self, prev, nxt, pts, win, max_level, criteria):
        p1, st, err = self.inner.pyrlk(prev, nxt, pts, win, max_level, criteria)
        if self.T == 0.0:
            return p1, st, err
        p0r, st0, _ = self.inner.pyrlk(nxt, prev, np.asarray(p1, np.float32).reshape(-1, 1, 2), win, max_level, criteria)
        status, _ = fb_check(pts, p1, st, p0r, st0, self.T)
        return p1, status.reshape(np.shape(st)), err
