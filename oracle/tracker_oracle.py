"""CPU ORACLE (test infrastructure, NOT product code) for the feature lifecycle around the tracker
(SURVEY 8f-2). Restates, step by step, what the reference's per-frame loops do (paths relative to
the original project's checkout):

* track + status filter      flight_experiments/evaluate_exp.py:97-99, velocity_measurment_node:133-136
* static_immobile            of_library.py:88-92
* r_tilde gate               velocity_measurment_node:238-245 (keeps r <= T), optical_flow_experiments/of_module.py:125-131
                             (keeps r - (status-1) >= T, i.e. r >= T for tracked points)
* px -> metric + solve_lgs   velocity_measurment_node:229-235, 247-250; evaluate_exp.py:113
* top-up                     evaluate_exp.py:105-107 ("exp": unmasked, maxCorners=max_feat, appended),
                             velocity_measurment_node:157-172 ("node": cv2.circle exclusion mask, maxCorners=max_feat-len),
                             of_module.py:83-86 ("module": the set is replaced)
* exclusion mask             cv2.circle(mask, centre, radius, 0, cv2.FILLED) of node:161 = OpenCV's Circle() in
                             imgproc/drawing.cpp (un-vendored dependency; restated from its published midpoint loop)

The loops themselves are module-level script code (they read yaml/video files and open windows), so they cannot be
exec'd; the restatement is pinned instead by tests/test_oracle_tracker.py, which runs the SAME steps with the real
cv2.calcOpticalFlowPyrLK / cv2.goodFeaturesToTrack / cv2.circle and the reference's own of_library.static_immobile,
of_library.r_tilde and solve_lgs (AST-extracted) where those are available, and by tests/golden/tracker_golden.npz
(made by tools/make_golden_tracker.py with cv2 4.13) where they are not.

Documented decisions where the reference code is ambiguous or does not run:
* evaluate_exp.py:113 forms `new_pos - old_pos` after filtering/appending, which only broadcasts when nothing was
  lost or added; the flow used here is new-old of the points that survived (what node:136 computes).
* The top-up runs on the CURRENT frame after the solve (evaluate_exp.py:105-107); appended points get their first
  flow on the next frame.
* Float coordinates passed to cv2.circle are truncated (Python-2 cv2 semantics).
* Points that fail a gate leave the set (node:245).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this.
"""
import numpy as np

from . import image_oracle as io
from . import velocity_oracle as vo


def circle_half_widths(radius):
    """Half width of every row of OpenCV's filled circle: Circle() walks (dx,dy) from (radius,0) while dx>=dy and
    fills rows cy+-dy over cx+-dx and rows cy+-dx over cx+-dy."""
    hw = [-1] * (radius + 1)
    err, dx, dy, plus, minus = 0, radius, 0, 1, (radius << 1) - 1
    while dx >= dy:
        hw[dy] = max(hw[dy], dx)
        hw[dx] = max(hw[dx], dy)
        dy += 1
        err += plus
        plus += 2
        mask = (1 if err <= 0 else 0) - 1          # 0 or -1
        err -= minus & mask
        dx += mask
        minus -= mask & 2
    return [max(v, 0) for v in hw]


def exclusion_mask(points, radius, width, height):
    """np.ones_like(gray) with cv2.circle(mask, (int(x), int(y)), radius, 0, cv2.FILLED) per point (node:159-161)."""
    m = np.ones((height, width), np.uint8)
    hw = circle_half_widths(radius)
    for x, y in np.asarray(points, dtype=np.float32).reshape(-1, 2):
        cx, cy = int(x), int(y)
        for dy in range(-radius, radius + 1):
            yy = cy + dy
            if 0 <= yy < height:
                half = hw[abs(dy)]
                x0, x1 = max(cx - half, 0), min(cx + half, width - 1)
                if x1 >= x0:
                    m[yy, x0:x1 + 1] = 0
    return m


def static_immobile(newpos, oldpos, maxspeed, distance, dummy_value):
    """of_library.py:88-92 on (N,1,2) float32 arrays."""
    newpos = np.asarray(newpos, dtype=np.float32).reshape(-1, 1, 2)
    oldpos = np.asarray(oldpos, dtype=np.float32).reshape(-1, 1, 2)
    speed = np.abs(newpos - oldpos) < np.float32(maxspeed / distance)
    dummy = oldpos != np.float32(dummy_value)
    stable = speed * dummy
    return stable[:, :, 0] * stable[:, :, 1]


class Engine:
    """The image operators a step uses. Default: the C restatement (oracle/of_oracle.c)."""

    def good_features(self, img, max_corners, quality, min_distance, block_size, mask=None):
        return io.good_features(img, max_corners, quality, min_distance, mask=mask, block_size=block_size)

    def pyrlk(self, prev, nxt, pts, win, max_level, criteria):
        return io.pyrlk(prev, nxt, pts, win=win, max_level=max_level, criteria=criteria)

    def mask(self, points, radius, width, height):
        return exclusion_mask(points, radius, width, height)

    def bgr2gray(self, bgr):
        return io.bgr2gray(bgr)

    def solve(self, x, u, d, n, w, t, variant):
        return vo.solve_lgs(x, u, d, n, w, t=t, variant=variant)

    def r_tilde(self, x, u, n, v, d):
        return vo.r_tilde(x, u, n, v, d)[0]

    def static_immobile(self, new, old, maxspeed, distance, dummy):
        return static_immobile(new, old, maxspeed, distance, dummy)


class TrackerOracle:
    """One camera stream. Parameters mirror ofb200.StreamTracker."""

    def __init__(self, width, height, max_features=100, min_features=20, feature_params=None, lk_params=None,
                 topup="exp", mask_radius=30, bgr=False, variant="exp", principal=None, scaling=1.0, max_speed=0.0,
                 dummy_value=float("nan"), gate=None, min_solve=3, engine=None):
        self.w, self.h = width, height
        self.K, self.min_feat = max_features, min_features
        self.fp = dict(qualityLevel=0.01, minDistance=10, blockSize=7)
        self.fp.update(feature_params or {})
        self.lk = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
        self.lk.update(lk_params or {})
        self.topup, self.radius, self.bgr, self.variant = topup, mask_radius, bgr, variant
        self.c = principal if principal is not None else vo.pix_trans((width, height))
        self.scaling, self.max_speed, self.dummy, self.gate, self.min_solve = scaling, max_speed, dummy_value, gate, min_solve
        self.E = engine or Engine()
        self.prev = None
        self.pts = np.zeros((0, 2), np.float32)
        self.v_last = np.zeros(3)

    def set_points(self, pts):
        self.pts = np.asarray(pts, dtype=np.float32).reshape(-1, 2).copy()

    def _detect(self, gray, max_corners, mask=None):
        f = self.E.good_features(gray, max_corners, self.fp["qualityLevel"], self.fp["minDistance"], self.fp["blockSize"],
                                 mask=mask)
        return np.zeros((0, 2), np.float32) if f is None else np.asarray(f, np.float32).reshape(-1, 2)

    def step(self, frame, d, n, w, t=None, v_prior=None):
        """-> dict(v, s, res, rank, solved, n_prev, n_tracked, n_kept, n_added, n_points, kept_prev, kept_next)."""
        gray = self.E.bgr2gray(frame) if self.bgr else np.ascontiguousarray(frame, dtype=np.uint8)
        old = self.pts
        out = dict(v=np.zeros(3), s=np.zeros(3), res=0.0, rank=0, solved=False, n_prev=len(old))
        if self.prev is None:
            new, keep = old.copy(), np.ones(len(old), bool)
            out["n_tracked"] = len(old)
        else:
            if len(old):
                new, st, _ = self.E.pyrlk(self.prev, gray, old, self.lk["winSize"], self.lk["maxLevel"], self.lk["criteria"])
                new, st = np.asarray(new, np.float32).reshape(-1, 2), np.asarray(st).reshape(-1)
            else:
                new, st = np.zeros((0, 2), np.float32), np.zeros(0, np.uint8)
            keep = st == 1                                                # evaluate_exp.py:99
            out["n_tracked"] = int(keep.sum())
            if self.max_speed > 0 and len(old):                            # of_library.py:88-92
                keep = keep & self.E.static_immobile(new, old, self.max_speed, d, self.dummy).reshape(-1).astype(bool)
            if self.gate is not None and len(old):                         # node:238-245, of_module.py:125-131
                vp = self.v_last if v_prior is None else np.asarray(v_prior, np.float64)
                x = (new.astype(np.float64) - np.asarray(self.c, np.float64)) * self.scaling
                u = (new - old).astype(np.float64) * self.scaling
                r = np.asarray(self.E.r_tilde(x, u, n, vp, d))
                keep = keep & ((r >= self.gate[1]) if self.gate[0] == "ge" else (r <= self.gate[1]))
        kp, kn = old[keep], new[keep]
        out["kept_prev"], out["kept_next"], out["n_kept"] = kp, kn, len(kn)
        if self.prev is not None and len(kn) >= self.min_solve and len(kn) > 0:
            x = (kn.astype(np.float64) - np.asarray(self.c, np.float64)) * self.scaling    # node:229-233
            u = (kn - kp).astype(np.float64) * self.scaling                                 # node:235 (fp32 flow)
            v, res, rank, s = self.E.solve(x, u, d, n, w, None if self.variant == "node" else t, self.variant)
            out.update(v=np.asarray(v), s=np.asarray(s), rank=int(rank), solved=True,
                       res=float(res[0]) if np.size(res) else 0.0)
            self.v_last = np.asarray(v, np.float64)
        pts, added = kn, 0
        if len(kn) <= self.min_feat:
            if self.topup == "exp":                                        # evaluate_exp.py:105-107
                f = self._detect(gray, self.K)
            elif self.topup == "node":                                     # node:157-172
                mask = self.E.mask(kn, self.radius, self.w, self.h) if self.radius > 0 else None
                f = self._detect(gray, self.K - len(kn), mask)
            else:                                                          # of_module.py:83-86
                f = self._detect(gray, self.K - len(kn))
                pts = np.zeros((0, 2), np.float32)
            added = len(f)
            pts = np.concatenate([pts, f], axis=0).astype(np.float32)
        self.pts, self.prev = pts, gray
        out["n_added"], out["n_points"] = added, len(pts)
        return out
