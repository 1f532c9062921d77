"""Writes tests/golden/gyro_golden.npz from cv2 (4.13) for the gyro prediction of the LK tracks (oracle/gyro_oracle.py):

* proj_xy, proj_<case>      cv2.projectPoints of (x, y, 1), zero rvec / tvec, with the K and the distortion of every
                            camera case <case> of camera_golden.npz, over a seeded grid of normalised points
* <scene>_p0, _g            rotation scenes of tests/gyro_cases.py: cv2.goodFeaturesToTrack on frame 1 and the
                            oracle's guesses under the scene's gyro rate
* <scene>_p1, _st           calcOpticalFlowPyrLK(prev, next, p0, g, flags=OPTFLOW_USE_INITIAL_FLOW)
* <scene>_p0r, _st0, _fb    the backward call from p1 seeded with p1 + (p0 - g), and fb_err = max(|p0 - p0r|) (float32,
                            +inf unless both statuses are 1)
Frames are not stored: they regenerate from their seeds.

    python tools/make_golden_gyro.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gyro_cases  # noqa: E402
from oracle import gyro_oracle  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def camera_cases():
    """-> list of (case, K, D): the camera cases of camera_golden.npz"""
    g = np.load(os.path.join(GOLDEN, "camera_golden.npz"))
    cases = sorted({k.split("_")[0] for k in g.files if k.startswith("c") and k.endswith("_dist")}, key=lambda c: int(c[1:]))
    return [(c, g["K"], g[c + "_dist"][:int(g[c + "_n_dist"])]) for c in cases]


def proj_grid():
    rng = np.random.default_rng(7)
    return np.concatenate([rng.uniform(-0.7, 0.7, (96, 2)), [[0.0, 0.0], [0.7, 0.4], [-0.7, -0.4], [1e-9, -1e-9]]])


def scene_points(a):
    import cv2
    win, _, _ = gyro_cases.LK
    return cv2.goodFeaturesToTrack(a, gyro_cases.N_FEATURES, 0.01, 10, blockSize=7).reshape(-1, 2).astype(np.float32)


def main():
    import cv2
    out = {"cv2_version": np.array(cv2.__version__)}
    xy = proj_grid()
    out["proj_xy"] = xy
    obj = np.c_[xy, np.ones(len(xy))].reshape(-1, 1, 3)
    for c, K, D in camera_cases():
        out["proj_" + c] = cv2.projectPoints(obj, np.zeros(3), np.zeros(3), K, D if len(D) else None)[0].reshape(-1, 2)
    model = gyro_oracle.pinhole(gyro_cases.CX, gyro_cases.CY, 1.0 / gyro_cases.F, 1.0 / (gyro_cases.F * gyro_cases.DT))
    win, ml, crit = gyro_cases.LK
    for name in gyro_cases.ROTATIONS:
        a, b, w = gyro_cases.rotation_scene(name)
        p0 = scene_points(a)
        g = gyro_oracle.predict(p0, w, model)
        p1, st, _ = cv2.calcOpticalFlowPyrLK(a, b, p0.reshape(-1, 1, 2), g.reshape(-1, 1, 2).copy(), winSize=win, maxLevel=ml,
                                             criteria=crit, flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
        p1f = p1.reshape(-1, 2)
        seed = (p1f + (p0 - g)).reshape(-1, 1, 2)
        p0r, st0, _ = cv2.calcOpticalFlowPyrLK(b, a, p1, seed, winSize=win, maxLevel=ml, criteria=crit,
                                               flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
        both = (st.ravel() == 1) & (st0.ravel() == 1)
        fb = np.where(both, np.abs(p0 - p0r.reshape(-1, 2)).max(-1), np.inf).astype(np.float32)
        out.update({name + "_p0": p0, name + "_g": g, name + "_p1": p1f, name + "_st": st.ravel(),
                    name + "_p0r": p0r.reshape(-1, 2), name + "_st0": st0.ravel(), name + "_fb": fb,
                    name + "_w": w})
    np.savez_compressed(os.path.join(GOLDEN, "gyro_golden.npz"), **out)


if __name__ == "__main__":
    main()
