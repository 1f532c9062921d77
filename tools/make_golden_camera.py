"""Writes tests/golden/camera_golden.npz: cv2.undistortPoints / cv2.undistortPointsIter outputs (OpenCV 4.13) for the
calibrated-camera tests. One set of 400 pixel positions on and beyond a 1280x720 frame (float64, and the same rounded
to float32), then per case the lens model (0, 4, 5 or 8 coefficients, one strong enough to hit OpenCV's icdist < 0
branch), the iteration count, the optional R / P and cv2's output.

    python tools/make_golden_camera.py          (needs cv2)
"""
import os

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "camera_golden.npz")

K = np.array([[900.0, 0.0, 641.5], [0.0, 903.0, 359.25], [0.0, 0.0, 1.0]])
LENSES = {
    "none": None,
    "d4": [-0.15, 0.03, 0.0008, -0.0004],
    "d5": [-0.3, 0.12, 0.001, -0.0005, -0.02],
    "d8": [-0.3, 0.12, 0.001, -0.0005, -0.02, 0.05, 0.01, 0.002],
    "icdist": [-2.0, 0.5, 0.0, 0.0, 0.0],          # 1 + k1 r2 + ... < 0 towards the corners: cv2 falls back to (x0, y0)
}
R = cv2.Rodrigues(np.array([0.01, -0.02, 0.03]))[0]
P3 = np.array([[820.0, 0.0, 630.0], [0.0, 815.0, 355.0], [0.0, 0.0, 1.0]])
P4 = np.array([[820.0, 0.0, 630.0, -45.0], [0.0, 815.0, 355.0, 0.0], [0.0, 0.0, 1.0, 0.0]])


def main():
    rng = np.random.default_rng(2024)
    src = np.stack([rng.uniform(-60, 1340, 400), rng.uniform(-40, 760, 400)], axis=1)
    src[:4] = [[0, 0], [1279, 719], [641.5, 359.25], [1279, 0]]          # corners and the principal point
    g = dict(src=src, src32=src.astype(np.float32), K=K, cv2_version=np.array(cv2.__version__))
    cases = []
    for lens, D in LENSES.items():
        for it in (5, 20):
            cases.append((lens, D, it, None, None, "f8"))
    cases += [("d5", LENSES["d5"], 5, R, None, "f8"), ("d5", LENSES["d5"], 5, None, P3, "f8"),
              ("d8", LENSES["d8"], 20, R, P4, "f8"), ("none", None, 5, R, P3, "f8"),
              ("d5", LENSES["d5"], 5, None, None, "f4"), ("d8", LENSES["d8"], 20, R, P3, "f4")]
    for i, (lens, D, it, Rc, Pc, dt) in enumerate(cases):
        s = src if dt == "f8" else g["src32"]
        Dn = None if D is None else np.array(D)
        if it == 5:
            out = cv2.undistortPoints(s.reshape(-1, 1, 2), K, Dn, R=Rc, P=Pc)
        else:
            out = cv2.undistortPointsIter(s.reshape(-1, 1, 2), K, Dn, Rc, Pc, (cv2.TERM_CRITERIA_COUNT, it, 0))
        d = np.zeros(8)
        if D is not None:
            d[:len(D)] = D
        pre = "c%d_" % i
        g[pre + "dist"], g[pre + "n_dist"], g[pre + "iterations"] = d, np.int32(0 if D is None else len(D)), np.int32(it)
        g[pre + "R"] = np.zeros((0, 3)) if Rc is None else Rc
        g[pre + "P"] = np.zeros((0, 3)) if Pc is None else Pc
        g[pre + "f32"] = np.int32(dt == "f4")
        g[pre + "out"] = out.reshape(-1, 2)
        print(i, lens, it, Rc is not None, Pc is not None, dt, out.dtype)
    g["n_cases"] = np.int32(len(cases))
    np.savez_compressed(OUT, **g)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
