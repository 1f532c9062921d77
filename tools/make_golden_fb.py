"""Writes tests/golden/fb_golden.npz: the forward-backward check of OpenCV's samples/python/lk_track.py run with cv2
(two calcOpticalFlowPyrLK calls) on seeded scenes (tests/fb_cases.py). Per case `<tag>_`: p0 (starting points), p1, st
(forward), p0r, st0 (backward from p1), fb_err = max(|p0 - p0r|) (float32, +inf unless both statuses are 1) and T.
Frames are not stored: the cv2_golden.npz pairs are read from that file, the others regenerate from their seeds.

    python tools/make_golden_fb.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import fb_cases  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def golden_inputs():
    """-> list of (tag, prev, next, p0, (win, max_level, criteria), T): the cases of fb_golden.npz"""
    g = np.load(os.path.join(GOLDEN, "cv2_golden.npz"))
    out = []
    for name in ("real", "c1", "odd"):
        for ls, lk in fb_cases.LK_SETS.items():
            out.append(("%s_%s" % (name, ls), g[name + "_prev"], g[name + "_next"], g["%s_gftt_bench" % name], lk,
                        fb_cases.GOLDEN_T))
    a, b, pts = fb_cases.border_scene()
    out.append(("border", a, b, pts, fb_cases.LK_SETS["node"], fb_cases.GOLDEN_T))
    return out


def occluder_points(a):
    import cv2
    return cv2.goodFeaturesToTrack(a, 500, 0.01, 10, blockSize=7)


def run_cv2(a, b, p0, lk, T):
    import cv2
    win, ml, crit = lk
    p1, st, _ = cv2.calcOpticalFlowPyrLK(a, b, p0, None, winSize=win, maxLevel=ml, criteria=crit)
    p0r, st0, _ = cv2.calcOpticalFlowPyrLK(b, a, p1, None, winSize=win, maxLevel=ml, criteria=crit)
    both = (st.ravel() == 1) & (st0.ravel() == 1)
    fb = np.where(both, np.abs(p0 - p0r).reshape(-1, 2).max(-1), np.inf).astype(np.float32)
    return dict(p0=p0, p1=p1, st=st, p0r=p0r, st0=st0, fb_err=fb, T=np.float64(T))


def main():
    import cv2
    out = {"cv2_version": np.array(cv2.__version__)}
    cases = golden_inputs()
    for k in fb_cases.OCCLUDER_SEEDS:
        a, b, _, _ = fb_cases.occluder_scene(k)
        cases.append(("occluder%d" % k, a, b, occluder_points(a), fb_cases.OCCLUDER_LK, fb_cases.OCCLUDER_T))
    for tag, a, b, p0, lk, T in cases:
        for key, v in run_cv2(a, b, np.asarray(p0, np.float32).reshape(-1, 1, 2), lk, T).items():
            out["%s_%s" % (tag, key)] = v
    np.savez_compressed(os.path.join(GOLDEN, "fb_golden.npz"), **out)


if __name__ == "__main__":
    main()
