"""Seeded scenes for the forward-backward check (oracle/fb_oracle.py, include/ofb200.h `ofb_pyrlk_fb`): shared by
tools/make_golden_fb.py (cv2 -> tests/golden/fb_golden.npz), tests/test_host_fb.py and tests/test_gpu_fb.py.

occluder_scene: an object that enters the view. synth.make_pair at 640x480 with known motion, and a foreign textured
patch (6 % of the image) pasted into the second frame only. Features inside the patch are tracked with LK status 1 to
wrong places; the check should drop them and keep the rest."""
import numpy as np

import synth

LK_SETS = {"node": ((15, 15), 3, (3, 20, 0.03)), "module": ((15, 15), 3, (3, 10, 0.5))}
OCCLUDER_LK = ((15, 15), 3, (3, 20, 0.03))
OCCLUDER_T = 0.5
OCCLUDER_SEEDS = range(6)
GOLDEN_T = 1.0


def occluder_scene(k, h=480, w=640, occ_frac=0.06):
    """-> (prev, next, motion dict, patch (x0, y0, ow, oh))"""
    a, b, mo = synth.make_pair(h, w, k, 10 + k)
    b = b.copy()
    rng = np.random.default_rng(k)
    oh, ow = int(h * np.sqrt(occ_frac)), int(w * np.sqrt(occ_frac))
    y0, x0 = int(rng.integers(0, h - oh)), int(rng.integers(0, w - ow))
    b[y0:y0 + oh, x0:x0 + ow] = synth.texture(oh, ow, 77 + k)
    return a, b, mo, (x0, y0, ow, oh)


def patch_masks(p0, patch, margin=20):
    """(inside the patch, farther than `margin` px from it) for the starting points p0"""
    x0, y0, ow, oh = patch
    q = np.asarray(p0, np.float32).reshape(-1, 2)
    inside = (q[:, 0] >= x0) & (q[:, 0] < x0 + ow) & (q[:, 1] >= y0) & (q[:, 1] < y0 + oh)
    near = (q[:, 0] >= x0 - margin) & (q[:, 0] < x0 + ow + margin) & (q[:, 1] >= y0 - margin) & (q[:, 1] < y0 + oh + margin)
    return inside, ~near


def velocity_error(p0, p1, keep, mo):
    """relative max-norm error of the node-variant solve on the kept tracks against the true velocity"""
    from oracle import velocity_oracle as vo
    n1 = np.asarray(p1, np.float32).reshape(-1, 2)[keep]
    n0 = np.asarray(p0, np.float32).reshape(-1, 2)[keep]
    x = (n1.astype(np.float64) - [mo["cx"], mo["cy"]]) / mo["f"]
    u = (n1 - n0).astype(np.float64) / (mo["f"] * mo["dt"])
    v = vo.solve_lgs(x, u, mo["d"], mo["n"], mo["w"], variant="node")[0]
    return np.abs(v - mo["v"]).max() / np.abs(mo["v"]).max()


def border_scene():
    """-> (prev, next, points): a shifted, slightly rotated pair and points on and next to every border, so that some
    forward or backward tracks leave the image"""
    a, b = synth.affine_pair(240, 320, 5, shift=(4.5, -3.0), rot=0.01)
    xs = np.array([0.0, 0.5, 2.0, 6.0, 160.0, 313.0, 317.5, 319.0])
    ys = np.array([0.0, 1.5, 5.0, 120.0, 233.0, 238.0, 239.0])
    pts = np.stack(np.meshgrid(xs, ys), -1).reshape(-1, 2).astype(np.float32)
    return a, b, pts.reshape(-1, 1, 2)
