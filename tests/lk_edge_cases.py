"""Inputs of the LK edge tests (tests/test_gpu_lk_edges.py) and of their oracle pins against cv2
(tests/test_oracle_vs_cv2.py): one definition, so that the device is checked on exactly the cases the oracle was
pinned on."""
import numpy as np

from oracle import image_oracle as io
import synth

# register-resident kernel (winW <= 16, winH <= 15), the dispatch boundary, the shared-memory kernel
FAST_WINDOWS = [(3, 3), (4, 4), (5, 5), (7, 3), (3, 15), (16, 3), (9, 13), (15, 15), (16, 15)]
BOUNDARY_WINDOWS = [(17, 15), (16, 16)]
GENERIC_WINDOWS = [(21, 21), (31, 31), (32, 32), (41, 41), (51, 51), (63, 65), (65, 63), (64, 64)]
# the largest dynamic shared-memory footprints: (3, 1365) takes 229,504 B per 4-warp CTA, just under 227 KB
SMEM_WINDOWS = [(4, 1024), (1024, 4), (3, 1365), (1365, 3)]

CHECKER_CELLS = (2, 4)
CHECKER_SHIFTS = [(1, 0), (2, 0), (1, 1), (-1, 0)]
CHECKER_WINDOWS = [(45, 45), (51, 51), (64, 64), (32, 128)]

TINY_SIZES = [(1, 1), (2, 3), (5, 4), (8, 8), (9, 7), (12, 20), (20, 12), (16, 16), (17, 33), (40, 6), (6, 40)]   # (h, w)
TINY_WINDOWS = [(3, 3), (9, 13), (15, 15), (16, 15), (21, 21), (64, 64)]

CRIT = (3, 30, 0.01)


def border_points(h, w):
    """points on, just inside and just outside every edge and corner"""
    xs = [0, 0.5, 2.25, w / 2 + 0.3, w - 3.5, w - 1, w - 0.25, -1.5, w + 2.0]
    ys = [0, 1.5, h / 3 + 0.7, h - 2.25, h - 1, -2.0, h + 0.5]
    return np.array([[x, y] for x in xs for y in ys], np.float32).reshape(-1, 1, 2)


def texture_scene(h=480, w=640, seed=40, n=250):
    """an affine-warped texture, the oracle's corners and the border points"""
    a, b = synth.affine_pair(h, w, seed, shift=(2.7, -1.8), rot=0.012, scale=1.004)
    pts = np.concatenate([io.good_features(a, n, 0.01, 8, block_size=7), border_points(h, w)])
    return a, b, pts


def wide_scene():
    """a 1100x1400 pair for the windows 1024 and more pixels long"""
    a, b = synth.affine_pair(1100, 1400, 41, shift=(1.6, 2.2), rot=0.004)
    ys, xs = np.mgrid[30:1100:70, 25:1400:90]
    pts = np.stack([xs.ravel() + 0.37, ys.ravel() + 0.61], 1).astype(np.float32).reshape(-1, 1, 2)
    return a, b, np.concatenate([pts, border_points(1100, 1400)])


def checkerboard(cell, shift, h=200, w=240):
    """a calibration target moved by whole pixels: the mismatch sums of large windows are as large as the
    arithmetic allows (every pixel's gradient and difference are at full scale, with the same sign)"""
    yy, xx = np.mgrid[0:h, 0:w]
    a = (((xx // cell) + (yy // cell)) % 2 * 255).astype(np.uint8)
    b = np.ascontiguousarray(np.roll(a, shift, axis=(1, 0)))
    pts = np.array([[91.5, 91.5], [120.5, 100.5], [91.0, 91.0], [100.25, 80.75], [131.7, 97.3], [110.5, 120.5]],
                   np.float32).reshape(-1, 1, 2)
    return a, b, pts


def tiny_scene(h, w):
    """an h x w crop of a texture and the same crop moved by (2, 1), with a grid of points reaching 2 px outside"""
    big = synth.texture(h + 8, w + 8, h * 100 + w)
    a = np.ascontiguousarray(big[:h, :w])
    b = np.ascontiguousarray(big[1:h + 1, 2:w + 2])
    ys, xs = np.mgrid[-2:h + 2:1.5, -2:w + 2:1.75]
    return a, b, np.stack([xs.ravel(), ys.ravel()], 1).astype(np.float32).reshape(-1, 1, 2)


def depth_scene(h, w, seed):
    a, b = synth.affine_pair(h, w, seed, shift=(5.5, -4.25), rot=0.008)
    pts = np.concatenate([io.good_features(a, 300, 0.01, 10, block_size=7), border_points(h, w)])
    return a, b, pts


def criteria_scene():
    a, b = synth.affine_pair(240, 320, 43, shift=(3.3, -2.6), rot=0.01)
    return a, b, np.concatenate([io.good_features(a, 120, 0.01, 8, block_size=7), border_points(240, 320)])


# (criteria, minEigThreshold): the clamps of maxCount and eps, the fp64 fall-back of the fp32 eps bracket (eps = 1e-20),
# a type without COUNT (30 iterations) or without EPS (eps 0.01), and minEigThreshold from 0 to everything lost
CRITERIA_CASES = [((3, 0, 0.01), 1e-4), ((3, 1, 0.01), 1e-4), ((3, 100, 0.01), 1e-4), ((3, 1000, 0.0), 1e-4),
                  ((3, 30, 0.0), 1e-4), ((3, 30, 1e-20), 1e-4), ((3, 30, 0.03), 1e-4), ((3, 30, 50.0), 1e-4),
                  ((1, 5, 0.5), 1e-4), ((2, 5, 0.5), 1e-4), ((1, 1000, 50.0), 1e-4), ((2, 0, 1e-20), 1e-4),
                  ((3, 20, 0.03), 0.0), ((3, 20, 0.03), 1e-2), ((3, 20, 0.03), 1e6)]


# Two summation orders of the same fp32 arithmetic (OpenCV's running sums and exact integer sums) can send a track
# down different Newton paths where an exit test (eps, the oscillation rule, the window bounds) is decided by the last
# bit of b: a "rounding-decided" point. Both results are then equally faithful to OpenCV, and cv2's own SIMD order can
# take a third path, so positions at such points are compared with nothing but their status. Elsewhere the 5e-3 px
# bar applies. A checkerboard moved by half its period (2-px cells by (2, 0) or (1, 1)) has no unique solution at all;
# there every point can be rounding-decided.
POS_TOL = 5e-3


def err_tol(dpos, err):
    """the L1 error is 255-Lipschitz in the position (one grey level per 1/255 px at a full-scale edge), so a position
    within dpos carries an error within 255 * dpos; any position change, however small, can flip the Q14 weights'
    and the Q5 values' rounding, by at most 1 per pixel, which moves the error by at most 1/32; OpenCV's running fp32
    sum of up to 4096 terms adds up to 4096 * 2^-24 < 2.5e-4 of the error's size"""
    return 1.0 / 32 + 255.0 * dpos + 2.5e-4 * np.abs(err)


def point_dist(p, q):
    return np.abs(np.asarray(p, np.float64) - np.asarray(q, np.float64)).reshape(-1, 2).max(1)


def rounding_decided(plain, exact):
    return point_dist(plain[0], exact[0]) > POS_TOL


def assert_close_to(got, ref, decided, what):
    """identical status; positions within 5e-3 px and errors within err_tol at the points `decided` does not flag;
    at most 1 % (and 2) of the tracked points flagged"""
    st, rs = np.asarray(got[1]).ravel(), np.asarray(ref[1]).ravel()
    assert np.array_equal(st, rs), (what, "status", np.nonzero(st != rs)[0][:10])
    ok = rs == 1
    assert (decided & ok).sum() <= max(2, 0.01 * ok.sum()), (what, "rounding-decided points", int((decided & ok).sum()))
    sel = ok & ~decided
    d = point_dist(got[0], ref[0])
    assert (d[sel] <= POS_TOL).all(), (what, "position", float(d[sel].max()), np.nonzero(sel & (d > POS_TOL))[0][:10])
    with np.errstate(invalid="ignore", over="ignore"):         # (cv2 leaves the error of a lost point unset)
        re_ = np.asarray(ref[2], np.float64).ravel()
        de = np.abs(np.asarray(got[2], np.float64).ravel() - re_)
    tol = err_tol(d[sel], re_[sel])
    assert (de[sel] <= tol).all(), (what, "err", float((de[sel] - tol).max()))


def assert_same_as_exact(got, exact, what, tol=1e-5):
    """the device against the exact-sum oracle: the same integers rounded once to fp32 in the same order of
    operations, so the same Newton path: identical status, positions and errors within 1e-5"""
    st, es = np.asarray(got[1]).ravel(), np.asarray(exact[1]).ravel()
    assert np.array_equal(st, es), (what, "status", np.nonzero(st != es)[0][:10], st[st != es][:10])
    ok = es == 1
    if ok.any():
        d = point_dist(got[0], exact[0])[ok]
        assert d.max() <= tol, (what, "position", float(d.max()), np.nonzero(ok)[0][np.argmax(d)])
        de = np.abs(np.asarray(got[2], np.float64) - np.asarray(exact[2], np.float64)).ravel()[ok]
        assert de.max() <= tol, (what, "err", float(de.max()))


def chaotic_checkerboard(cell, shift):
    return cell == 2 and tuple(shift) in ((2, 0), (1, 1))
