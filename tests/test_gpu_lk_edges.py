"""The LK stage at every window shape, image size, pyramid depth and stopping rule the API accepts.

ofb_lk_device runs the register-resident kernel for winW <= 16 and winH <= 15 and the shared-memory kernel for every
other window up to 4096 pixels. Both sum A, b and the error as exact integers and round each sum to fp32 once, so the
sharp bar is the oracle's exact-sum mode (image_oracle.pyrlk(..., exact_sums=True)): identical status, positions and
errors within 1e-5. cv2 4.13 run live is the second check (lk_edge_cases.assert_close_to: 5e-3 px outside the points
whose Newton path is decided by fp32 rounding). Every input is pinned oracle-against-cv2 in test_oracle_vs_cv2.py."""
import re
import os

import numpy as np
import pytest

import lk_edge_cases as lc
import synth
from conftest import ROOT
from oracle import image_oracle as io


@pytest.fixture(scope="module")
def ofb200():
    import ofb200
    return ofb200


def check(ofb200, ctx, a, b, pts, win, ml, crit=lc.CRIT, min_eig=1e-4, chaotic=False, what=""):
    """the device against the exact-sum oracle and against cv2 live; returns the device result"""
    what = (what, win, ml, crit, min_eig)
    got = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, winSize=win, maxLevel=ml, criteria=crit,
                                      minEigThreshold=min_eig, ctx=ctx)
    exact = io.pyrlk(a, b, pts, win, ml, crit, min_eig, exact_sums=True)
    lc.assert_same_as_exact(got, exact, what)
    try:
        import cv2
    except ImportError:
        return got
    ref = cv2.calcOpticalFlowPyrLK(a, b, pts, None, winSize=win, maxLevel=ml, criteria=crit, minEigThreshold=min_eig)
    if chaotic:
        assert np.array_equal(got[1], ref[1]), what
    else:
        plain = io.pyrlk(a, b, pts, win, ml, crit, min_eig)
        lc.assert_close_to(got, ref, lc.rounding_decided(plain, exact), what)
    return got


@pytest.fixture(scope="module")
def texture():
    return lc.texture_scene()


@pytest.mark.gpu
@pytest.mark.parametrize("win", lc.FAST_WINDOWS + lc.BOUNDARY_WINDOWS + lc.GENERIC_WINDOWS)
def test_window_sweep(ofb200, ctx, texture, win):
    a, b, pts = texture
    got = check(ofb200, ctx, a, b, pts, win, 3, what="texture")
    assert got[1].sum() >= 0.75 * len(pts) - 63        # every corner but a few; the border points partly


@pytest.mark.gpu
@pytest.mark.parametrize("win", lc.FAST_WINDOWS)
def test_generic_kernel_equals_fast_kernel(ofb200, ctx, monkeypatch, texture, win):
    """OFB_LK_GENERIC=1 sends the register-resident kernel's shapes to the shared-memory kernel: same integers, same
    fp32 operations, the same bits"""
    a, b, pts = texture
    kw = dict(winSize=win, maxLevel=3, criteria=lc.CRIT, ctx=ctx)
    fast = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, **kw)
    monkeypatch.setenv("OFB_LK_GENERIC", "1")
    gen = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, **kw)
    for x, y, name in zip(fast, gen, ("nextPts", "status", "err")):
        assert np.array_equal(x, y), (win, name, np.abs(x.astype(np.float64) - y).max())


@pytest.mark.gpu
@pytest.mark.parametrize("win", lc.SMEM_WINDOWS)
def test_largest_shared_memory_windows(ofb200, ctx, win):
    a, b, pts = lc.wide_scene()
    got = check(ofb200, ctx, a, b, pts, win, 3, what="wide")
    assert got[1].sum() >= len(pts) // 2


@pytest.mark.gpu
@pytest.mark.parametrize("ml", [0, 2])
@pytest.mark.parametrize("win", lc.CHECKER_WINDOWS)
def test_checkerboard_full_scale_sums(ofb200, ctx, win, ml):
    """Every pixel of a checkerboard window adds a mismatch term of the same sign near the largest the arithmetic
    allows (|diff| <= 8160 in Q5, |I'| <= 4080): the per-lane partials of b outgrow int32 for windows of more than
    2048 pixels. The 4-px board moved by (1, 0) under a 64x64 window at level 0 lands 3.7 px short with int32
    partials and status 1; cv2 and both oracle modes give x = 92.499."""
    for cell in lc.CHECKER_CELLS:
        for shift in lc.CHECKER_SHIFTS:
            a, b, pts = lc.checkerboard(cell, shift)
            got = check(ofb200, ctx, a, b, pts, win, ml, chaotic=lc.chaotic_checkerboard(cell, shift),
                        what=("checkerboard", cell, shift))
            assert got[1].all()
            if cell == 4 and shift == (1, 0) and win == (64, 64) and ml == 0:
                assert abs(float(got[0][0, 0, 0]) - 92.499) <= 1e-3, got[0][0]


def _declared_type(src, kernel, name):
    body = src[src.index(kernel):]
    m = re.search(r"\b(int|long long|unsigned int)\s+(?:\w+\s*=\s*0\s*,\s*)*" + name + r"\s*=\s*0", body)
    assert m, (kernel, name)
    return m.group(1)


def test_lane_partials_fit_their_accumulators():
    """The largest per-lane partial either LK kernel can form, over every legal window (3 <= winW, winH and
    winW * winH <= 4096), against the type the kernel declares for it. Template and warped values are Q5 (<= 255 * 32),
    so |diff| <= 8160; interpolated Scharr gradients are at most 16 * 255 = 4080 in magnitude. The shared-memory kernel
    gives each lane ceil(npx / 32) pixels; the register-resident one 8 pixels."""
    src = open(os.path.join(ROOT, "drone-stabilisation-using-optical-flow-gps-and-inertial-sensors_b200", "csrc",
                            "pyrlk.cu")).read()
    limits = {"int": 2 ** 31 - 1, "long long": 2 ** 63 - 1}
    dmax, gmax = 255 * 32, 16 * 255
    generic_px = max(-(-(w * h) // 32) for w in range(3, 4097) for h in range(3, 4096 // w + 1))
    assert generic_px == 128
    for kernel, px in (("lk_track_kernel(", generic_px), ("lk_track_fast2_kernel(", 8)):
        for name, bound in (("iA11", px * gmax * gmax), ("iA12", px * gmax * gmax), ("iA22", px * gmax * gmax),
                            ("ib1", px * dmax * gmax), ("ib2", px * dmax * gmax), ("ie", px * dmax)):
            t = _declared_type(src, kernel, name)
            assert bound <= limits[t], (kernel, name, t, bound)


@pytest.mark.gpu
@pytest.mark.parametrize("win", lc.TINY_WINDOWS)
def test_tiny_and_narrow_images(ofb200, ctx, win):
    """level 0 of images smaller than the window, down to 1x1: reflect-101 folds many times over a window"""
    for h, w in lc.TINY_SIZES:
        a, b, pts = lc.tiny_scene(h, w)
        check(ofb200, ctx, a, b, pts, win, 0, what=("tiny", h, w))
        check(ofb200, ctx, a, b, pts, win, 3, what=("tiny", h, w))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,seed", [((1080, 1920), 44), ((97, 1003), 45)])
@pytest.mark.parametrize("win", [(15, 15), (21, 21), (3, 41), (61, 3)])
def test_pyramid_depth_and_window_cut(ofb200, ctx, shape, seed, win):
    """maxLevel 0..8 and 20; (3, 41) and (61, 3) have the cut set by the height or by the width alone"""
    a, b, pts = lc.depth_scene(shape[0], shape[1], seed)
    for ml in list(range(9)) + [20]:
        check(ofb200, ctx, a, b, pts, win, ml, what=("depth", shape))


@pytest.mark.gpu
@pytest.mark.parametrize("win", [(15, 15), (31, 31)])
def test_pyramid_objects_of_other_depths(ofb200, ctx, win):
    """Pyramid objects deeper than maxLevel, and prev / next pyramids of different depths: the levels used are
    min(prev levels, next levels, maxLevel + 1), then OpenCV's window cut"""
    a, b, pts = lc.depth_scene(480, 640, 46)
    for lp, ln, ml in [(6, 6, 2), (6, 2, 4), (2, 6, 4), (0, 5, 3), (5, 1, 20), (8, 8, 8)]:
        pp, pn = ofb200.Pyramid(a, lp, ctx=ctx), ofb200.Pyramid(b, ln, ctx=ctx)
        try:
            got = ofb200.calcOpticalFlowPyrLK(pp, pn, pts, None, winSize=win, maxLevel=ml, criteria=lc.CRIT, ctx=ctx)
        finally:
            pp.close()
            pn.close()
        exact = io.pyrlk(a, b, pts, win, min(lp, ln, ml), lc.CRIT, exact_sums=True)
        lc.assert_same_as_exact(got, exact, ("pyramids", lp, ln, ml, win))


@pytest.mark.gpu
@pytest.mark.parametrize("win", [(15, 15), (21, 21)])
@pytest.mark.parametrize("crit,min_eig", lc.CRITERIA_CASES)
def test_stopping_rules_and_thresholds(ofb200, ctx, win, crit, min_eig):
    a, b, pts = lc.criteria_scene()
    got = check(ofb200, ctx, a, b, pts, win, 3, crit, min_eig, what="criteria")
    if min_eig >= 1e6:
        assert not got[1].any()
    if crit[0] & 1 and crit[1] == 0:                 # no Newton step: every tracked point stays where it started
        ok = got[1].ravel() == 1
        assert ok.any() and np.array_equal(got[0].reshape(-1, 2)[ok], pts.reshape(-1, 2)[ok])


@pytest.mark.gpu
def test_forward_backward_at_generic_windows(ofb200, ctx, texture):
    from test_gpu_fb import assert_fused_is_composition
    a, b, pts = texture
    for win in [(31, 31), (64, 64), (3, 41)]:
        for T in (0.25, 1.0):
            assert_fused_is_composition(ofb200, ctx, a, b, pts, T, winSize=win, maxLevel=3, criteria=lc.CRIT)
    a, b, pts = lc.checkerboard(4, (1, 0))
    got = assert_fused_is_composition(ofb200, ctx, a, b, pts, 0.5, winSize=(64, 64), maxLevel=0, criteria=lc.CRIT)
    assert got[1].all() and (got[3] < 0.01).all(), got[3]


@pytest.mark.gpu
@pytest.mark.parametrize("win", [(31, 31), (64, 64)])
def test_frame_pairs_generic_window_equals_per_pair_calls(ofb200, ctx, win):
    """a batch of pairs with different feature counts: the shared-memory kernel reads pair p's points at
    p * pts_stride and its count at counts[p]"""
    pairs = [synth.affine_pair(240, 320, 50 + i, shift=(2.0 + i, -1.5 * i), rot=0.01 * i) for i in range(3)]
    prev = np.stack([p[0] for p in pairs])
    nxt = np.stack([p[1] for p in pairs])
    crit = (3, 20, 0.03)
    cfg = ofb200.make_pair_cfg(320, 240, 3000, quality=0.01, min_distance=8, block_size=7, win=win, max_level=3,
                               criteria=crit)
    imu = np.zeros(3, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"] = 1.0, (0.0, 0.0, 1.0)
    res, pp, pn, st = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx)
    counts = res["n_features"].astype(int)
    assert len(set(counts.tolist())) == 3 and counts.min() > 50, counts
    for i, n in enumerate(counts):
        q, s, _ = ofb200.calcOpticalFlowPyrLK(prev[i], nxt[i], pp[i, :n], None, winSize=win, maxLevel=3, criteria=crit,
                                              ctx=ctx)
        assert np.array_equal(st[i, :n], s.ravel()) and np.array_equal(pn[i, :n], q.reshape(-1, 2)), (win, i)
        assert int(res["n_tracked"][i]) == int(s.sum())


@pytest.mark.gpu
def test_rejected_windows_leave_the_context_usable(ofb200, ctx, texture):
    a, b, pts = texture
    before = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, winSize=(21, 21), ctx=ctx)
    for win in [(2, 15), (15, 2), (64, 65), (4097, 1)]:
        with pytest.raises(ValueError):
            ofb200.calcOpticalFlowPyrLK(a, b, pts, None, winSize=win, ctx=ctx)
        with pytest.raises(ValueError):
            ofb200.track_forward_backward(a, b, pts, 1.0, winSize=win, ctx=ctx)
    after = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, winSize=(21, 21), ctx=ctx)
    for x, y in zip(before, after):
        assert np.array_equal(x, y)
