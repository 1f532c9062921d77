"""Pins the C oracle of the image stages (oracle/of_oracle.c) to OpenCV 4.13.0: against the committed
cv2 outputs (tests/golden/cv2_golden.npz) and, where cv2 is importable, against cv2 run live with the
reference's literal parameter sets."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import image_oracle as io
import synth

FEATURE_SETS = {"node": (100, 0.7, 10, 12), "exp": (20, 0.7, 10, 7), "module": (50, 0.3, 20, 32), "bench": (200, 0.01, 10, 7)}
LK_SETS = {"node": ((15, 15), 3, (3, 20, 0.03)), "module": ((15, 15), 3, (3, 10, 0.5))}


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLDEN, "cv2_golden.npz"))


@pytest.mark.parametrize("name", ["real", "c1", "odd"])
def test_pyrdown_bit_exact(g, name):
    lv = g[name + "_prev"]
    for l in range(1, 5):
        lv = io.pyr_down(lv)
        assert np.array_equal(lv, g["%s_pyr%d" % (name, l)])


def test_bgr2gray_bit_exact(g):
    real = np.load(os.path.join(GOLDEN, "picture_test.npy"))
    assert np.array_equal(io.bgr2gray(real), g["real_gray"])


@pytest.mark.parametrize("name", ["real", "c1", "odd"])
def test_min_eig_map_close(g, name):
    img = g[name + "_prev"]
    for bs in (3, 7, 12):
        e = io.min_eig_map(img, bs)
        mx = float(g["%s_eigmax_%d" % (name, bs)])
        assert abs(e.max() - mx) <= 2e-6 * mx
        assert np.abs(e[::7, ::5] - g["%s_eigsub_%d" % (name, bs)]).max() <= 2e-6 * mx


@pytest.mark.parametrize("name", ["real", "c1", "odd"])
def test_lk_matches_cv2(g, name):
    a, b = g[name + "_prev"], g[name + "_next"]
    pts = g["%s_gftt_bench" % name]
    for ls, (win, ml, crit) in LK_SETS.items():
        nxt, st, err = io.pyrlk(a, b, pts, win, ml, crit)
        gs = g["%s_lk_%s_status" % (name, ls)]
        assert np.array_equal(st, gs)
        ok = gs.ravel() == 1
        assert np.abs(nxt - g["%s_lk_%s_next" % (name, ls)])[ok].max() <= 5e-3
        assert np.abs(err - g["%s_lk_%s_err" % (name, ls)])[ok].max() <= 5e-3


cv2 = pytest.importorskip("cv2")


@pytest.mark.parametrize("shape,seed", [((240, 320), 1), ((241, 323), 2), ((480, 640), 3)])
def test_selection_exact_on_cv2_map(shape, seed):
    """Feature SELECTION (threshold, NMS, ordering, tie rule, min-distance grid) must equal cv2's
    exactly when both start from cv2's own lambda_min map."""
    img = synth.texture(shape[0], shape[1], seed)
    for mc, q, md, bs in list(FEATURE_SETS.values()) + [(0, 0.05, 0, 3), (300, 0.02, 7.5, 5), (50, 0.01, 1.0, 3)]:
        ce = cv2.cornerMinEigenVal(img, bs)
        ours = io.select_features(ce, mc, q, md)
        ref = cv2.goodFeaturesToTrack(img, mc, q, md, blockSize=bs)
        if ref is None:
            assert ours is None
        else:
            assert np.array_equal(ours, ref), (mc, q, md, bs)


def test_selection_mask_and_ties():
    img = synth.texture(240, 320, 5)
    mask = np.ones_like(img)
    mask[60:140, 100:220] = 0
    ce = cv2.cornerMinEigenVal(img, 7)
    assert np.array_equal(io.select_features(ce, 100, 0.01, 10, mask), cv2.goodFeaturesToTrack(img, 100, 0.01, 10, mask=mask, blockSize=7))
    # exact ties: a periodic pattern repeats the same lambda_min many times
    yy, xx = np.mgrid[0:128, 0:160]
    tie = (((xx // 8) + (yy // 8)) % 2 * 200).astype(np.uint8)
    ce = cv2.cornerMinEigenVal(tie, 3)
    ref = cv2.goodFeaturesToTrack(tie, 0, 0.5, 5, blockSize=3)
    assert np.array_equal(io.select_features(ce, 0, 0.5, 5), ref)
    # all-zero mask / flat image -> None
    assert io.select_features(ce, 10, 0.5, 5, np.zeros_like(tie)) is None
    assert io.good_features(np.full((50, 60), 7, np.uint8), 10, 0.01, 5) is None


@pytest.mark.parametrize("case", ["shift40", "halfflat", "small_nonsquare", "border"])
def test_lk_edge_cases_live(case):
    if case == "shift40":
        a = synth.texture(240, 320, 7); b = np.roll(a, 40, axis=1)
        pts = cv2.goodFeaturesToTrack(a, 80, 0.01, 10, blockSize=7); kw = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
    elif case == "halfflat":
        a = synth.texture(240, 320, 8); a[:, 160:] = 128; b = np.roll(a, 2, axis=0)
        yy, xx = np.mgrid[20:220:25, 20:300:28]; pts = np.stack([xx.ravel(), yy.ravel()], 1).astype(np.float32).reshape(-1, 1, 2)
        kw = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
    elif case == "small_nonsquare":
        a, b = synth.affine_pair(50, 70, 9, shift=(1.2, 0.7), rot=0.0, scale=1.0)
        pts = cv2.goodFeaturesToTrack(a, 30, 0.01, 5, blockSize=3); kw = dict(winSize=(21, 11), maxLevel=4, criteria=(3, 30, 0.01))
    else:
        a, b = synth.affine_pair(120, 160, 10, shift=(-2.5, 3.5))
        pts = np.array([[0, 0], [1.5, 2.5], [159, 119], [158.2, 3.3], [4, 117.5], [80, 0.4], [0.2, 60]], np.float32).reshape(-1, 1, 2)
        kw = dict(winSize=(15, 15), maxLevel=2, criteria=(3, 20, 0.03))
    n2, s2, e2 = cv2.calcOpticalFlowPyrLK(a, b, pts, None, **kw)
    n1, s1, e1 = io.pyrlk(a, b, pts, kw["winSize"], kw["maxLevel"], kw["criteria"])
    assert np.array_equal(s1, s2)
    ok = s2.ravel() == 1
    if ok.any():
        assert np.abs(n1 - n2)[ok].max() <= 0.05
        assert np.abs(e1 - e2)[ok].max() <= 0.05


def test_feature_lists_vs_live_cv2_with_tie_rule():
    """End to end on the CPU: the oracle's own lists (lambda_min from exact integer window sums + OpenCV's selection
    rule) against cv2.goodFeaturesToTrack, the reference's literal parameter sets and the bench ones, up to 1080p.
    Every difference must be a reordering of corners that tie to 2^-20 of the maximum on cv2's own map (tie_rule.py);
    the golden lists from cv2 4.13 are checked the same way."""
    from tie_rule import explain_by_ties
    ties = total = 0
    for (h, w), seed in [((240, 320), 1), ((241, 323), 2), ((480, 640), 3), ((720, 1280), 4), ((1080, 1920), 5), ((1080, 1920), 7)]:
        img = synth.texture(h, w, seed)
        for mc, q, md, bs in [(200, 0.01, 10, 7), (1000, 0.01, 10, 7), (5000, 0.01, 10, 7), (100, 0.7, 10, 12), (50, 0.3, 20, 32),
                              (20, 0.7, 10, 7)]:
            ref = cv2.goodFeaturesToTrack(img, mc, q, md, blockSize=bs)
            ties += explain_by_ties(io.good_features(img, mc, q, md, block_size=bs), ref, cv2.cornerMinEigenVal(img, bs))
            total += 1
    assert total == 36 and ties <= 6           # 2 tie groups on these frames with cv2 4.13 (both 1080p / 5000 corners)
    # both oracle maps stay within a few ulp of cv2's; the exact-sum one is the closer of the two
    img = synth.texture(241, 323, 2)
    for bs in (3, 7, 12, 32):
        e = cv2.cornerMinEigenVal(img, bs)
        d_exact = np.abs(io.min_eig_map(img, bs) - e).max() / e.max()
        d_f32 = np.abs(io.min_eig_map(img, bs, fp32_sums=True) - e).max() / e.max()
        assert d_exact <= 2e-6 and d_f32 <= 4e-6, (bs, d_exact, d_f32)


def _lk_edge_cases():
    import lk_edge_cases as lc
    tex = lc.texture_scene()
    for win in lc.FAST_WINDOWS + lc.BOUNDARY_WINDOWS + lc.GENERIC_WINDOWS:
        yield "texture", tex, win, 3, lc.CRIT, 1e-4, False
    wide = lc.wide_scene()
    for win in lc.SMEM_WINDOWS:
        yield "wide", wide, win, 3, lc.CRIT, 1e-4, False
    for cell in lc.CHECKER_CELLS:
        for shift in lc.CHECKER_SHIFTS:
            board = lc.checkerboard(cell, shift)
            for win in lc.CHECKER_WINDOWS:
                for ml in (0, 2):
                    yield ("checkerboard", cell, shift), board, win, ml, lc.CRIT, 1e-4, lc.chaotic_checkerboard(cell, shift)
    for h, w in lc.TINY_SIZES:
        tiny = lc.tiny_scene(h, w)
        for win in lc.TINY_WINDOWS:
            for ml in (0, 3):
                yield ("tiny", h, w), tiny, win, ml, lc.CRIT, 1e-4, False
    crit = lc.criteria_scene()
    for c, me in lc.CRITERIA_CASES:
        for win in ((15, 15), (21, 21)):
            yield "criteria", crit, win, 3, c, me, False
    for (h, w), seed in (((1080, 1920), 44), ((97, 1003), 45)):
        scene = lc.depth_scene(h, w, seed)
        for win in ((15, 15), (21, 21), (3, 41), (61, 3)):
            for ml in list(range(9)) + [20]:
                yield ("depth", h, w), scene, win, ml, lc.CRIT, 1e-4, False


def test_lk_edge_inputs_pinned_to_cv2():
    """The inputs of test_gpu_lk_edges.py, oracle against cv2 4.13: identical status everywhere; positions within
    5e-3 px and errors within lk_edge_cases.err_tol except at the points whose Newton path fp32 rounding decides
    (the two summation modes of the oracle part there by more than 5e-3; at most 1 % of the tracked points, or 2),
    status only on the checkerboards moved by half their period. The exact-sum mode is pinned to the default one
    by the same rule."""
    import lk_edge_cases as lc
    n = 0
    for what, (a, b, pts), win, ml, crit, me, chaotic in _lk_edge_cases():
        what = (what, win, ml, crit, me)
        ref = cv2.calcOpticalFlowPyrLK(a, b, pts, None, winSize=win, maxLevel=ml, criteria=crit, minEigThreshold=me)
        plain = io.pyrlk(a, b, pts, win, ml, crit, me)
        exact = io.pyrlk(a, b, pts, win, ml, crit, me, exact_sums=True)
        decided = lc.rounding_decided(plain, exact)
        if chaotic:
            assert np.array_equal(plain[1], ref[1]) and np.array_equal(exact[1], ref[1]), what
        else:
            lc.assert_close_to(plain, ref, decided, what)
            lc.assert_close_to(exact, plain, decided, what)
        n += 1
    assert n == 19 + 4 + 64 + 132 + 30 + 80


def test_lk_exact_sums_mode_where_fp32_sums_are_exact():
    """Windows of at most 8 pixels with gradients and differences of a few grey levels: every fp32 partial sum is an
    integer below 2^24, so OpenCV's running sums are exact and both oracle modes must agree to the bit (the error
    aside, which the default mode divides by 32 * npx and the exact one multiplies by its fp32 reciprocal)."""
    rng = np.random.default_rng(3)
    a = (rng.random((40, 50)) * 4).astype(np.uint8) + 100
    b = np.roll(a, 1, axis=1)
    pts = np.stack(np.meshgrid(np.arange(5, 45, 3.3), np.arange(5, 35, 2.7)), -1).astype(np.float32).reshape(-1, 1, 2)
    for win in ((3, 3), (4, 3)):
        plain = io.pyrlk(a, b, pts, win, 0, (3, 30, 0.01), 0.0)
        exact = io.pyrlk(a, b, pts, win, 0, (3, 30, 0.01), 0.0, exact_sums=True)
        assert np.array_equal(plain[0], exact[0]) and np.array_equal(plain[1], exact[1])
        assert np.abs(plain[2] - exact[2]).max() <= 1e-6 * np.abs(plain[2]).max()
