"""GPU parity, stages 0-3 (through the C ABI) against the C oracle, the committed cv2 4.13 outputs and
cv2 live (the GPU box runs the same image). Bars (BASELINE.md 4): pyramid bit-exact; feature lists equal
as ordered lists except documented float ties; LK <= 0.05 px with identical status."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import image_oracle as io
import synth

pytestmark = pytest.mark.gpu

FEATURE_SETS = {"node": (100, 0.7, 10, 12), "exp": (20, 0.7, 10, 7), "module": (50, 0.3, 20, 32), "bench": (200, 0.01, 10, 7)}
LK_SETS = {"node": ((15, 15), 3, (3, 20, 0.03)), "module": ((15, 15), 3, (3, 10, 0.5))}


def half_trace_max(img, bs):
    """max over the image of a+c = (S_xx+S_yy)/2 in cornerMinEigenVal's units, from exact integer sums."""
    p = np.pad(img.astype(np.int64), 1, mode="reflect")
    gx = (p[:-2, 2:] - p[:-2, :-2]) + 2 * (p[1:-1, 2:] - p[1:-1, :-2]) + (p[2:, 2:] - p[2:, :-2])
    gy = (p[2:, :-2] + 2 * p[2:, 1:-1] + p[2:, 2:]) - (p[:-2, :-2] + 2 * p[:-2, 1:-1] + p[:-2, 2:])
    e = gx * gx + gy * gy
    a0 = bs // 2
    q = np.pad(e, ((a0, bs - 1 - a0), (a0, bs - 1 - a0)), mode="reflect")
    c = np.pad(np.cumsum(np.cumsum(q, 0), 1), ((1, 0), (1, 0)))
    S = c[bs:, bs:] - c[:-bs, bs:] - c[bs:, :-bs] + c[:-bs, :-bs]
    return 0.5 * float(S.max()) * (1.0 / (4 * 255 * bs)) ** 2


def tie_tol(img, bs):
    """Documented float tie (DESIGN.md): lambda_min = (a+c) - sqrt(..) carries the fp32 rounding of a+c, and
    OpenCV's box filter adds ~blockSize ulps of summation-order noise, so two correct fp32 maps differ by up
    to 2*blockSize*2^-23*max(a+c). The GPU map is built from EXACT integer sums (no summation noise)."""
    return 2.0 * bs * 2.0 ** -23 * max(half_trace_max(img, bs), 1e-30)


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLDEN, "cv2_golden.npz"))


def as_list(p):
    return np.zeros((0, 2), np.float32) if p is None else np.asarray(p).reshape(-1, 2)


def min_eig_map_unaligned(ofb200, ctx, img, bs):
    """cornerMinEigenVal of a device copy of img that starts 1 byte past an aligned address and has an odd pitch: every
    strip of the marching kernel then takes its general row loop (the lean loops need 4-byte-aligned rows)."""
    import torch
    h, w = img.shape
    pitch = w + 1 + w % 2
    host = np.zeros(1 + h * pitch, np.uint8)
    host[1:].reshape(h, pitch)[:, :w] = img
    dev = torch.from_numpy(host).cuda()
    torch.cuda.synchronize()
    out = np.empty((h, w), np.float32)
    ofb200._lib.check(ctx.lib.ofb_min_eig_map(ctx.h, ofb200._lib.ptr(dev.data_ptr() + 1), w, h, pitch, bs, ofb200._lib.ptr(out)))
    return out


from tie_rule import TIE_REL, cv2_eig, explain_by_ties  # noqa: E402,F401


def check_features(ofb200, ctx, img, mc, q, md, bs, mask=None, ref=None):
    """The contract, all three parts asserted: (i) the GPU list is OpenCV's selection rule applied EXACTLY to the GPU's
    lambda_min map; (ii) that map is within the tie tolerance of the oracle map; (iii) against a cv2 list, any difference
    is a reordering of corners whose lambda_min on cv2's own map tie to 2^-20 of the maximum (explain_by_ties).
    Returns the number of tie groups needed (0 = byte-identical to cv2)."""
    got = as_list(ofb200.goodFeaturesToTrack(img, mc, q, md, mask=mask, blockSize=bs, ctx=ctx))
    eig = ofb200.cornerMinEigenVal(img, bs, ctx=ctx)
    expect = as_list(io.select_features(eig, mc, q, md, mask))
    assert np.array_equal(got, expect), "selection differs from OpenCV's rule on the GPU's own map"
    oeig = io.min_eig_map(img, bs)
    assert np.abs(eig - oeig).max() <= tie_tol(img, bs), "lambda_min map outside tie tolerance"
    if ref is not None:
        return explain_by_ties(got, ref, cv2_eig(img, bs))
    return 0


@pytest.mark.parametrize("name", ["real", "c1", "odd"])
def test_pyramid_bit_exact_vs_cv2_golden(ctx, g, name):
    import ofb200
    lv = ofb200.buildPyramid(g[name + "_prev"], 4, ctx=ctx)
    assert len(lv) == 5
    for l in range(1, 5):
        assert np.array_equal(lv[l], g["%s_pyr%d" % (name, l)]), (name, l)


@pytest.mark.parametrize("shape", [(1, 1), (2, 3), (5, 4), (17, 33), (63, 129), (64, 128), (65, 131), (240, 320), (1080, 1920)])
def test_pyramid_shapes_vs_oracle(ctx, shape):
    import ofb200
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    lv = ofb200.buildPyramid(img, 6, ctx=ctx)
    ref = io.build_pyramid(img, len(lv) - 1)
    for a, b in zip(lv, ref):
        assert a.shape == b.shape and np.array_equal(a, b)


def test_pyramid_batch_and_checksum_at_full_size(ctx):
    """Batch of 1080p frames: every image's levels equal the single-image result (size-independent
    property) and level 1 of a constant image stays constant."""
    import ofb200
    rng = np.random.default_rng(5)
    imgs = rng.integers(0, 256, (3, 1080, 1920), dtype=np.uint8)
    imgs[2] = 137
    p = ofb200.Pyramid(imgs, 4, ctx=ctx)
    for i in range(3):
        single = ofb200.buildPyramid(imgs[i], 4, ctx=ctx)
        for l in range(5):
            assert np.array_equal(p.level(l, i), single[l])
    assert np.all(p.level(4, 2) == 137)
    assert np.array_equal(p.level(1, 0), io.pyr_down(imgs[0]))
    p.close()


def test_bgr2gray(ctx, g):
    import ofb200
    real = np.load(os.path.join(GOLDEN, "picture_test.npy"))
    assert np.array_equal(ofb200.cvtColor(real, ofb200.COLOR_BGR2GRAY, ctx=ctx), g["real_gray"])
    rng = np.random.default_rng(0)
    bgr = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    assert np.array_equal(ofb200.cvtColor(bgr, ctx=ctx), io.bgr2gray(bgr))


@pytest.mark.parametrize("name", ["real", "c1", "odd"])
def test_features_vs_cv2_golden(ctx, g, name):
    import ofb200
    img = g[name + "_prev"]
    for fs, (mc, q, md, bs) in FEATURE_SETS.items():
        # every difference from cv2's committed list must be explained by ties on cv2's own map (asserted inside)
        check_features(ofb200, ctx, img, mc, q, md, bs, ref=g["%s_gftt_%s" % (name, fs)])


def test_features_masked_and_edge_cases(ctx, g):
    import ofb200
    img = g["c1_prev"]
    check_features(ofb200, ctx, img, 80, 0.01, 10, 7, mask=g["c1_mask"], ref=g["c1_gftt_masked"])
    # unlimited corners, no min distance; non-integer distance; distance 1
    for mc, q, md, bs in [(0, 0.05, 0, 3), (300, 0.02, 7.5, 5), (50, 0.01, 1.0, 3), (5000, 0.001, 3, 3), (0, 0.2, 12, 7)]:
        check_features(ofb200, ctx, img, mc, q, md, bs)
    # flat image and all-zero mask -> None, as cv2
    assert ofb200.goodFeaturesToTrack(np.full((50, 60), 7, np.uint8), 10, 0.01, 5, ctx=ctx) is None
    assert ofb200.goodFeaturesToTrack(img, 10, 0.01, 5, mask=np.zeros_like(img), ctx=ctx) is None
    # exact ties (periodic pattern): ordering rule "larger address first"
    yy, xx = np.mgrid[0:128, 0:160]
    tie = (((xx // 8) + (yy // 8)) % 2 * 200).astype(np.uint8)
    check_features(ofb200, ctx, tie, 0, 0.5, 5, 3)
    check_features(ofb200, ctx, tie, 40, 0.5, 0, 3)
    with pytest.raises(ValueError):
        ofb200.goodFeaturesToTrack(img.astype(np.float32), 10, 0.01, 5, ctx=ctx)
    with pytest.raises(ValueError):
        ofb200.goodFeaturesToTrack(img, 10, 0.01, 5, blockSize=99, ctx=ctx)


def test_features_live_cv2_many_sizes(ctx):
    import ofb200
    cv2 = pytest.importorskip("cv2")
    ties = total = 0
    for (h, w), seed in [((240, 320), 1), ((241, 323), 2), ((480, 640), 3), ((720, 1280), 4), ((1080, 1920), 5),
                         ((1080, 1920), 6), ((1080, 1920), 7), ((720, 1280), 8)]:
        img = synth.texture(h, w, seed)
        for mc, q, md, bs in [(200, 0.01, 10, 7), (500, 0.01, 10, 7), (1000, 0.01, 10, 7), (100, 0.7, 10, 12), (50, 0.3, 20, 32)]:
            ref = cv2.goodFeaturesToTrack(img, mc, q, md, blockSize=bs)
            ties += check_features(ofb200, ctx, img, mc, q, md, bs, ref=ref)      # asserts the tie rule for every difference
            total += 1
    print("feature lists vs live cv2: %d cases, %d tie groups" % (total, ties))


def test_tie_checker_rejects_real_differences():
    """The checker itself: a swap of two corners cv2 tells apart, a substituted corner and a count mismatch must fail;
    a swap inside the tolerance passes."""
    lam = np.zeros((10, 10), np.float32)
    lam[1, 1], lam[2, 2], lam[3, 3], lam[4, 4] = 1.0, 0.5, 0.5 * (1 + 2.0 ** -22), 0.25
    a = np.array([[1, 1], [3, 3], [2, 2], [4, 4]], np.float32)
    assert explain_by_ties(a, a.copy(), lam) == 0
    assert explain_by_ties(a[[0, 2, 1, 3]], a, lam) == 1                       # 0.5 vs 0.5(1+2^-22): a tie
    for bad in (a[[1, 0, 2, 3]], a[[0, 1, 3, 2]], np.array([[1, 1], [3, 3], [2, 2], [5, 5]], np.float32), a[:3]):
        with pytest.raises(AssertionError):
            explain_by_ties(bad, a, lam)


def test_c5_shape_against_live_cv2(ctx):
    """BASELINE config 5 geometry -- 1280x720, 500 features, maxLevel 3 -- against cv2 itself on three streams:
    feature lists (tie rule), LK status and positions, and the velocity of the fused call against the fp64 NumPy solve
    on cv2's own tracks."""
    import ofb200
    from oracle import velocity_oracle as vo
    cv2 = pytest.importorskip("cv2")
    kw = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
    for s in range(3):
        a, b, mo = synth.make_pair(720, 1280, s, 300 + s)
        ref = cv2.goodFeaturesToTrack(a, 500, 0.01, 10, blockSize=7)
        check_features(ofb200, ctx, a, 500, 0.01, 10, 7, ref=ref)
        rn, rs, re_ = cv2.calcOpticalFlowPyrLK(a, b, ref, None, **kw)
        n, st, e = ofb200.calcOpticalFlowPyrLK(a, b, ref, None, ctx=ctx, **kw)
        assert np.array_equal(st, rs)
        ok = rs.ravel() == 1
        assert ok.sum() >= 450 and np.abs(n - rn)[ok].max() <= 0.05 and np.abs(e - re_)[ok].max() <= 0.05
        cfg = ofb200.make_pair_cfg(1280, 720, 500, 0.01, 10, 7, (15, 15), 3, (3, 20, 0.03), variant="node",
                                   principal=(mo["cx"], mo["cy"]), pos_scale=1.0 / mo["f"], flow_scale=1.0 / (mo["f"] * mo["dt"]))
        imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
        imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
        res, pp, pn, stt = ofb200.frame_pairs(a[None], b[None], imu, cfg, want_tracks=True, ctx=ctx)
        k = int(res["n_features"][0])
        explain_by_ties(pp[0, :k], ref, cv2.cornerMinEigenVal(a, 7))
        # velocity: the reference's solve on cv2's tracks of cv2's corners
        newp = rn.reshape(-1, 2)[ok]
        x = (newp.astype(np.float64) - np.array([mo["cx"], mo["cy"]])) / mo["f"]
        u = (newp - ref.reshape(-1, 2)[ok]).astype(np.float64) / (mo["f"] * mo["dt"])
        v_ref = vo.solve_lgs(x, u, mo["d"], mo["n"], mo["w"], variant="node")[0]
        # (LK positions agree to <= 0.05 px, typically 1e-4: the velocities agree far inside the 5 % truth band)
        assert np.abs(res["v"][0] - v_ref).max() <= 2e-3 * max(1.0, np.abs(v_ref).max()), (res["v"][0], v_ref)
        okg = stt[0, :k] == 1
        xg = (pn[0, :k][okg].astype(np.float64) - np.array([mo["cx"], mo["cy"]])) / mo["f"]
        ug = (pn[0, :k][okg] - pp[0, :k][okg]).astype(np.float64) / (mo["f"] * mo["dt"])
        v_same = vo.solve_lgs(xg, ug, mo["d"], mo["n"], mo["w"], variant="node")[0]
        assert np.abs(res["v"][0] - v_same).max() <= 1e-4 * np.abs(v_same).max()      # the 1e-4 contract, identical inputs


@pytest.mark.parametrize("name", ["real", "c1", "odd"])
def test_lk_vs_cv2_golden(ctx, g, name):
    import ofb200
    a, b = g[name + "_prev"], g[name + "_next"]
    pts = g["%s_gftt_bench" % name]
    for ls, (win, ml, crit) in LK_SETS.items():
        nxt, st, err = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, winSize=win, maxLevel=ml, criteria=crit, ctx=ctx)
        gs = g["%s_lk_%s_status" % (name, ls)]
        assert nxt.shape == pts.shape and st.shape == gs.shape and st.dtype == np.uint8 and nxt.dtype == np.float32
        assert np.array_equal(st, gs), (name, ls, int((st != gs).sum()))
        ok = gs.ravel() == 1
        dpos = np.abs(nxt - g["%s_lk_%s_next" % (name, ls)])[ok].max()
        assert dpos <= 0.05, dpos
        assert np.abs(err - g["%s_lk_%s_err" % (name, ls)])[ok].max() <= 0.05
        # and the tighter, informative bound against the scalar oracle (same arithmetic, exact sums)
        on, os_, oe = io.pyrlk(a, b, pts, win, ml, crit)
        assert np.array_equal(st, os_)
        assert np.abs(nxt - on)[ok].max() <= 5e-3


@pytest.mark.parametrize("case", ["shift40", "halfflat", "small_nonsquare", "border", "win21", "initial_flow"])
def test_lk_edge_cases(ctx, case):
    import ofb200
    flags = 0
    init = None
    if case == "shift40":
        a = synth.texture(240, 320, 7); b = np.roll(a, 40, axis=1)
        pts = io.good_features(a, 80, 0.01, 10, block_size=7); kw = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
    elif case == "halfflat":
        a = synth.texture(240, 320, 8); a[:, 160:] = 128; b = np.roll(a, 2, axis=0)
        yy, xx = np.mgrid[20:220:25, 20:300:28]; pts = np.stack([xx.ravel(), yy.ravel()], 1).astype(np.float32).reshape(-1, 1, 2)
        kw = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
    elif case == "small_nonsquare":
        a, b = synth.affine_pair(50, 70, 9, shift=(1.2, 0.7), rot=0.0, scale=1.0)
        pts = io.good_features(a, 30, 0.01, 5, block_size=3); kw = dict(winSize=(21, 11), maxLevel=4, criteria=(3, 30, 0.01))
    elif case == "border":
        a, b = synth.affine_pair(120, 160, 10, shift=(-2.5, 3.5))
        pts = np.array([[0, 0], [1.5, 2.5], [159, 119], [158.2, 3.3], [4, 117.5], [80, 0.4], [0.2, 60], [-3, 50], [170, 60]],
                       np.float32).reshape(-1, 1, 2)
        kw = dict(winSize=(15, 15), maxLevel=2, criteria=(3, 20, 0.03))
    elif case == "win21":
        a, b = synth.affine_pair(240, 320, 11, shift=(4.2, -3.1))
        pts = io.good_features(a, 60, 0.01, 10, block_size=7); kw = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    else:
        a, b = synth.affine_pair(240, 320, 12, shift=(6.0, 5.0))
        pts = io.good_features(a, 40, 0.01, 10, block_size=7); kw = dict(winSize=(15, 15), maxLevel=0, criteria=(3, 20, 0.03))
        flags = 4
        init = pts + np.float32([5.5, 4.5])
    if case == "initial_flow":
        cv2 = pytest.importorskip("cv2")
        rn, rs, re_ = cv2.calcOpticalFlowPyrLK(a, b, pts, init.copy(), flags=flags, **kw)
    else:
        rn, rs, re_ = io.pyrlk(a, b, pts, kw["winSize"], kw["maxLevel"], kw["criteria"])
    n, s, e = ofb200.calcOpticalFlowPyrLK(a, b, pts, None if init is None else init.copy(), flags=flags, ctx=ctx, **kw)
    assert np.array_equal(s, rs), (case, s.ravel(), rs.ravel())
    ok = rs.ravel() == 1
    if ok.any():
        assert np.abs(n - rn)[ok].max() <= 0.05
        assert np.abs(e - re_)[ok].max() <= 0.05
    # empty point set
    n0, s0, e0 = ofb200.calcOpticalFlowPyrLK(a, b, np.zeros((0, 1, 2), np.float32), None, ctx=ctx, **kw)
    assert n0.shape == (0, 1, 2) and s0.shape == (0, 1)


def test_lk_live_cv2_1080p(ctx):
    """BASELINE config 2 geometry: 1080p, 1000 features, maxLevel 4, against cv2 itself."""
    import ofb200
    cv2 = pytest.importorskip("cv2")
    a, b, mo = synth.make_pair(1080, 1920, 0, 0)
    pts = cv2.goodFeaturesToTrack(a, 1000, 0.01, 10, blockSize=7)
    rn, rs, re_ = cv2.calcOpticalFlowPyrLK(a, b, pts, None, winSize=(15, 15), maxLevel=4, criteria=(3, 20, 0.03))
    n, s, e = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, winSize=(15, 15), maxLevel=4, criteria=(3, 20, 0.03), ctx=ctx)
    assert np.array_equal(s, rs)
    ok = rs.ravel() == 1
    assert ok.sum() >= 900
    assert np.abs(n - rn)[ok].max() <= 0.05
    assert np.median(np.abs(n - rn)[ok]) <= 1e-3


def test_two_kernel_variants_agree(ctx):
    """The marching, the tile and the generic lambda_min kernels build the map from the same exact integer sums:
    bit-identical maps and feature lists; the register-resident LK kernel and the generic shared-memory one:
    identical status, positions equal to fp32 rounding (both accumulate the same integers exactly)."""
    import ofb200

    def with_env(name, fn):
        os.environ[name] = "1"
        try:
            return fn()
        finally:
            os.environ[name] = "0"

    rng = np.random.default_rng(5)
    for (h, w), seed in [((240, 320), 21), ((131, 517), 22), ((480, 640), 23), ((97, 1003), 24), ((300, 121), 25)]:
        img = synth.texture(h, w, seed)
        mask = (rng.random((h, w)) > 0.3).astype(np.uint8)
        for bs in (3, 7, 12, 32):
            both = lambda: (ofb200.cornerMinEigenVal(img, bs, ctx=ctx),
                            ofb200.goodFeaturesToTrack(img, 300, 0.01, 7, blockSize=bs, ctx=ctx),
                            ofb200.goodFeaturesToTrack(img, 0, 0.05, 3, mask=mask, blockSize=bs, ctx=ctx))
            fast, pts_fast, ptsm_fast = both()                      # marching kernel for blockSize 3, 7, 12
            # ... with its general row loop on every strip: unaligned rows (map), a mask that passes every pixel (list)
            general = min_eig_map_unaligned(ofb200, ctx, img, bs)
            pts_general = ofb200.goodFeaturesToTrack(img, 300, 0.01, 7, mask=np.full_like(img, 255), blockSize=bs, ctx=ctx)
            assert np.array_equal(fast, general) and np.array_equal(as_list(pts_fast), as_list(pts_general))
            tile, pts_tile, ptsm_tile = with_env("OFB_EIG_TILE", both)
            gen, pts_gen, ptsm_gen = with_env("OFB_EIG_GENERIC", both)
            assert np.array_equal(fast, tile), (h, w, bs, np.abs(fast - tile).max(), np.argwhere(fast != tile)[:5])
            assert np.array_equal(fast, gen), (h, w, bs, np.abs(fast - gen).max())
            assert np.array_equal(as_list(pts_fast), as_list(pts_gen))
            assert np.array_equal(as_list(pts_fast), as_list(pts_tile))
            assert np.array_equal(as_list(ptsm_fast), as_list(ptsm_gen))
            assert np.array_equal(as_list(ptsm_fast), as_list(ptsm_tile))
    for case in range(3):
        a, b = synth.affine_pair(240, 320, 30 + case, shift=(3.5 + case, -2.25), rot=0.01 * case)
        pts = io.good_features(a, 150, 0.01, 8, block_size=7)
        extra = np.array([[0, 0], [2.5, 3.5], [319, 239], [318.2, 5.3], [4, 237.5], [160, 0.4], [0.2, 120]], np.float32).reshape(-1, 1, 2)
        pts = np.concatenate([pts, extra])
        for win in ((15, 15), (9, 13), (16, 15)):
            kw = dict(winSize=win, maxLevel=3, criteria=(3, 20, 0.03))
            n1, s1, e1 = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, ctx=ctx, **kw)
            os.environ["OFB_LK_GENERIC"] = "1"
            try:
                n2, s2, e2 = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, ctx=ctx, **kw)
            finally:
                os.environ["OFB_LK_GENERIC"] = "0"
            assert np.array_equal(s1, s2), (case, win)
            ok = s1.ravel() == 1
            # both kernels sum the same integers exactly and round once to fp32 (test_gpu_lk_edges checks them for
            # bit equality), far inside the 0.05 px contract
            assert np.abs(n1 - n2)[ok].max() <= 1e-3, (case, win, np.abs(n1 - n2)[ok].max())
            assert np.abs(e1 - e2)[ok].max() <= 1e-3
            on, os_, oe = io.pyrlk(a, b, pts, win, 3, (3, 20, 0.03))
            assert np.array_equal(s1, os_)
            assert np.abs(n1 - on)[ok].max() <= 5e-3


def test_marching_fast_rows_at_full_size(ctx):
    """The lean row loops of the marching kernel against its general row loop at 1080p and at a size whose band count /
    band height parity differs: identical maps (the general loop on unaligned rows), identical candidate-derived lists (the
    general loop through a mask that passes every pixel), with and without a batch (bands get shorter as the batch grows)."""
    import ofb200
    for (h, w), seed, bs in [((1080, 1920), 71, 7), ((721, 1283), 72, 7), ((540, 960), 73, 3), ((487, 1001), 74, 12)]:
        img = synth.texture(h, w, seed)
        fast_map = ofb200.cornerMinEigenVal(img, bs, ctx=ctx)
        fast_pts = ofb200.goodFeaturesToTrack(img, 1000, 0.01, 10, blockSize=bs, ctx=ctx)
        ref_map = min_eig_map_unaligned(ofb200, ctx, img, bs)
        ref_pts = ofb200.goodFeaturesToTrack(img, 1000, 0.01, 10, mask=np.full_like(img, 255), blockSize=bs, ctx=ctx)
        assert np.array_equal(fast_map, ref_map), (h, w, bs, np.argwhere(fast_map != ref_map)[:4])
        assert np.array_equal(as_list(fast_pts), as_list(ref_pts)), (h, w, bs)
    # batches: 1, 3 and 9 images of 720p through the fused path (feature lists per image must not depend on the batch)
    a, b, mo = synth.make_pair(720, 1280, 1, 77)
    cfg = ofb200.make_pair_cfg(1280, 720, 300, 0.01, 10, 7, (15, 15), 3, (3, 20, 0.03), variant="node",
                               principal=(mo["cx"], mo["cy"]), pos_scale=1.0 / mo["f"], flow_scale=1.0 / (mo["f"] * mo["dt"]))
    lists = []
    for nb in (1, 3, 9):
        imu = np.zeros(nb, ofb200._lib.IMU_DTYPE); imu["d"][:], imu["n"][:], imu["w"][:] = mo["d"], mo["n"], mo["w"]
        res, pp, pn, st = ofb200.frame_pairs(np.stack([a] * nb), np.stack([b] * nb), imu, cfg, want_tracks=True, ctx=ctx)
        for i in range(nb):
            lists.append(pp[i, :int(res["n_features"][i])])
    for l in lists[1:]:
        assert np.array_equal(l, lists[0])


def test_marching_kernel_shapes_vs_generic(ctx):
    """Strip/band decomposition of the marching lambda_min kernel: widths around the strip pitch (128-bs-1 columns),
    heights around the band height, aligned and unaligned pitches, multi-image batches -- maps and candidate-derived
    feature lists must be bit-identical to the generic kernel's (same exact integer sums, same fp32 expression)."""
    import ofb200
    rng = np.random.default_rng(11)
    shapes = [(48, 96), (49, 97), (64, 120), (65, 121), (100, 239), (100, 240), (100, 241), (77, 360), (203, 476),
              (301, 488), (150, 1000), (111, 1284)]
    for k, (h, w) in enumerate(shapes):
        img = synth.texture(h, w, 40 + k)
        if k % 3 == 0:                                   # flat borders and a saturated block: plateaus, zero gradients
            img[:, :5] = 17; img[-4:, :] = 200; img[h // 3:h // 3 + 9, w // 4:w // 4 + 30] = 255
        bs = (3, 7, 12)[k % 3]
        q = float(rng.choice([0.01, 0.05, 0.2]))
        fast = ofb200.cornerMinEigenVal(img, bs, ctx=ctx)
        pts_fast = ofb200.goodFeaturesToTrack(img, 500, q, 5, blockSize=bs, ctx=ctx)
        os.environ["OFB_EIG_GENERIC"] = "1"
        try:
            gen = ofb200.cornerMinEigenVal(img, bs, ctx=ctx)
            pts_gen = ofb200.goodFeaturesToTrack(img, 500, q, 5, blockSize=bs, ctx=ctx)
        finally:
            os.environ["OFB_EIG_GENERIC"] = "0"
        assert np.array_equal(fast, gen), (h, w, bs, np.argwhere(fast != gen)[:4])
        assert np.array_equal(as_list(pts_fast), as_list(pts_gen)), (h, w, bs)
        # and against the CPU oracle's map within the documented tie tolerance
        ref = io.min_eig_map(img, bs)
        tol = 2.0 * bs * 2.0 ** -23 * half_trace_max(img, bs)
        assert np.abs(fast - ref).max() <= tol, (h, w, bs, np.abs(fast - ref).max(), tol)


def test_selection_cluster_mode_equals_single_cta(ctx):
    """Cluster mode of the selection kernel (2/4/8 CTAs per image share the key scans through DSMEM) must return
    exactly the single-CTA list: one chunk, many chunks (maxCorners=0 with a small minDistance), masks, no
    min-distance, and a batch of images."""
    import ofb200
    cases = [(synth.texture(240, 320, 61), dict(maxCorners=200, qualityLevel=0.01, minDistance=10, blockSize=7)),
             (synth.texture(480, 640, 62), dict(maxCorners=0, qualityLevel=0.001, minDistance=2, blockSize=3)),
             (synth.texture(300, 500, 63), dict(maxCorners=5000, qualityLevel=0.01, minDistance=0, blockSize=7)),
             (synth.texture(131, 517, 64), dict(maxCorners=60, qualityLevel=0.3, minDistance=20, blockSize=12)),
             # a tiled image: every interior corner value occurs 80 times, so chunk boundaries fall inside plateaus of equal
             # lambda_min (the routed preparation must fall back or split the plateau by address exactly)
             (np.ascontiguousarray(np.tile(synth.texture(32, 32, 65), (8, 10))),
              dict(maxCorners=3000, qualityLevel=0.01, minDistance=3, blockSize=5)),
             (np.ascontiguousarray(np.tile(synth.texture(16, 16, 66), (30, 40))),
              dict(maxCorners=0, qualityLevel=0.05, minDistance=1, blockSize=3))]
    for img, kw in cases:
        os.environ["OFB_SELECT_CLUSTER"] = "1"
        try:
            ref = as_list(ofb200.goodFeaturesToTrack(img, ctx=ctx, **kw))
            for cs in ("2", "4", "8"):
                os.environ["OFB_SELECT_CLUSTER"] = cs
                got = as_list(ofb200.goodFeaturesToTrack(img, ctx=ctx, **kw))
                assert np.array_equal(got, ref), (img.shape, kw, cs, len(got), len(ref))
            # the block size (chunk of 512 / 1024 / 2048 keys, normally chosen from maxCorners) must not matter either
            for ts, cs in (("256", "1"), ("512", "1"), ("1024", "1"), ("256", "8"), ("512", "4")):
                os.environ["OFB_SELECT_THREADS"], os.environ["OFB_SELECT_CLUSTER"] = ts, cs
                got = as_list(ofb200.goodFeaturesToTrack(img, ctx=ctx, **kw))
                assert np.array_equal(got, ref), (img.shape, kw, ts, cs, len(got), len(ref))
        finally:
            del os.environ["OFB_SELECT_CLUSTER"]
            os.environ.pop("OFB_SELECT_THREADS", None)
    assert len(ref) > 0
    # a batch through the fused path
    a, b, mo = synth.make_pair(240, 320, 5, 5, max_disp=4.0)
    cfg = ofb200.make_pair_cfg(320, 240, 100, 0.01, 8, 7, (15, 15), 3, (3, 20, 0.03), variant="node",
                               principal=(mo["cx"], mo["cy"]), pos_scale=1.0 / mo["f"], flow_scale=1.0 / (mo["f"] * mo["dt"]))
    imu = np.zeros(3, ofb200._lib.IMU_DTYPE); imu["d"][:], imu["n"][:], imu["w"][:] = mo["d"], mo["n"], mo["w"]
    A, B = np.stack([a, b, a]), np.stack([b, a, b])
    out = {}
    for cs in ("1", "8"):
        os.environ["OFB_SELECT_CLUSTER"] = cs
        try:
            out[cs] = ofb200.frame_pairs(A, B, imu, cfg, want_tracks=True, ctx=ctx)
        finally:
            del os.environ["OFB_SELECT_CLUSTER"]
    for k in range(1, 4):
        assert np.array_equal(out["1"][k], out["8"][k])
    assert np.array_equal(out["1"][0]["v"], out["8"][0]["v"])
