"""CPU side of the forward-backward check (oracle/fb_oracle.py, include/ofb200.h `ofb_pyrlk_fb`): the fold over the C
oracle's LK against cv2 4.13 (tests/golden/fb_golden.npz), FBEngine against the three lines of OpenCV's
samples/python/lk_track.py, the outlier scene through cv2, and the threshold checks of the Python layer."""
import os
import sys

import numpy as np
import pytest

import fb_cases
from oracle import fb_oracle, image_oracle as io
from oracle import tracker_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_golden_fb  # noqa: E402

NEAR = 0.05          # the project's LK position contract against cv2 (tests/test_gpu_vision.py)


def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "fb_golden.npz"))


def golden_cases(g):
    """(tag, prev, next, p0, lk, T) of every case in the golden file; the occluder frames regenerate from their seeds"""
    cases = make_golden_fb.golden_inputs()
    for k in fb_cases.OCCLUDER_SEEDS:
        a, b, _, _ = fb_cases.occluder_scene(k)
        cases.append(("occluder%d" % k, a, b, g["occluder%d_p0" % k], fb_cases.OCCLUDER_LK, fb_cases.OCCLUDER_T))
    return cases


def compare_to_golden(g, tag, status, fb_err):
    """statuses equal except where cv2's fb_err lies within NEAR of T; fb_err within 0.1 px where both are finite.
    -> number of points the near-threshold exception covered"""
    T = float(g[tag + "_T"])
    gst, gfb = fb_oracle.fb_check(g[tag + "_p0"], g[tag + "_p1"], g[tag + "_st"], g[tag + "_p0r"], g[tag + "_st0"], T)
    assert np.array_equal(gfb, g[tag + "_fb_err"]), tag          # the fold restates the sample's lines
    status = np.asarray(status).reshape(-1)
    near = np.abs(gfb.astype(np.float64) - T) <= NEAR
    bad = (status != gst) & ~near
    assert not bad.any(), (tag, np.nonzero(bad)[0][:10], gfb[bad][:10])
    fin = np.isfinite(gfb) & np.isfinite(fb_err)
    assert np.array_equal(np.isfinite(gfb) | near, np.isfinite(fb_err) | near), tag
    if fin.any():
        assert np.abs(fb_err[fin] - gfb[fin]).max() <= 0.1, tag
    return int(((status != gst) & near).sum())


def test_fold_over_c_oracle_reproduces_cv2_golden():
    g = golden()
    covered, total = 0, 0
    for tag, a, b, p0, (win, ml, crit), T in golden_cases(g):
        assert np.array_equal(np.asarray(p0, np.float32).reshape(-1, 2), g[tag + "_p0"].reshape(-1, 2)), tag
        p1, st, _ = io.pyrlk(a, b, p0, win, ml, crit)
        p0r, st0, _ = io.pyrlk(b, a, p1, win, ml, crit)
        status, fb = fb_oracle.fb_check(p0, p1, st, p0r, st0, T)
        covered += compare_to_golden(g, tag, status, fb)
        total += len(status)
    print("near-threshold exception covered %d of %d points" % (covered, total))
    assert covered <= 0.01 * total


def test_fb_check_fold():
    p0 = np.array([[10, 10], [20, 20], [30, 30], [40, 40]], np.float32)
    p0r = p0 + np.array([[0.25, -0.75], [1.0, 0.0], [0.0, 0.0], [0.0, 0.0]], np.float32)
    st, fb = fb_oracle.fb_check(p0, p0, [1, 1, 0, 1], p0r, [1, 1, 1, 0], 1.0)
    assert st.tolist() == [1, 0, 0, 0]                           # 1.0 < 1.0 is false: the comparison is strict
    assert fb[0] == np.float32(0.75) and fb[1] == 1.0 and np.isinf(fb[2:]).all()
    st, fb = fb_oracle.fb_check(p0, p0, [1, 1, 0, 1], p0r, [1, 1, 1, 0], 0)
    assert st.tolist() == [1, 1, 0, 1] and np.isinf(fb).all()
    with pytest.raises(ValueError):
        fb_oracle.fb_check(p0, p0, [1] * 4, p0r, [1] * 4, -1.0)


def test_fb_engine_equals_sample_lines():
    cv2 = pytest.importorskip("cv2")
    import tracker_cases as tc
    g = np.load(os.path.join(ROOT, "tests", "golden", "cv2_golden.npz"))
    a, b, p0 = g["c1_prev"], g["c1_next"], g["c1_gftt_bench"]
    lk = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
    p1, st, err = cv2.calcOpticalFlowPyrLK(a, b, p0, None, **lk)
    p0r, st0, _ = cv2.calcOpticalFlowPyrLK(b, a, p1, None, **lk)
    d = abs(p0 - p0r).reshape(-1, 2).max(-1)
    good = (d < 1) & (st.ravel() == 1) & (st0.ravel() == 1)
    eng = fb_oracle.FBEngine(tc.cv2_engine(reference=False), 1.0)
    q1, qst, qerr = eng.pyrlk(a, b, p0, (15, 15), 3, (3, 20, 0.03))
    assert np.array_equal(q1, p1) and np.array_equal(qerr, err)
    assert np.array_equal(qst.ravel(), good.astype(np.uint8)) and qst.shape == st.shape
    assert 0 < int((st.ravel() == 1).sum() - good.sum()) or good.all()
    # every other operator is the inner engine's
    assert eng.good_features(a, 10, 0.01, 10, 7) is not None


def test_fb_engine_on_tracker_oracle_drops_only_failed_tracks():
    """TrackerOracle with the check: the set after the first tracked step is the plain oracle's minus the points the
    check rejected."""
    import tracker_cases as tc
    frames, imus, kw = tc.random_case(21)
    okw = {k: v for k, v in kw.items() if k != "bgr"}
    plain = tracker_oracle.TrackerOracle(tc.W, tc.H, **okw)
    fb = tracker_oracle.TrackerOracle(tc.W, tc.H, engine=fb_oracle.FBEngine(tracker_oracle.Engine(), 0.25), **okw)
    im = imus[0]
    for k in range(2):
        r0 = plain.step(frames[0][k], im[k]["d"], im[k]["n"], im[k]["w"], im[k]["t"], im[k]["v_prior"])
        r1 = fb.step(frames[0][k], im[k]["d"], im[k]["n"], im[k]["w"], im[k]["t"], im[k]["v_prior"])
    assert r1["n_prev"] == r0["n_prev"] and r1["n_tracked"] <= r0["n_tracked"]
    kn0 = {tuple(p) for p in r0["kept_next"].tolist()}
    assert all(tuple(p) in kn0 for p in r1["kept_next"].tolist())


def test_outlier_scene_through_cv2():
    """The occluder scene with cv2's LK: the check drops most tracks that start inside the patch, keeps almost all that
    start far from it, and more than halves the mean velocity error."""
    g = golden()
    rej, far_kept, e_plain, e_fb = [], [], [], []
    for k in fb_cases.OCCLUDER_SEEDS:
        _, _, mo, patch = fb_cases.occluder_scene(k)
        t = "occluder%d" % k
        p0, p1, st = g[t + "_p0"], g[t + "_p1"], g[t + "_st"].ravel() == 1
        good, _ = fb_oracle.fb_check(p0, p1, g[t + "_st"], g[t + "_p0r"], g[t + "_st0"], fb_cases.OCCLUDER_T)
        good = good == 1
        inside, far = fb_cases.patch_masks(p0, patch)
        rej.append(1 - (inside & good).sum() / (inside & st).sum())
        far_kept.append((far & good).sum() / (far & st).sum())
        e_plain.append(fb_cases.velocity_error(p0, p1, st, mo))
        e_fb.append(fb_cases.velocity_error(p0, p1, good, mo))
    print("rejected inside", np.round(rej, 3), "kept far", np.round(far_kept, 3), "error", np.round(e_plain, 3), np.round(e_fb, 3))
    assert min(rej) >= 0.70 and min(far_kept) >= 0.97
    assert np.mean(e_fb) < 0.5 * np.mean(e_plain)


@pytest.mark.parametrize("bad", [-1.0, -1e-30, float("nan"), "1", "abc", [1.0], True])
def test_python_layer_rejects_invalid_thresholds(bad):
    import ofb200
    from ofb200.vision import _fb_threshold
    with pytest.raises(ValueError):
        _fb_threshold(bad)
    img = np.zeros((32, 32), np.uint8)
    with pytest.raises(ValueError):
        ofb200.track_forward_backward(img, img, np.zeros((1, 2), np.float32), threshold=bad)
    cfg = ofb200.make_pair_cfg(32, 32, 10)
    with pytest.raises(ValueError):
        ofb200.frame_pairs(img[None], img[None], np.zeros(1, ofb200._lib.IMU_DTYPE), cfg, fb_threshold=bad)
    with pytest.raises(ValueError):
        ofb200.StreamTracker(32, 32, fb_threshold=bad)


def test_python_layer_threshold_values():
    from ofb200.vision import _fb_threshold
    assert _fb_threshold(None) == 0.0 and _fb_threshold(0) == 0.0 and _fb_threshold(np.float32(0.5)) == 0.5
    assert _fb_threshold(float("inf")) == float("inf") and _fb_threshold(2) == 2.0
