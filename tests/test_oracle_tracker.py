"""Pins oracle/tracker_oracle.py (the lifecycle restatement, SURVEY 8f-2): against tests/golden/tracker_golden.npz
(made by tools/make_golden_tracker.py with the real cv2 4.13 operators and the reference's own static_immobile /
r_tilde / solve_lgs) and, where cv2 and a checkout of the reference (OFB_REFERENCE_DIR) exist, against those run live."""
import os

import numpy as np
import pytest

import tracker_cases as tc
from conftest import GOLDEN
from oracle import ref_loader, tracker_oracle

LK_TOL = 2e-4          # oracle LK vs cv2 (tests/test_oracle_vs_cv2.py)


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLDEN, "tracker_golden.npz"))


def test_circle_mask_equals_cv2_circle(g):
    for m, meta in zip(g["circle_masks"], g["circle_meta"]):
        radius, pts = int(meta[0]), meta[1:].reshape(-1, 2)
        got = tracker_oracle.exclusion_mask(pts, radius, m.shape[1], m.shape[0])
        assert np.array_equal(got, m), "radius %d" % radius


def close_positions(a, b, tol, worst=0.05):
    """Positions agree: every point within the north star's 0.05 px (points tracked into an occluding noise block
    converge chaotically) and 80 % of them within `tol`; tol == 0 demands equality."""
    d = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).reshape(-1)
    if d.size == 0:
        return True
    if tol == 0:
        return d.max() == 0
    return d.max() <= max(worst, tol) and np.quantile(d, 0.8) <= tol


def teacher_from_golden(g, name):
    pts, n = g[name + "_pts"], g[name + "_n_points"]
    S, T = n.shape
    return [[None] + [pts[s, k - 1, :n[s, k - 1]] for k in range(1, T)] for s in range(S)]


def compare_with_golden(g, name, res, pos_tol, v_rtol, exact_prev=True, worst=0.05):
    for s, steps in enumerate(res):
        for k, r in enumerate(steps):
            tag = "%s stream %d step %d" % (name, s, k)
            for key in ("n_prev", "n_tracked", "n_kept", "n_added", "n_points"):
                assert r[key] == g["%s_%s" % (name, key)][s, k], "%s: %s" % (tag, key)
            nk, npts = r["n_kept"], r["n_points"]
            assert close_positions(r["kept_next"], g[name + "_kept_next"][s, k, :nk], pos_tol, worst), tag
            if exact_prev:
                assert np.array_equal(r["kept_prev"], g[name + "_kept_prev"][s, k, :nk]), tag
            else:
                assert close_positions(r["kept_prev"], g[name + "_kept_prev"][s, k, :nk], pos_tol, worst), tag
            assert close_positions(r["pts"], g[name + "_pts"][s, k, :npts], pos_tol, worst), tag
            # appended corners are integer pixel positions: exact
            na = r["n_added"]
            if na:
                assert np.array_equal(r["pts"][npts - na:], g[name + "_pts"][s, k, npts - na:npts]), tag + ": top-up"
            assert bool(r["solved"]) == bool(g[name + "_solved"][s, k]), tag
            if r["solved"]:
                gv = g[name + "_v"][s, k]
                assert np.abs(r["v"] - gv).max() <= v_rtol * max(np.abs(gv).max(), 1e-12), tag + ": velocity"


@pytest.mark.parametrize("name", sorted(tc.SCENARIOS))
def test_oracle_steps_equal_cv2_golden(g, name):
    """Teacher-forced: every step starts from the golden point set, so each step is compared on identical inputs."""
    frames, imus, kw = tc.build(name)
    res = tc.run_oracle_tracker(lambda: tracker_oracle.TrackerOracle(tc.W, tc.H, **kw), frames, imus,
                                teacher=teacher_from_golden(g, name))
    compare_with_golden(g, name, res, LK_TOL, 2e-3)


@pytest.mark.parametrize("name", ["exp"])
def test_oracle_free_running_stays_on_golden(g, name):
    """No teacher: over the chain of 8 frames 80 % of the points stay within the LK tolerance of the north star
    (0.05 px); points tracked into the occluding noise block wander freely (LK on noise is chaotic)."""
    frames, imus, kw = tc.build(name)
    res = tc.run_oracle_tracker(lambda: tracker_oracle.TrackerOracle(tc.W, tc.H, **kw), frames, imus)
    compare_with_golden(g, name, res, 0.05, 0.05, exact_prev=False, worst=float("inf"))


def test_static_immobile_equals_reference():
    rng = np.random.default_rng(5)
    new = rng.uniform(0, 100, (200, 1, 2)).astype(np.float32)
    old = (new + rng.normal(0, 3, new.shape)).astype(np.float32)
    old[::17, 0, 0] = 42.0
    got = tracker_oracle.static_immobile(new, old, 6.0, 1.7, 42.0)
    # independent statement of of_library.py:88-92
    thr = np.float32(6.0 / 1.7)
    d = np.abs(new - old)
    exp = (d[:, :, 0] < thr) & (d[:, :, 1] < thr) & (old[:, :, 0] != 42.0) & (old[:, :, 1] != 42.0)
    assert np.array_equal(got.astype(bool), exp)
    if ref_loader.available():
        ref = ref_loader.of_library("root")["static_immobile"](new, old, 6.0, 1.7, 42.0)
        assert np.array_equal(got.astype(bool), np.asarray(ref).astype(bool))


def test_golden_is_what_cv2_and_the_reference_produce_here(g):
    """Fixture freshness: where cv2 and the reference exist the golden file is regenerated live and compared."""
    cv2 = pytest.importorskip("cv2")
    if not ref_loader.available() or not cv2.__version__.startswith("4.13"):
        pytest.skip(ref_loader.MISSING + " and cv2 4.13")
    eng = tc.cv2_engine()
    for name in tc.SCENARIOS:
        frames, imus, kw = tc.build(name)
        res = tc.run_oracle_tracker(lambda: tracker_oracle.TrackerOracle(tc.W, tc.H, engine=eng, **kw), frames, imus)
        compare_with_golden(g, name, res, 0.0, 1e-12)


@pytest.mark.parametrize("seed", tc.RANDOM_SEEDS)
def test_oracle_vs_live_cv2_on_random_sequences(seed):
    """Beyond the committed fixture: random drift / rotation / occlusion / parameters, the oracle step against the same
    step made of the real cv2 operators (tests/golden/tracker_random_golden.npz, made by tools/make_golden_tracker.py;
    run live, with the reference's own functions, where cv2 4.13 and the reference exist), teacher-forced on the cv2
    chain."""
    cv2 = pytest.importorskip("cv2")
    frames, imus, kw = tc.random_case(seed)
    if ref_loader.available() and cv2.__version__.startswith("4.13"):
        eng = tc.cv2_engine()
        ref = tc.run_oracle_tracker(lambda: tracker_oracle.TrackerOracle(tc.W, tc.H, engine=eng, **kw), frames, imus)
        g = {"live_" + k: v for k, v in tc.pack(ref, kw["max_features"] + kw["min_features"]).items()}
    else:
        stored = np.load(os.path.join(GOLDEN, "tracker_random_golden.npz"))
        g = {"live_" + k[len("s%d_" % seed):]: stored[k] for k in stored.files if k.startswith("s%d_" % seed)}
        assert g, "no stored sequence for seed %d" % seed

    class OwnSelectionOnCv2Map(tracker_oracle.Engine):
        """the oracle's selection on cv2's lambda_min map: two correct fp32 maps may order near-ties differently (the
        documented float tie, DESIGN.md), which is not what this test is about"""

        def good_features(self, img, max_corners, quality, min_distance, block_size, mask=None):
            from oracle import image_oracle as io
            return io.select_features(cv2.cornerMinEigenVal(img, block_size), max_corners, quality, min_distance, mask)
    res = tc.run_oracle_tracker(lambda: tracker_oracle.TrackerOracle(tc.W, tc.H, engine=OwnSelectionOnCv2Map(), **kw), frames,
                                imus, teacher=teacher_from_golden(g, "live"))
    compare_with_golden(g, "live", res, LK_TOL, 5e-3)
