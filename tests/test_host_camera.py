"""Calibrated camera on the CPU: oracle/camera_oracle.py against cv2 4.13's undistortPoints / undistortPointsIter
(stored in tests/golden/camera_golden.npz by tools/make_golden_camera.py, and live where cv2 imports), the
icdist < 0 fallback, the calibrated tracker oracle (CameraTrackerOracle) against the pinhole one, and the argument
checks of the Python layer (they run before any device call)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import camera_oracle as co


def golden_cases():
    """-> (golden npz, list of dicts: src, K, D, iterations, R, P, out)"""
    g = np.load(os.path.join(GOLDEN, "camera_golden.npz"))
    cases = []
    for i in range(int(g["n_cases"])):
        k = lambda s: g["c%d_%s" % (i, s)]
        n = int(k("n_dist"))
        cases.append(dict(src=g["src32"] if int(k("f32")) else g["src"], K=g["K"], D=k("dist")[:n] if n else None,
                          iterations=int(k("iterations")), R=k("R") if k("R").size else None,
                          P=k("P") if k("P").size else None, out=k("out"), tag="case %d" % i))
    return g, cases


def test_oracle_equals_cv2_golden():
    g, cases = golden_cases()
    assert len(cases) >= 16
    for c in cases:
        got = co.undistort(c["src"], c["K"], c["D"], c["iterations"], co.rectification(c["R"], c["P"]))
        got = got.astype(c["out"].dtype)
        assert np.abs(got - c["out"]).max() <= 1e-15, c["tag"]


def test_golden_covers_the_icdist_fallback():
    """The strong lens (k1 = -2) sends the corners through OpenCV's icdist < 0 branch: those points come back as the
    undistorted-by-nothing (x0, y0)."""
    g, cases = golden_cases()
    c = [c for c in cases if c["D"] is not None and c["D"][0] == -2.0][0]
    x0 = co.undistort(c["src"], c["K"], None)
    fell_back = np.all(c["out"] == x0, axis=1)
    assert 0 < fell_back.sum() < len(fell_back)


def test_oracle_equals_live_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    src = np.stack([rng.uniform(-50, 1330, 3000), rng.uniform(-50, 770, 3000)], axis=1)
    K = np.array([[880.0, 0.0, 650.0], [0.0, 870.0, 350.0], [0.0, 0.0, 1.0]])
    R = cv2.Rodrigues(np.array([-0.02, 0.01, 0.05]))[0]
    P = np.array([[800.0, 0.0, 640.0, 12.0], [0.0, 800.0, 360.0, 0.0], [0.0, 0.0, 1.0, 0.0]])
    for D in (None, [-0.2, 0.05, 0.001, 0.002], [-0.3, 0.12, 0.001, -0.0005, -0.02], [0.1, -0.05, 0, 0, 0.01, 0.2, -0.1, 0.03]):
        Dn = None if D is None else np.array(D)
        for it in (1, 5, 20):
            for r, p in ((None, None), (R, None), (None, P), (R, P)):
                ref = cv2.undistortPointsIter(src.reshape(-1, 1, 2), K, Dn, r, p, (cv2.TERM_CRITERIA_COUNT, it, 0))
                got = co.undistort(src, K, Dn, it, co.rectification(r, p))
                assert np.abs(got - ref.reshape(-1, 2)).max() <= 1e-15, (D, it, r is None, p is None)


def test_calibrate_reduces_to_the_pinhole_without_distortion():
    """n_dist = 0, fx = fy = 1/pos_scale, rate = flow_scale/pos_scale: the pinhole of node:229-235 up to rounding."""
    rng = np.random.default_rng(1)
    new = rng.uniform(0, 640, (50, 2)).astype(np.float32)
    old = (new + rng.normal(0, 2, (50, 2))).astype(np.float32)
    f, c, dt = 512.0, (320.0, 240.0), 1 / 30.0
    K = np.array([[f, 0, c[0]], [0, f, c[1]], [0, 0, 1.0]])
    x, u = co.calibrate(new, old, (K, None, 1 / dt, 20))
    np.testing.assert_allclose(x, (new.astype(np.float64) - c) / f, rtol=1e-15, atol=1e-17)
    np.testing.assert_allclose(u, (new - old).astype(np.float64) / (f * dt), rtol=1e-6)    # fp32 flow vs fp64 difference


K_OK = [[900.0, 0.0, 640.0], [0.0, 900.0, 360.0], [0.0, 0.0, 1.0]]


@pytest.mark.parametrize("K, D, rate, iterations", [
    ([[900.0, 1.0, 640.0], [0.0, 900.0, 360.0], [0.0, 0.0, 1.0]], None, 30.0, 20),     # skew
    ([[0.0, 0.0, 640.0], [0.0, 900.0, 360.0], [0.0, 0.0, 1.0]], None, 30.0, 20),       # fx = 0
    ([[900.0, 0.0, 640.0], [0.0, -900.0, 360.0], [0.0, 0.0, 1.0]], None, 30.0, 20),    # fy < 0
    ([[900.0, 0.0, np.nan], [0.0, 900.0, 360.0], [0.0, 0.0, 1.0]], None, 30.0, 20),    # non-finite K
    (np.eye(2), None, 30.0, 20),                                                        # not 3x3
    (K_OK, [0.1, 0.2, 0.0], 30.0, 20),                                                  # 3 coefficients
    (K_OK, [0.1] * 12, 30.0, 20),                                                       # thin prism: out of scope
    (K_OK, [0.1, np.inf, 0.0, 0.0], 30.0, 20),                                          # non-finite D
    (K_OK, None, 0.0, 20),                                                              # rate
    (K_OK, None, -30.0, 20),
    (K_OK, None, np.nan, 20),
    (K_OK, None, 30.0, 0),                                                              # iterations
    (K_OK, None, 30.0, 1001),
    (K_OK, None, 30.0, 2.5),
])
def test_make_camera_rejects(K, D, rate, iterations):
    import ofb200
    with pytest.raises(ValueError):
        ofb200.make_camera(K, D, rate, iterations)


def test_make_camera_fields():
    import ofb200
    cam = ofb200.make_camera([[910.0, 0, 641.0], [0, 905.0, 362.0], [0, 0, 1]], [-0.3, 0.1, 0.001, 0.002, -0.02], 30.0)
    assert (cam.fx, cam.fy, cam.cx, cam.cy, cam.n_dist, cam.iterations, cam.rate) == (910.0, 905.0, 641.0, 362.0, 5, 20, 30.0)
    assert list(cam.dist) == [-0.3, 0.1, 0.001, 0.002, -0.02, 0.0, 0.0, 0.0]
    assert ofb200.CAMERA_ITERATIONS == 20
    assert ofb200.vision.as_camera(None) is None and ofb200.vision.as_camera(cam) is cam
    assert ofb200.vision.as_camera((np.array(K_OK), None, 25.0, 7)).iterations == 7
    for bad in ((np.array(K_OK), None), (np.array(K_OK), None, 1.0, 5, 0), "camera"):
        with pytest.raises(ValueError):
            ofb200.vision.as_camera(bad)


def test_undistort_points_argument_checks():
    import ofb200
    pts = np.zeros((4, 2))
    with pytest.raises(ValueError):                                       # EPS is not supported
        ofb200.undistortPointsIter(pts, K_OK, None, None, None, (ofb200.TERM_CRITERIA_COUNT | ofb200.TERM_CRITERIA_EPS, 5, 0.1))
    with pytest.raises(ValueError):
        ofb200.undistortPointsIter(pts, K_OK, None, None, None, (ofb200.TERM_CRITERIA_EPS, 5, 0.1))
    for bad in (np.zeros((4, 3)), np.zeros((4, 2, 2)), np.zeros((4, 2), np.int32), np.zeros(8)):
        with pytest.raises(ValueError):
            ofb200.undistortPoints(bad, K_OK, None)
    with pytest.raises(ValueError):
        ofb200.undistortPoints(pts, K_OK, None, R=np.eye(2))
    with pytest.raises(ValueError):
        ofb200.undistortPoints(pts, K_OK, None, P=np.eye(4))
    with pytest.raises(ValueError):
        ofb200.undistortPoints(pts, K_OK, [0.1, 0.1])
    # an empty input needs no device and keeps cv2's shape and dtype
    for dt in (np.float32, np.float64):
        out = ofb200.undistortPoints(np.zeros((0, 1, 2), dt), K_OK, [-0.3, 0.1, 0, 0, 0])
        assert out.shape == (0, 1, 2) and out.dtype == dt


def test_rectification_matches_the_oracle():
    import ofb200
    rng = np.random.default_rng(3)
    R, P = rng.normal(size=(3, 3)), rng.normal(size=(3, 4))
    assert np.array_equal(ofb200.vision._rectification(R, P), co.rectification(R, P))
    assert np.array_equal(ofb200.vision._rectification(None, P[:, :3]), P[:, :3])
    assert np.array_equal(ofb200.vision._rectification(R, None), R)
    assert ofb200.vision._rectification(None, None) is None


@pytest.mark.parametrize("seed", [22, 24, 26])
def test_camera_tracker_oracle_reduces_to_the_pinhole_oracle(seed):
    """CameraTrackerOracle with a distortion-free camera equal to the pinhole (f = 1/scaling = 256 px, c = the principal
    point, rate 1: every scale a power of two) keeps the same points and solves the same velocities as TrackerOracle on
    the gated random sequences; with a wide-angle lens the velocities move."""
    import tracker_cases as tc
    from oracle import tracker_oracle
    from oracle import velocity_oracle as vo
    frames, imus, kw = tc.random_case(seed)
    assert kw["gate"] is not None and 1.0 / kw["scaling"] == 256.0
    c = vo.pix_trans((tc.W, tc.H))
    K = np.array([[256.0, 0.0, c[0]], [0.0, 256.0, c[1]], [0.0, 0.0, 1.0]])

    def run(orc):
        out = []
        for k in range(len(frames[0])):
            im = imus[0][k]
            out.append(orc.step(frames[0][k], im["d"], im["n"], im["w"], im["t"], im["v_prior"]))
        return out
    ref = run(tracker_oracle.TrackerOracle(tc.W, tc.H, **kw))
    got = run(co.CameraTrackerOracle(tc.W, tc.H, (K, None, 1.0, 20), **kw))
    wide = run(co.CameraTrackerOracle(tc.W, tc.H, (K, [-0.3, 0.1, 0.0, 0.0, -0.02], 1.0, 20), **kw))
    moved = 0
    for a, b, w in zip(ref, got, wide):
        for key in ("n_prev", "n_tracked", "n_kept", "n_added", "n_points", "solved"):
            assert a[key] == b[key], key
        assert np.array_equal(a["kept_next"], b["kept_next"])
        if a["solved"]:
            assert np.abs(b["v"] - a["v"]).max() <= 1e-9 * np.abs(a["v"]).max()
            if w["solved"]:
                moved += np.abs(w["v"] - a["v"]).max() > 1e-3 * np.abs(a["v"]).max()
    assert sum(a["solved"] for a in ref) >= 3 and moved >= 1
