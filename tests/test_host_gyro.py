"""Gyro prediction of the LK tracks on the host: the NumPy predictor (oracle/gyro_oracle.py) against the reference's flow
model, its fallbacks, cv2.projectPoints and the C LK oracle with initial flow against cv2 4.13 (tests/golden/
gyro_golden.npz), and the Python-side argument checks."""
import os

import numpy as np
import pytest

import gyro_cases
from conftest import ROOT
from oracle import camera_oracle as co
from oracle import fb_oracle
from oracle import gyro_oracle as go
from oracle import velocity_oracle as vo

GOLD = np.load(os.path.join(ROOT, "tests", "golden", "gyro_golden.npz"))
CAM = np.load(os.path.join(ROOT, "tests", "golden", "camera_golden.npz"))
CASES = ["c%d" % i for i in range(16)]


def _predict64(x, w, dt):
    """the predictor's rotation on normalised fp64 points (pinhole with c = 0, pos_scale = 1, no fp32 rounding)"""
    r = np.asarray(w, np.float64) * dt
    a, b = go.rotation_coeffs(r)
    X = np.c_[x, np.ones(len(x))]
    c = np.cross(r, X)
    X2 = X + a * c + b * np.cross(r, c)
    return X2[:, :2] / X2[:, 2:]


@pytest.mark.parametrize("w", [[0.3, -0.5, 0.8], [2.0, 0.1, -0.4], [0.0, 0.0, 3.0], [-1.5, 2.5, 0.2]])
def test_sign_matches_the_reference_flow_model(w):
    """(predict(x) - x) / dt -> generate_test_data(x, v=0, w, d, n) as dt -> 0: the solve's sign convention for w"""
    x = np.array([[0.1, -0.2], [0.3, 0.05], [-0.4, 0.3], [0.0, 0.0], [0.6, -0.5]])
    ref = vo.generate_test_data(x, np.zeros(3), np.asarray(w, np.float64), 2.0, np.array([0.0, 0.0, 1.0]))
    errs = []
    for dt in (1e-2, 1e-3, 1e-4):
        e = np.abs((_predict64(x, w, dt) - x) / dt - ref).max()
        errs.append(e)
        assert e < 10 * dt * (1 + np.abs(w).max() ** 2), (dt, e)
    assert errs[2] < errs[1] < errs[0]            # O(dt)


def test_roll_keeps_the_principal_point():
    m = go.pinhole(640.0, 360.0, 1 / 900.0, 1 / (900.0 / 30))
    p = np.array([[640.0, 360.0], [700.0, 360.0]], np.float32)
    g = go.predict(p, [0.0, 0.0, 5.0], m)
    assert np.array_equal(g[0], p[0])
    r = np.hypot(*(g[1] - p[0]))
    assert abs(r - 60.0) < 1e-3 and g[1, 1] > p[1, 1]       # rotated about c, radius kept


def test_fallbacks():
    m = go.pinhole(640.0, 360.0, 1 / 900.0, 1 / (900.0 * 0.5))
    p = np.array([[100.0, 50.0], [640.0, 360.0], [1200.0, 700.0]], np.float32)
    assert np.array_equal(go.predict(p, [0, 0, 0], m), p)                     # w = 0: the point, bit for bit
    assert np.array_equal(go.predict(p, [np.nan, 0, 0], m), p)                # NaN gyro sample
    assert np.array_equal(go.predict(p, [0, np.inf, 0], m), p)
    # a yaw of 3 rad over dt = 0.5 s turns points behind the camera (X'_z <= 0)
    g = go.predict(p, [0, 6.0, 0], m)
    assert np.array_equal(g, p)
    cam = go.camera(CAM["K"], CAM["c4_dist"][:5], 30.0, 20)
    assert np.array_equal(go.predict(p, [0, 0, 0], cam), p)


@pytest.mark.parametrize("case", CASES)
def test_project_points_matches_cv2_golden(case):
    K, D = CAM["K"], CAM[case + "_dist"][:int(CAM[case + "_n_dist"])]
    assert np.array_equal(go.project_points(GOLD["proj_xy"], K, D if len(D) else None), GOLD["proj_" + case])


def test_project_points_matches_live_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    xy = rng.uniform(-0.8, 0.8, (200, 2))
    obj = np.c_[xy, np.ones(len(xy))].reshape(-1, 1, 3)
    for case in CASES:
        K, D = CAM["K"], CAM[case + "_dist"][:int(CAM[case + "_n_dist"])]
        ref = cv2.projectPoints(obj, np.zeros(3), np.zeros(3), K, D if len(D) else None)[0].reshape(-1, 2)
        assert np.array_equal(go.project_points(xy, K, D if len(D) else None), ref), case


def _converging(case, p):
    """the inverse lens model of `case` has converged after 20 iterations at the pixels p"""
    K, D = CAM["K"], CAM[case + "_dist"][:int(CAM[case + "_n_dist"])]
    return np.abs(co.undistort(p, K, D, 20) - co.undistort(p, K, D, 200)).max() < 1e-12


_P = np.c_[np.random.default_rng(4).uniform(200, 1080, 300), np.random.default_rng(5).uniform(120, 600, 300)]


@pytest.mark.parametrize("case", [c for c in CASES if _converging(c, _P)])
def test_project_inverts_converged_undistort(case):
    K, D = CAM["K"], CAM[case + "_dist"][:int(CAM[case + "_n_dist"])]
    p = _P
    x = co.undistort(p, K, D, 20)
    q = go.project_points(x, K, D if len(D) else None)
    assert np.abs(q - p).max() < 1e-6


@pytest.mark.parametrize("name", list(gyro_cases.ROTATIONS))
def test_c_oracle_lk_with_initial_flow_matches_cv2_golden(name):
    a, b, w = gyro_cases.rotation_scene(name)
    assert np.array_equal(w, GOLD[name + "_w"])
    p0, g = GOLD[name + "_p0"], GOLD[name + "_g"]
    m = go.pinhole(gyro_cases.CX, gyro_cases.CY, 1.0 / gyro_cases.F, 1.0 / (gyro_cases.F * gyro_cases.DT))
    assert np.array_equal(go.predict(p0, w, m), g)
    win, ml, crit = gyro_cases.LK
    p1, st, _ = go.pyrlk_init(a, b, p0, g, win, ml, crit)
    st = st.ravel()
    assert np.array_equal(st, GOLD[name + "_st"])
    ok = st == 1
    assert ok.sum() > 0.7 * len(st)
    assert np.abs(p1.reshape(-1, 2)[ok] - GOLD[name + "_p1"][ok]).max() <= 2e-4
    # the forward-backward composition: backward pass seeded with p1 + (p0 - g)
    p1c = GOLD[name + "_p1"]
    p0r, st0, _ = go.pyrlk_init(b, a, p1c, p1c + (p0 - g), win, ml, crit)
    both = ok & (st0.ravel() == 1)
    assert np.array_equal(st0.ravel(), GOLD[name + "_st0"])
    assert np.abs(p0r.reshape(-1, 2)[both] - GOLD[name + "_p0r"][both]).max() <= 2e-4
    status, fb = fb_oracle.fb_check(p0, p1c, ok.astype(np.uint8), GOLD[name + "_p0r"], GOLD[name + "_st0"], 1.0)
    assert np.array_equal(fb, GOLD[name + "_fb"])


def test_plain_lk_fails_and_prediction_holds_in_the_rotation_scene():
    """the scenes are hard enough: plain LK keeps fewer than half of the features within 0.5 px, LK from the prediction
    keeps at least 95 % of those that stay in the frame (C oracle, no GPU)"""
    from oracle import image_oracle as io
    m = go.pinhole(gyro_cases.CX, gyro_cases.CY, 1.0 / gyro_cases.F, 1.0 / (gyro_cases.F * gyro_cases.DT))
    win, ml, crit = gyro_cases.LK
    for name in gyro_cases.ROTATIONS:
        a, b, w = gyro_cases.rotation_scene(name)
        p0 = GOLD[name + "_p0"]
        t, inside = gyro_cases.true_positions(p0, w)
        p1, st, _ = io.pyrlk(a, b, p0, win, ml, crit)
        good = (st.ravel() == 1) & (np.abs(p1.reshape(-1, 2) - t).max(1) < 0.5)
        assert good.sum() < 0.5 * len(p0), (name, good.sum(), len(p0))
        q1, qs, _ = go.pyrlk_init(a, b, p0, go.predict(p0, w, m), win, ml, crit)
        good = (qs.ravel() == 1) & (np.abs(q1.reshape(-1, 2) - t).max(1) < 0.5)
        assert (good & inside).sum() >= 0.95 * inside.sum(), (name, (good & inside).sum(), inside.sum())


def test_python_validation():
    import ofb200
    p = np.zeros((3, 2), np.float32)
    with pytest.raises(ValueError):
        ofb200.gyro_predict(p, [0, 0], principal=(1, 1))                     # omega needs 3 entries
    with pytest.raises(ValueError):
        ofb200.gyro_predict(p, [0, 0, 0], principal=(1, 1), flow_scale=0.0)
    with pytest.raises(ValueError):
        ofb200.gyro_predict(p, [0, 0, 0])                                     # no model
    with pytest.raises(ValueError):
        ofb200.gyro_predict(np.zeros((3, 3)), [0, 0, 0], principal=(1, 1))
    with pytest.raises(ValueError):
        ofb200.gyro_predict(p, [0, 0, 0], camera=(np.eye(3), None, 30.0), principal=(1, 1))
    cfg = ofb200.make_pair_cfg(64, 48, 10, flow_scale=0.0)
    a = np.zeros((1, 48, 64), np.uint8)
    imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
    with pytest.raises(ValueError):
        ofb200.frame_pairs(a, a, imu, cfg, gyro_prediction=True)
    with pytest.raises(ValueError):
        ofb200.frame_pairs(a, a, imu, cfg, gyro_prediction="yes")
