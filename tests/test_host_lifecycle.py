"""Host-side rows of SURVEY 8f: replay ingestion + velocity Kalman filter (8f-4, ofb200.replay) and the element-wise
helpers of initialize_ft (8f-3: calc_height, convert_to_of, dynamic_immobile, eval_ft in ofb200.of_library).
CPU only: no compute call into libofb200.so."""
import io
import os

import numpy as np
import pytest

import ofb200
import ofb200.of_library as of
from ofb200 import replay
from oracle import ref_loader, velocity_oracle as vo

RANGE_YAML = """\
- !!python/object/new:sensor_msgs.msg._Range.Range
  state:
  - !!python/object/new:std_msgs.msg._Header.Header
    state:
    - 3991
    - !!python/object/new:genpy.rostime.Time
      state: [1455209081, 675119360]
    - hrlv_ez4_sonar
  - 0
  - 0.0
  - 0.2
  - 7.0
  - 0.83
- !!python/object/new:sensor_msgs.msg._Range.Range
  state:
  - !!python/object/new:std_msgs.msg._Header.Header
    state:
    - 3992
    - !!python/object/new:genpy.rostime.Time
      state: [1455209082, 96119360]
    - hrlv_ez4_sonar
  - 0
  - 0.0
  - 0.2
  - 7.0
  - 0.91
"""

IMU_YAML = """\
- !!python/object/new:sensor_msgs.msg._Imu.Imu
  state:
  - !!python/object/new:std_msgs.msg._Header.Header
    state:
    - 7
    - !!python/object/new:genpy.rostime.Time
      state: [1455209081, 700000000]
    - fcu
  - !!python/object/new:geometry_msgs.msg._Quaternion.Quaternion
    state: [0.01, -0.02, 0.3, 0.9535]
  - [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]
  - !!python/object/new:geometry_msgs.msg._Vector3.Vector3
    state: [0.1, -0.2, 0.05]
  - [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]
  - !!python/object/new:geometry_msgs.msg._Vector3.Vector3
    state: [0.0, 0.0, 9.81]
  - [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]
"""


def test_ros_yaml_without_ros_classes():
    rng = replay.load_ros_yaml(io.StringIO(RANGE_YAML))
    assert [m._type for m in rng] == ["Range", "Range"]
    assert rng[0].header.seq == 3991 and rng[0].header.frame_id == "hrlv_ez4_sonar"
    assert rng[0].header.stamp.secs == 1455209081 and rng[0].header.stamp.nsecs == 675119360
    assert rng[1].range == 0.91 and rng[0].max_range == 7.0
    imu = replay.load_ros_yaml(io.StringIO(IMU_YAML))
    assert imu[0].orientation.w == 0.9535 and imu[0].angular_velocity.y == -0.2 and imu[0].linear_acceleration.z == 9.81
    # evaluate_exp.py:68-75 time base and :79-80 nearest association
    t = replay.stamps(rng, t0_secs=1455209081)
    assert np.allclose(t, [0.67511936, 1.09611936])
    assert replay.nearest(t, [0.0, 0.88, 0.89, 5.0]).tolist() == [0, 0, 1, 1]
    assert replay.nearest([1.0, 3.0], [2.0]).tolist() == [0]           # tie -> first, as np.argmin
    s = replay.imu_samples(imu, rng, [0, 0], [0, 1])
    q = imu[0].orientation
    R = vo.quat_to_rot(q.x, q.y, q.z, q.w)                              # evaluate_exp.py:88-92
    assert np.allclose(s["n"][0], R @ np.array([0, 0, 1.0])) and s["d"].tolist() == [0.83, 0.91]
    assert np.allclose(s["w"][1], [0.1, -0.2, 0.05]) and np.allclose(s["t"][0], [0, 0, 1])


def test_reference_recordings_load():
    if not ref_loader.available():
        pytest.skip(ref_loader.MISSING)
    path = os.path.join(ref_loader.REF, "flight_experiments", "hgtData.yaml")
    with open(path) as f:
        head = "".join(f.readline() for _ in range(13 * 200))
    msgs = replay.load_ros_yaml(io.StringIO(head))
    assert len(msgs) == 200 and all(m._type == "Range" for m in msgs)
    t = replay.stamps(msgs)
    assert np.all(np.diff(t) > 0) and 0.01 < np.median(np.diff(t)) < 0.05       # a ~47 Hz sonar
    assert 0.2 <= min(m.range for m in msgs) and max(m.range for m in msgs) <= 7.0
    tw = os.path.join(ref_loader.REF, "flight_experiments", "first_data", "vlsData.yaml")
    tws = replay.load_ros_yaml(tw)                                      # the whole file (437 messages)
    assert len(tws) > 400 and all(m._type == "TwistStamped" for m in tws)
    assert tws[0].twist.linear._type == "Vector3" and tws[0].header.frame_id == "map"
    assert [m.header.seq for m in tws[:3]] == [107, 108, 109] and replay.stamps(tws).shape == (len(tws),)


def test_velocity_kalman_equals_cv2():
    cv2 = pytest.importorskip("cv2")
    k = cv2.KalmanFilter(3, 3, 0)                                       # of_module.py:63-76, verbatim settings
    k.transitionMatrix = np.eye(3)
    k.controlMatrix = np.eye(3)
    k.measurementMatrix = np.eye(3)
    k.processNoiseCov = 1e-5 * np.eye(3)
    k.measurementNoiseCov = 1e1 * np.eye(3)
    k.errorCovPost = 0.1 * np.eye(3)
    k.statePost = np.zeros(3)
    mine = replay.VelocityKalman()
    rng = np.random.default_rng(3)
    for i in range(50):
        u = rng.normal(0, 0.01, 3)
        a, b = k.predict(u), mine.predict(u)                            # of_module.py:122
        assert np.allclose(np.ravel(a), np.ravel(b), rtol=1e-12, atol=1e-15)
        if i % 3 != 2:                                                  # of_module.py:139 skips frames (continue)
            z = -rng.normal([0.3, -0.1, 0.05], 0.05)                    # of_module.py:152 corrects with -v_obs
            assert np.allclose(np.ravel(k.correct(z)), np.ravel(mine.correct(z)), rtol=1e-12, atol=1e-15)
    assert np.allclose(k.errorCovPost, mine.P_post, rtol=1e-10)


def test_calc_height_inverts_the_pinhole_model():
    """of_library.py:270-286: a static ground point at height Z seen by a camera moving with vel has the flow
    (f vel_a - p_a vel_z) / Z per axis, so calc_height returns Z; the variance terms are non-negative."""
    rng = np.random.default_rng(1)
    n, f = 40, 600.0
    pos = rng.uniform(-200, 200, (n, 2))
    Z = rng.uniform(2.0, 9.0, n)
    vel = np.array([0.8, -0.5, 0.2])
    flow = np.stack([(f * vel[0] - pos[:, 0] * vel[2]) / Z, (f * vel[1] - pos[:, 1] * vel[2]) / Z], axis=1)
    h, he = of.calc_height(flow, 0.05 * np.ones((n, 2)), vel, 0.01 * np.ones(3), f, pos, 0.1 * np.ones((n, 2)))
    assert np.allclose(h, Z, rtol=1e-12) and np.all(he >= 0) and he.shape == (n,)


def test_convert_to_of_and_dynamic_immobile():
    n, f, dim = 30, 500.0, (640, 480)
    rng = np.random.default_rng(2)
    pos = np.stack([rng.uniform(0, 640, n), rng.uniform(0, 480, n)])                  # (2, N) as of_library.py:66-67
    height = rng.uniform(1.0, 4.0, n)
    speed, speed_err = np.array([0.4, -0.3, 0.0]), np.array([0.01, 0.01, 0.01])
    exp, err = of.convert_to_of(pos, 0.1 * np.ones((2, n)), speed, speed_err, height, 0.05, f, dim)
    tx, ty = of.pix_trans(dim)
    assert np.allclose(exp[0], (f - (pos[0] - tx) / height) * speed[0] / height)      # of_library.py:66
    assert np.allclose(exp[1], (f - (pos[1] - ty) / height) * speed[1] / height)
    assert np.all(np.asarray(err) >= 0)
    with pytest.raises(ValueError):
        of.convert_to_of(pos, np.ones((2, n)), speed, speed_err, np.zeros(n), 0.05, f, dim)      # of_library.py:56-57
    # a point moving exactly as expected is immobile; one moving 50 px off is not; the dummy position never is
    new = pos.T.reshape(n, 1, 2).copy()
    old = new - np.stack(exp, axis=-1).reshape(n, 1, 2)
    old[3] += 50.0
    dummy = -1.0
    old[7] = dummy
    keep = of.dynamic_immobile(new, 0.1 * np.ones((n, 1, 1)), old, 0.1 * np.ones((n, 1, 1)), speed, speed_err, f, dummy,
                               height, 0.05, dim).reshape(-1).astype(bool)
    assert not keep[3] and not keep[7] and keep[[0, 1, 2, 4, 5, 6]].all()


def test_eval_ft_ranks_by_weighted_score():
    """of_library.py:291-317: ascending score; with weight on the height-error term only the order is by error."""
    rng = np.random.default_rng(4)
    n = 25
    height, herr = rng.uniform(1, 5, n), rng.uniform(0.01, 1.0, n)
    pos, perr = rng.uniform(0, 640, (n, 1, 2)), rng.uniform(0, 1, (n, 1))
    hs, es, ps, pes = of.eval_ft([0, 1, 0, 0], height, herr, pos, perr, (640, 480))
    order = np.argsort(herr)
    assert np.array_equal(es, herr[order]) and np.array_equal(hs, height[order]) and np.array_equal(ps, pos[order])
    hs2, _, _, _ = of.eval_ft([1, 0, 0, 0], height, herr, pos, perr, (640, 480))
    assert np.array_equal(hs2, np.sort(height)[::-1])                  # (1 - height_norm) ascending = tallest first
