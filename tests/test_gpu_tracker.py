"""GPU parity of the device-resident feature lifecycle (ofb_tracker_*, csrc/tracker.cu) through the C ABI against
oracle/tracker_oracle.py and the cv2-made golden fixture (tests/golden/tracker_golden.npz). Tolerances: counts and
appended corners exact (documented float ties are resolved on the GPU's own lambda_min map), tracked positions
within 2e-4 px for 80 % of the points and 0.05 px for all (north star: 0.05 px), velocities within 1e-9 of the fp64
NumPy solve on the same kept points (north star: 1e-4 relative)."""
import os

import numpy as np
import pytest

import tracker_cases as tc
from conftest import GOLDEN
from oracle import image_oracle as io
from oracle import tracker_oracle
from oracle import velocity_oracle as vo
from test_oracle_tracker import LK_TOL, close_positions, teacher_from_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLDEN, "tracker_golden.npz"))


@pytest.fixture(scope="module")
def ofb200():
    import ofb200
    return ofb200


def imu_records(ofb200, samples):
    a = np.zeros(len(samples), ofb200._lib.IMU_DTYPE)
    for i, s in enumerate(samples):
        a["d"][i], a["n"][i], a["w"][i], a["t"][i] = s["d"], s["n"], s["w"], s["t"]
    return a


def priors(samples):
    if samples[0]["v_prior"] is None:
        return None
    return np.stack([s["v_prior"] for s in samples])


def same_record(a, b):
    """field-wise equality of two result records (the struct's tail padding is not defined)"""
    return all(np.array_equal(a[f], b[f]) for f in a.dtype.names)


def make_gpu_tracker(ofb200, ctx, kw, n_streams):
    return ofb200.StreamTracker(tc.W, tc.H, n_streams=n_streams, ctx=ctx, **kw)


def test_exclusion_mask_equals_cv2_circle(ofb200, ctx, g):
    for m, meta in zip(g["circle_masks"], g["circle_meta"]):
        radius, pts = int(meta[0]), meta[1:].reshape(-1, 2)
        got = ofb200.exclusion_mask(pts, radius, m.shape[1], m.shape[0], ctx=ctx)
        assert np.array_equal(got, m), "radius %d" % radius
    assert ofb200.exclusion_mask(np.zeros((0, 2)), 5, 33, 17, ctx=ctx).min() == 1


def check_topup(ofb200, ctx, kw, gray, kept_next, added, tag):
    """Appended corners = OpenCV's selection rule applied exactly to the GPU's own lambda_min map (tie contract of
    tests/test_gpu_vision.py), under the same mask / maxCorners the reference's loop would use."""
    fp = kw["feature_params"]
    K, mode = kw["max_features"], kw["topup"]
    mask = None
    if mode == "node" and kw.get("mask_radius", 30) > 0:
        mask = tracker_oracle.exclusion_mask(kept_next, kw.get("mask_radius", 30), tc.W, tc.H)
    mc = K if mode == "exp" else K - len(kept_next)
    eig = ofb200.cornerMinEigenVal(gray, fp["blockSize"], ctx=ctx)
    exp = io.select_features(eig, mc, fp["qualityLevel"], fp["minDistance"], mask)
    exp = np.zeros((0, 2), np.float32) if exp is None else exp.reshape(-1, 2)
    assert np.array_equal(added, exp), tag + ": top-up differs from the selection rule on the GPU's own map"


@pytest.mark.parametrize("name", sorted(tc.SCENARIOS))
def test_tracker_steps_vs_golden_and_oracle(ofb200, ctx, g, name):
    """Teacher-forced: before every step the point sets are set to the golden ones, so each step is compared with
    the cv2 + reference result on identical inputs. All streams of the scenario advance in one tracker."""
    frames, imus, kw = tc.build(name)
    S, T = len(frames), len(frames[0])
    teacher = teacher_from_golden(g, name)
    trk = make_gpu_tracker(ofb200, ctx, kw, S)
    try:
        identical_topups = total_topups = 0
        for k in range(T):
            if k > 0:
                trk.set_points([teacher[s][k] for s in range(S)])
            fr = np.stack([frames[s][k] for s in range(S)])
            samples = [imus[s][k] for s in range(S)]
            res, pts, kp, kn = trk.step(fr, imu_records(ofb200, samples), v_prior=priors(samples), want_points=True,
                                        want_kept=True)
            for s in range(S):
                tag = "%s stream %d step %d" % (name, s, k)
                for key in ("n_prev", "n_tracked", "n_kept", "n_added", "n_points"):
                    assert res[key][s] == g["%s_%s" % (name, key)][s, k], "%s: %s" % (tag, key)
                nk, npts, na = int(res["n_kept"][s]), int(res["n_points"][s]), int(res["n_added"][s])
                assert len(pts[s]) == npts
                assert close_positions(kn[s], g[name + "_kept_next"][s, k, :nk], LK_TOL), tag
                assert np.array_equal(kp[s], g[name + "_kept_prev"][s, k, :nk]), tag
                P = pts[s].reshape(-1, 2)
                if kw["topup"] != "module" or na == 0:
                    assert np.array_equal(P[:npts - na], kn[s]), tag + ": kept points lead the new set"
                if na:
                    total_topups += 1
                    gray = io.bgr2gray(frames[s][k]) if kw["bgr"] else frames[s][k]
                    added = P[npts - na:]
                    if np.array_equal(added, g[name + "_pts"][s, k, npts - na:npts]):
                        identical_topups += 1
                    check_topup(ofb200, ctx, kw, gray, kn[s], added, tag)
                solved = bool(res["flags"][s] & ofb200._lib.TRACK_SOLVED)
                assert solved == bool(g[name + "_solved"][s, k]), tag
                if solved:
                    gv = g[name + "_v"][s, k]
                    assert np.abs(res["v"][s] - gv).max() <= 2e-3 * np.abs(gv).max(), tag + ": velocity vs cv2 golden"
                    c = np.array([kw.get("principal") or vo.pix_trans((tc.W, tc.H))], np.float64)
                    x = (kn[s].astype(np.float64) - c) * kw["scaling"]
                    u = (kn[s] - kp[s]).astype(np.float64) * kw["scaling"]
                    sm = samples[s]
                    v, r_, rank, sv = vo.solve_lgs(x, u, sm["d"], sm["n"], sm["w"], None if kw["variant"] == "node" else sm["t"],
                                                   kw["variant"])
                    assert np.abs(res["v"][s] - v).max() <= 1e-9 * max(np.abs(v).max(), 1.0), tag + ": velocity vs fp64 solve"
                    assert int(res["rank"][s]) == int(rank), tag
                    assert np.allclose(res["s"][s], sv, rtol=1e-7), tag
                    if np.size(r_):
                        assert abs(res["res"][s] - float(r_[0])) <= 1e-7 * max(float(r_[0]), 1e-12), tag
        assert total_topups >= 2
        assert identical_topups >= total_topups - 1, "more than one top-up needed the tie rule"
    finally:
        trk.close()


def run_free(ofb200, ctx, kw, frames, imus, device_frames=False, borrow=False):
    import torch
    S, T = len(frames), len(frames[0])
    trk = make_gpu_tracker(ofb200, ctx, dict(kw, borrow_frames=borrow), S)
    out = []
    try:
        for k in range(T):
            fr = np.stack([frames[s][k] for s in range(S)])
            if device_frames:
                fr = torch.from_numpy(fr).cuda()
            samples = [imus[s][k] for s in range(S)]
            res, pts = trk.step(fr, imu_records(ofb200, samples), v_prior=priors(samples), want_points=True)
            out.append((res.copy(), pts))
    finally:
        trk.close()
    return out


def test_free_running_device_resident_chain(ofb200, ctx, g):
    """No teacher: the point set lives on the device for 8 frames; counts equal the cv2 chain and 80 % of the points
    stay within 0.05 px of it (points tracked into the occluding noise block wander chaotically)."""
    name = "exp"
    frames, imus, kw = tc.build(name)
    out = run_free(ofb200, ctx, kw, frames, imus)
    for k, (res, pts) in enumerate(out):
        for key in ("n_prev", "n_tracked", "n_kept", "n_added", "n_points"):
            assert res[key][0] == g["%s_%s" % (name, key)][0, k], "step %d: %s" % (k, key)
        assert close_positions(pts[0].reshape(-1, 2), g[name + "_pts"][0, k, :len(pts[0])], 0.05, worst=float("inf"))
        if res["flags"][0] & 1:
            gv = g[name + "_v"][0, k]
            assert np.abs(res["v"][0] - gv).max() <= 0.05 * np.abs(gv).max()


@pytest.mark.parametrize("name", ["module", "node"])
def test_streams_are_independent_and_device_frames_match(ofb200, ctx, name):
    """A multi-stream tracker gives every stream exactly what a single-stream tracker gives it, from host frames
    and from device-resident frames (bit-identical: same kernels, same per-stream data)."""
    frames, imus, kw = tc.build(name)
    if len(frames) == 1:        # make it a 3-stream fleet: the stream, a shifted copy and the stream again
        frames = [frames[0], frames[0][::-1].copy(), frames[0]]
        imus = [imus[0], imus[0][::-1], imus[0]]
    both = run_free(ofb200, ctx, kw, frames, imus)
    dev = run_free(ofb200, ctx, kw, frames, imus, device_frames=True)
    lent = run_free(ofb200, ctx, kw, frames, imus, device_frames=True, borrow=True)      # frames used in place
    for k in range(len(frames[0])):
        for s in range(len(frames)):
            assert same_record(lent[k][0][s], dev[k][0][s]) and np.array_equal(lent[k][1][s], dev[k][1][s])
    for s in range(len(frames)):
        single = run_free(ofb200, ctx, kw, [frames[s]], [imus[s]])
        for k in range(len(frames[0])):
            for other in (both, dev):
                assert same_record(other[k][0][s], single[k][0][0]), "stream %d step %d" % (s, k)
                assert np.array_equal(other[k][1][s], single[k][1][0])


def test_seeded_points_and_reset(ofb200, ctx):
    """set_points before the first frame (node:123-128 seeds test points): the first step keeps them and only tops
    up when they are few; reset() forgets frame and points."""
    frames, imus, kw = tc.build("exp")
    kw = dict(kw, min_features=3)
    trk = make_gpu_tracker(ofb200, ctx, kw, 1)
    try:
        seed = np.array([[50.0, 60.0], [200.0, 100.0], [120.0, 180.0], [260.0, 40.0], [30.0, 200.0]], np.float32)
        trk.set_points(seed)
        im = imu_records(ofb200, [imus[0][0]])
        res, pts = trk.step(frames[0][0], im, want_points=True)
        assert res["n_prev"][0] == 5 and res["n_added"][0] == 0 and not (res["flags"][0] & 1)
        assert np.array_equal(pts[0].reshape(-1, 2), seed)
        res, pts = trk.step(frames[0][1], imu_records(ofb200, [imus[0][1]]), want_points=True)
        exp, st, _ = io.pyrlk(frames[0][0], frames[0][1], seed, win=(15, 15), max_level=3, criteria=(3, 20, 0.03))
        assert res["n_tracked"][0] == int(st.sum())
        assert close_positions(pts[0].reshape(-1, 2)[:int(st.sum())], exp.reshape(-1, 2)[st.reshape(-1) == 1], LK_TOL)
        trk.reset()
        res, pts = trk.step(frames[0][2], im, want_points=True)
        assert res["n_prev"][0] == 0 and res["n_tracked"][0] == 0 and res["n_added"][0] == res["n_points"][0] > 0
    finally:
        trk.close()


def test_invalid_configurations_raise(ofb200, ctx):
    with pytest.raises(ValueError):
        ofb200.StreamTracker(320, 240, max_features=10, min_features=10, ctx=ctx)
    with pytest.raises(ValueError):
        ofb200.StreamTracker(320, 240, n_streams=0, ctx=ctx)
    trk = ofb200.StreamTracker(320, 240, ctx=ctx)
    try:
        with pytest.raises(ValueError):
            trk.step(np.zeros((100, 100), np.uint8), np.zeros(1, ofb200._lib.IMU_DTYPE))
        with pytest.raises(ValueError):
            trk.set_points(np.zeros((trk.capacity + 1, 2), np.float32))
    finally:
        trk.close()


def test_fleet_size_streams_match_single_stream(ofb200, ctx):
    """Fleet shape (SURVEY 8d C5, scaled to 24 streams of 1280x720, 500 features): streams 0, 11 and 23 of the
    fleet tracker equal single-stream trackers run on the same frames."""
    import synth
    w, h, S, T = 1280, 720, 24, 3
    base = [synth.texture(h + 16, w + 16, 40 + i) for i in range(3)]
    frames = [[np.ascontiguousarray(base[s % 3][2 * k + (s % 5):2 * k + (s % 5) + h, 3 * k + (s % 7):3 * k + (s % 7) + w]) for k in range(T)]
              for s in range(S)]
    kw = dict(max_features=500, min_features=480, topup="node", mask_radius=12, variant="node", scaling=1.0 / (0.8 * w),
              lk_params=dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03)))
    imu = np.zeros(S, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"] = 1.5, [0.0, 0.0, 1.0]

    def run(sel):
        trk = ofb200.StreamTracker(w, h, n_streams=len(sel), ctx=ctx, **kw)
        try:
            return [trk.step(np.stack([frames[s][k] for s in sel]), imu[sel], want_points=True) for k in range(T)]
        finally:
            trk.close()
    fleet = run(list(range(S)))
    assert fleet[0][0]["n_points"].min() == 500
    assert fleet[T - 1][0]["n_tracked"].min() > 400 and (fleet[T - 1][0]["flags"] & 1).all()
    for s in (0, 11, 23):
        single = run([s])
        for k in range(T):
            assert same_record(fleet[k][0][s], single[k][0][0]), "stream %d step %d" % (s, k)
            assert np.array_equal(fleet[k][1][s], single[k][1][0])
    # pure shift by (3, 2) px per frame at height 1.5 m: v = -(3, 2) / f * d
    v = fleet[T - 1][0]["v"]
    assert np.abs(v[:, 0] + 3 * 1.5 / (0.8 * w)).max() < 2e-4 and np.abs(v[:, 1] + 2 * 1.5 / (0.8 * w)).max() < 2e-4


def test_replay_flight_end_to_end(ofb200, ctx):
    """evaluate_exp.py:77-120 through ofb200.replay: nearest IMU / sonar sample per frame, then the tracker. The
    result equals stepping the tracker by hand with the associated samples."""
    from ofb200 import replay
    frames, imus, kw = tc.build("exp")
    T = len(frames[0])
    M = replay.RosMessage
    cam_t = 0.05 * np.arange(T)
    imu_msgs, rng_msgs = [], []
    for k in range(3 * T):                                             # IMU at 3x the camera rate, offset by 4 ms
        q = np.array([0.01 * np.sin(k), 0.02 * np.cos(k), 0.1, 1.0]); q /= np.linalg.norm(q)
        stamp = M("Time", [100 + int((0.004 + k * 0.05 / 3) // 1), int(((0.004 + k * 0.05 / 3) % 1) * 1e9)])
        imu_msgs.append(M("Imu", [M("Header", [k, stamp, "fcu"]), M("Quaternion", list(q)), [0.0] * 9,
                                  M("Vector3", [0.01 * k, -0.02, 0.03]), [0.0] * 9, M("Vector3", [0, 0, 9.81]), [0.0] * 9]))
    for k in range(2 * T):
        stamp = M("Time", [100, int((0.01 + k * 0.025) * 1e9)])
        rng_msgs.append(M("Range", [M("Header", [k, stamp, "sonar"]), 0, 0.0, 0.2, 7.0, 1.0 + 0.01 * k]))
    it, rt = replay.stamps(imu_msgs, 100), replay.stamps(rng_msgs, 100)
    trk = make_gpu_tracker(ofb200, ctx, kw, 1)
    try:
        got = [(k, r.copy(), s.copy()) for k, r, s in replay.replay_flight(frames[0], cam_t, imu_msgs, it, rng_msgs, rt, trk,
                                                                          translation=(0.02, 0.0, 0.205))]
    finally:
        trk.close()
    ii, hi = replay.nearest(it, cam_t), replay.nearest(rt, cam_t)
    assert ii.tolist() == [int(np.argmin(np.abs(it - t))) for t in cam_t]
    samples = replay.imu_samples(imu_msgs, rng_msgs, ii, hi, (0.02, 0.0, 0.205))
    trk = make_gpu_tracker(ofb200, ctx, kw, 1)
    try:
        for k in range(T):
            r = trk.step(frames[0][k], samples[k:k + 1])
            assert same_record(r[0], got[k][1]), "frame %d" % k
            assert got[k][2]["d"] == rng_msgs[hi[k]].range
    finally:
        trk.close()
    assert sum(int(g_[1]["flags"]) & 1 for g_ in got) == T - 1


def test_initialize_ft_as_intended(ofb200, ctx):
    """of_library.py:231-263 (8f-3): first frame -> goodFeaturesToTrack -> LK steps with the dynamic-immobile filter ->
    eval_ft ranking; ValueError for non-positive iterations / end_count (of_library.py:240-243)."""
    import ofb200.of_library as of
    frames, _, _ = tc.build("exp")
    fp = dict(maxCorners=40, qualityLevel=0.05, minDistance=10, blockSize=7)
    lk = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
    # the window drifts by (7.5, -3.25) px per frame: with f = 256 px and height 2 m the camera moves at
    # v = flow * Z / f; a generous velocity error keeps every static point inside the immobile band
    f, Z = 256.0, 2.0
    vel = np.array([-7.5 * Z / f, 3.25 * Z / f, 0.0])
    with pytest.raises(ValueError):
        of.initialize_ft(list(frames[0]), fp, lk, 0, 10, vel, 0.5 * np.ones(3), f, -1.0, (tc.W, tc.H), [1, 1, 1, 1])
    with pytest.raises(ValueError):
        of.initialize_ft(list(frames[0]), fp, lk, 2, 0, vel, 0.5 * np.ones(3), f, -1.0, (tc.W, tc.H), [1, 1, 1, 1])
    h, he, pos, perr = of.initialize_ft(list(frames[0][:4]), fp, lk, 3, 10, vel, 0.5 * np.ones(3), f, -1.0, (tc.W, tc.H),
                                        [0, 1, 0, 0])
    assert len(h) == len(he) == len(pos) == len(perr) and 10 <= len(h) <= 40
    assert np.all(np.diff(he) >= 0), "eval_ft with weight on the height error sorts by it"
    assert np.abs(np.median(np.abs(h)) - Z) < 0.5 * Z


@pytest.mark.parametrize("name", ["exp", "node", "module"])
def test_graph_replay_equals_plain_launches(ofb200, ctx, name, monkeypatch):
    """Small fleets fed from host memory replay the steady-state step from a captured CUDA graph (include/ofb200.h,
    ofb_tracker_graph_steps). Results and the device-resident point sets are identical to the launch-by-launch path
    (OFB_TRACKER_GRAPH=0), including steps whose top-up fires inside the graph."""
    frames, imus, kw = tc.build(name)
    S, T = len(frames), len(frames[0])
    # a longer run: the sequence forwards, then backwards
    order = list(range(T)) + list(range(T - 2, -1, -1))

    def run(graph):
        monkeypatch.setenv("OFB_TRACKER_GRAPH", "1" if graph else "0")
        trk = make_gpu_tracker(ofb200, ctx, kw, S)
        out = []
        try:
            for j, k in enumerate(order):
                if j == 8:
                    # another call on the same context grows its scratch arenas (they move): the graphs hold stale
                    # addresses and must be rebuilt, not replayed
                    big = np.random.default_rng(3).integers(0, 256, (768, 1024), dtype=np.uint8)
                    assert ofb200.goodFeaturesToTrack(big, 0, 0.001, 1, blockSize=3, ctx=ctx) is not None
                samples = [imus[s][k] for s in range(S)]
                fr = np.stack([frames[s][k] for s in range(S)])
                out.append(trk.step(fr, imu_records(ofb200, samples), v_prior=priors(samples)).copy())
            n_graph = trk.graph_info()
            res, pts = trk.step(np.stack([frames[s][1] for s in range(S)]), imu_records(ofb200, [imus[s][1] for s in range(S)]),
                                v_prior=priors([imus[s][1] for s in range(S)]), want_points=True)
            out.append(res.copy())
        finally:
            trk.close()
        return out, pts, n_graph
    plain, ppts, n0 = run(False)
    graph, gpts, n1 = run(True)
    assert n0 == (0, False) and n1 == (len(order) - 3, False), (n0, n1)   # three plain steps first
    assert sum(int((r["n_added"] > 0).sum()) for r in graph[3:]) >= 1, "no top-up inside a graph step: weak test"
    for k, (a, b) in enumerate(zip(plain, graph)):
        for s in range(S):
            assert same_record(a[s], b[s]), "step %d stream %d" % (k, s)
    for s in range(S):
        assert np.array_equal(ppts[s], gpts[s])


@pytest.mark.parametrize("bgr", [False, True])
def test_odd_geometry_matches_the_pair_path(ofb200, ctx, bgr):
    """Width/height that are not multiples of 4 or 16 (staging pitch != row length, unaligned BGR rows), two streams,
    enough steps to reach the graph replay: tracks and velocity equal ofb_frame_pairs on the same grey frames."""
    import synth
    w, h, K = 333, 247, 120
    seq = []
    for s in range(2):
        big = synth.texture(h + 40, w + 40, 70 + s)
        seq.append([np.ascontiguousarray(big[3 * k + s:3 * k + s + h, 2 * k:2 * k + w]) for k in range(6)])
    col = [[tc._bgr(f, s) for f in seq[s]] for s in range(2)]
    gray = [[io.bgr2gray(f) for f in col[s]] for s in range(2)] if bgr else seq
    kw = dict(max_features=K, min_features=K // 4, topup="node", mask_radius=9, variant="node", scaling=1.0 / 270.0,
              feature_params=dict(qualityLevel=0.02, minDistance=7, blockSize=3), bgr=bgr)
    imu = np.zeros(2, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"] = [1.2, 2.0], [0.0, 0.0, 1.0]
    trk = ofb200.StreamTracker(w, h, n_streams=2, ctx=ctx, **kw)
    cfg = ofb200.make_pair_cfg(w, h, K, 0.02, 7, 3, (15, 15), 3, (3, 20, 0.03), variant="node", pos_scale=1.0 / 270.0,
                               flow_scale=1.0 / 270.0, detect=False)
    src = col if bgr else seq
    try:
        res, pts = trk.step(np.stack([src[0][0], src[1][0]]), imu, want_points=True)
        for k in range(1, 6):
            want = k in (1, 2)                       # later steps without optional outputs: graph replay
            out = trk.step(np.stack([src[0][k], src[1][k]]), imu, want_points=want)
            prev = np.zeros((2, K, 2), np.float32); n_in = np.zeros(2, np.int32)
            for s in range(2):
                n_in[s] = len(pts[s]); prev[s, :n_in[s]] = pts[s].reshape(-1, 2)
            ref, pp, pn, st = ofb200.frame_pairs(np.stack([gray[0][k - 1], gray[1][k - 1]]), np.stack([gray[0][k], gray[1][k]]), imu,
                                                 cfg, pts_in=prev, n_in=n_in, want_tracks=True, ctx=ctx)
            res = out[0] if want else out
            for s in range(2):
                ok = st[s, :n_in[s]] == 1
                assert int(res["n_tracked"][s]) == int(ok.sum()) and int(res["n_prev"][s]) == int(n_in[s])
                assert np.abs(res["v"][s] - ref["v"][s]).max() <= 1e-12 * max(1.0, np.abs(ref["v"][s]).max())
                if want:
                    assert np.array_equal(out[1][s].reshape(-1, 2)[:int(ok.sum())], pn[s, :n_in[s]][ok])
            if want:
                pts = out[1]
            else:                                    # keep following the chain through the pair path's own tracks
                pts = [np.concatenate([pn[s, :n_in[s]][st[s, :n_in[s]] == 1]]) for s in range(2)]
                assert all(int(res["n_added"][s]) == 0 for s in range(2)), "a top-up would need the point set back"
        assert trk.graph_steps() >= 2
    finally:
        trk.close()


def test_fleet_tracker_single_rank_equals_stream_tracker(ofb200, ctx):
    """ofb200.FleetTracker without a process group (world size 1): the gathered velocity table is the StreamTracker's
    (the multi-rank gather is covered by the gloo test in test_host_logic.py and by tools/fleet_smoke.py over NCCL)."""
    frames, imus, kw = tc.build("module")
    S, T = len(frames), 3
    fleet = ofb200.FleetTracker(S, tc.W, tc.H, ctx=ctx, **kw)
    ref = make_gpu_tracker(ofb200, ctx, kw, S)
    try:
        assert fleet.streams == list(range(S)) and fleet.world == 1
        for k in range(T):
            samples = [imus[s][k] for s in range(S)]
            fr = np.stack([frames[s][k] for s in range(S)])
            fleet.step(np.stack(fleet.select(list(fr))), imu_records(ofb200, samples), v_prior=priors(samples))
            r = ref.step(fr, imu_records(ofb200, samples), v_prior=priors(samples))
        table = fleet.gather_velocities()
        solved = (r["flags"] & 1) != 0
        assert np.array_equal(np.isnan(table[:, 0]), ~solved)
        assert np.array_equal(table[solved], r["v"][solved])
    finally:
        fleet.close()
        ref.close()
