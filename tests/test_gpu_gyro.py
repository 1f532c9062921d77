"""Gyro prediction of the LK tracks on the GPU (include/ofb200.h `ofb_gyro_predict`, `ofb_frame_pairs_gyro`,
`ofb_tracker_set_gyro_prediction`) against oracle/gyro_oracle.py, cv2 and the fp64 solve; and the scenes it exists for."""
import ctypes as C

import numpy as np
import pytest

import gyro_cases as gc
import synth
import tracker_cases as tc
from oracle import camera_oracle as co
from oracle import fb_oracle, tracker_oracle
from oracle import gyro_oracle as go
from oracle import velocity_oracle as vo
from test_gpu_camera import cam_for, relerr
from test_gpu_tracker import imu_records, same_record

pytestmark = pytest.mark.gpu

CAM = np.load(__import__("os").path.join(__import__("conftest").ROOT, "tests", "golden", "camera_golden.npz"))
LK = dict(winSize=gc.LK[0], maxLevel=gc.LK[1], criteria=gc.LK[2])


@pytest.fixture(scope="module")
def ofb200():
    import ofb200
    return ofb200


def ulps(a, b):
    """distance in float32 ulps"""
    ia = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    ib = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


def scene_model():
    return go.pinhole(gc.CX, gc.CY, 1.0 / gc.F, 1.0 / (gc.F * gc.DT))


def scene_cfg(ofb200, K=gc.N_FEATURES):
    return ofb200.make_pair_cfg(gc.W, gc.H, K, 0.01, 10, 7, LK["winSize"], LK["maxLevel"], LK["criteria"], variant="node",
                                **gc.pinhole_kw())


def scene_imu(ofb200, ws):
    imu = np.zeros(len(ws), ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"][:, 2] = 3.0, 1.0
    imu["w"] = np.asarray(ws)
    return imu


# ---- the predictor ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["pinhole", "c0", "c3", "c5", "c7"])
@pytest.mark.parametrize("device", [False, True])
def test_predict_equals_oracle(ofb200, ctx, case, device):
    """fp32 guesses identical to the NumPy oracle, or one ulp off where the fp64 value rounds at a boundary; pinhole and
    0 / 4 / 5 / 8-coefficient cameras, host and device pointers"""
    import torch
    rng = np.random.default_rng(9)
    p = np.c_[rng.uniform(0, gc.W, 2000), rng.uniform(0, gc.H, 2000)].astype(np.float32)
    worst = 0
    for w in ([0.0, 0.0, 0.0], [0.4, -0.3, 0.9], [3.0, 4.5, -1.0], [1e-7, 0.0, -2e-7], [0.0, 60.0, 0.0]):
        if case == "pinhole":
            cfg = scene_cfg(ofb200)
            cam, model = None, scene_model()
        else:
            D = CAM[case + "_dist"][:int(CAM[case + "_n_dist"])]
            cam = ofb200.make_camera(CAM["K"], D if len(D) else None, 1.0 / gc.DT, int(CAM[case + "_iterations"]))
            cfg, model = None, go.camera(CAM["K"], D, 1.0 / gc.DT, int(CAM[case + "_iterations"]))
        ref = go.predict(p, w, model)
        if device:
            dp = torch.from_numpy(p).cuda()
            dw = torch.tensor(w, dtype=torch.float64, device="cuda")
            dg = torch.zeros_like(dp)
            ofb200._lib.check(ctx.lib.ofb_gyro_predict(ctx.h, C.byref(cfg) if cfg is not None else None,
                                                       C.byref(cam) if cam is not None else None, ofb200._lib.ptr(dp),
                                                       len(p), ofb200._lib.ptr(dw), ofb200._lib.ptr(dg)))
            ctx.sync()
            got = dg.cpu().numpy()
        else:
            got = ofb200.gyro_predict(p, w, camera=cam, cfg=cfg, ctx=ctx).reshape(-1, 2)
        if not np.any(w):
            assert np.array_equal(got, p)
        d = ulps(got, ref)
        assert d.max() <= 1, (case, w, d.max())
        worst = max(worst, int((d > 0).sum()))
    assert worst <= 0.01 * len(p)


def test_predict_invalid_input(ofb200, ctx):
    p = np.zeros((4, 2), np.float32)
    g = np.zeros_like(p)
    w = np.zeros(3)
    cfg = scene_cfg(ofb200)
    lib, ptr = ctx.lib, ofb200._lib.ptr
    assert lib.ofb_gyro_predict(ctx.h, C.byref(cfg), None, ptr(p), 4, None, ptr(g)) == ofb200._lib.OFB_E_INVALID
    assert lib.ofb_gyro_predict(ctx.h, C.byref(cfg), None, ptr(p), -1, ptr(w), ptr(g)) == ofb200._lib.OFB_E_INVALID
    cfg.flow_scale = 0.0
    assert lib.ofb_gyro_predict(ctx.h, C.byref(cfg), None, ptr(p), 4, ptr(w), ptr(g)) == ofb200._lib.OFB_E_INVALID
    cfg.flow_scale = 1e-320                             # pos_scale / flow_scale overflows
    assert lib.ofb_gyro_predict(ctx.h, C.byref(cfg), None, ptr(p), 4, ptr(w), ptr(g)) == ofb200._lib.OFB_E_INVALID
    a = np.zeros((1, gc.H, gc.W), np.uint8)
    res = np.zeros(1, ofb200._lib.RESULT_DTYPE)
    imu = scene_imu(ofb200, [w])
    cfg.flow_scale = 0.0
    rc = lib.ofb_frame_pairs_gyro(ctx.h, C.byref(cfg), None, 0.0, 1, 1, ptr(a), ptr(a), gc.W, gc.W * gc.H, ptr(imu), None, None,
                                  ptr(res), None, None, None)
    assert rc == ofb200._lib.OFB_E_INVALID
    trk = ofb200.StreamTracker(64, 48, ctx=ctx, scaling=1.0, flow_scaling=0.0)
    try:
        with pytest.raises(ValueError):
            trk.set_gyro_prediction(True)
        assert lib.ofb_tracker_set_gyro_prediction(trk.h, 1) == ofb200._lib.OFB_E_INVALID
    finally:
        trk.close()


# ---- frame pairs ------------------------------------------------------------------------------------------------
def test_frame_pairs_rotation_scene_vs_lk_with_initial_flow(ofb200, ctx):
    """status identical to LK with OPTFLOW_USE_INITIAL_FLOW on the oracle's guesses (C oracle, and cv2 live when
    installed), positions within 2e-4 px; and the scene is why the prediction exists"""
    cv2 = None
    try:
        import cv2
    except ImportError:
        pass
    names = list(gc.ROTATIONS)
    scenes = [gc.rotation_scene(n) for n in names]
    prev = np.stack([s[0] for s in scenes]); nxt = np.stack([s[1] for s in scenes])
    imu = scene_imu(ofb200, [s[2] for s in scenes])
    cfg = scene_cfg(ofb200)
    res, pp, pn, st = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx, gyro_prediction=True)
    _, qp, qn, qs = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx)
    assert np.array_equal(pp, qp)
    msg = []
    for i, (a, b, w) in enumerate(scenes):
        n = int(res["n_features"][i])
        p0 = pp[i, :n]
        g = go.predict(p0, w, scene_model())
        for lk in ([go.pyrlk_init] + ([lambda a_, b_, p_, g_, *r: cv2.calcOpticalFlowPyrLK(
                a_, b_, p_.reshape(-1, 1, 2), g_.reshape(-1, 1, 2).copy(), winSize=r[0], maxLevel=r[1], criteria=r[2],
                flags=cv2.OPTFLOW_USE_INITIAL_FLOW)] if cv2 else [])):
            r1, rs, _ = lk(a, b, p0, g, *gc.LK)
            rs = rs.ravel()
            assert np.array_equal(st[i, :n], rs)
            ok = rs == 1
            assert np.abs(pn[i, :n][ok] - r1.reshape(-1, 2)[ok]).max() <= 2e-4
        t, inside = gc.true_positions(p0, w)
        good = (st[i, :n] == 1) & (np.abs(pn[i, :n] - t).max(1) < 0.5)
        plain = (qs[i, :n] == 1) & (np.abs(qn[i, :n] - t).max(1) < 0.5)
        msg.append("%s: plain LK %d / %d, predicted %d / %d inside" % (names[i], plain.sum(), n, (good & inside).sum(),
                                                                      inside.sum()))
        assert plain.sum() < 0.5 * n, msg[-1]
        assert (good & inside).sum() >= 0.95 * inside.sum(), msg[-1]
    print("; ".join(msg))


def test_frame_pairs_velocity_error_falls(ofb200, ctx):
    """warp_pair scenes dominated by a 3 rad/s rotation: the velocity error of the solve falls with the prediction, and
    the velocity is the fp64 solve on the kept tracks"""
    e_plain, e_gyro = [], []
    for k in range(4):
        a, b, mo = gc.rotation_pair(k)
        imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
        imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
        cfg = ofb200.make_pair_cfg(gc.W, gc.H, gc.N_FEATURES, 0.01, 10, 7, LK["winSize"], LK["maxLevel"], LK["criteria"],
                                   variant="node", principal=(mo["cx"], mo["cy"]), pos_scale=1.0 / mo["f"],
                                   flow_scale=1.0 / (mo["f"] * mo["dt"]))
        for gyro, errs in ((False, e_plain), (True, e_gyro)):
            res, pp, pn, st = ofb200.frame_pairs(a[None], b[None], imu, cfg, want_tracks=True, ctx=ctx, gyro_prediction=gyro)
            n = int(res["n_features"][0])
            ok = st[0, :n] == 1
            x = (pn[0, :n][ok].astype(np.float64) - [cfg.cx, cfg.cy]) * cfg.pos_scale
            u = (pn[0, :n][ok] - pp[0, :n][ok]).astype(np.float64) * cfg.flow_scale
            v = vo.solve_lgs(x, u, mo["d"], mo["n"], mo["w"], variant="node")[0]
            assert relerr(res["v"][0], v) <= 1e-6
            errs.append(np.abs(res["v"][0] - mo["v"]).max() / np.abs(mo["v"]).max())
    msg = "velocity error plain %s, predicted %s" % (np.round(e_plain, 4).tolist(), np.round(e_gyro, 4).tolist())
    print(msg)
    assert np.mean(e_gyro) < 0.5 * np.mean(e_plain), msg


def test_frame_pairs_routes_identical(ofb200, ctx):
    """resident single pass, resident twin chunks, host-frame pipeline, sequence layout: one result, with and without
    the forward-backward check"""
    import torch
    h, w, n = 240, 320, 12
    frames = np.stack([synth.make_pair(h, w, 3, k, max_disp=5.0)[0 if k == 0 else 1] for k in range(n + 1)])
    imu = np.zeros(n, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"][:, 2] = 2.0, 1.0
    imu["w"] = np.random.default_rng(1).normal(0, 1.0, (n, 3))
    cfg = ofb200.make_pair_cfg(w, h, 150, 0.01, 8, 7, (15, 15), 3, (3, 20, 0.03), variant="node", pos_scale=1 / 256.0,
                               flow_scale=1 / 8.0)
    d = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    for T in (None, 0.5):
        kw = dict(want_tracks=True, ctx=ctx, fb_threshold=T, gyro_prediction=True)
        host = ofb200.frame_pairs(frames[:-1].copy(), frames[1:].copy(), imu, cfg, **kw)
        seq = ofb200.frame_sequence(frames, imu, cfg, **kw)
        twin = ofb200.frame_pairs(d[:-1].contiguous(), d[1:].contiguous(), imu, cfg, **kw)
        ofb200._lib.check(ctx.lib.ofb_ctx_set_profile(ctx.h, 1))
        try:
            single = ofb200.frame_pairs(d[:-1].contiguous(), d[1:].contiguous(), imu, cfg, **kw)
        finally:
            ofb200._lib.check(ctx.lib.ofb_ctx_set_profile(ctx.h, 0))
        for other in (seq, twin, single):
            assert all(same_record(host[0][i], other[0][i]) for i in range(n))
            for x, y in zip(host[1:], other[1:]):
                assert np.array_equal(x, y)
        # detect = 0 with the detected points as input: the same tracks
        pts_in, n_in = host[1], host[0]["n_features"].astype(np.int32)
        cfg.detect = 0
        given = ofb200.frame_pairs(frames[:-1], frames[1:], imu, cfg, pts_in=pts_in, n_in=n_in, **kw)
        cfg.detect = 1
        assert np.array_equal(given[2], host[2]) and np.array_equal(given[3], host[3])


def test_frame_pairs_with_camera(ofb200, ctx):
    """the camera's lens model predicts, LK is the oracle's from those guesses, the solve is the calibrated fp64 one"""
    a, b, mo = gc.rotation_pair(1)
    imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
    cfg = ofb200.make_pair_cfg(gc.W, gc.H, 300, 0.01, 10, 7, LK["winSize"], LK["maxLevel"], LK["criteria"], variant="node")
    K = np.array([[mo["f"] * 1.01, 0.0, mo["cx"] + 1.5], [0.0, mo["f"], mo["cy"] - 0.5], [0.0, 0.0, 1.0]])
    cam = (K, np.array([-0.05, 0.01, 0.0005, -0.0005, 0.001]), 1.0 / mo["dt"], 20)
    res, pp, pn, st = ofb200.frame_pairs(a[None], b[None], imu, cfg, want_tracks=True, ctx=ctx, camera=cam, gyro_prediction=True)
    n = int(res["n_features"][0])
    g = go.predict(pp[0, :n], mo["w"], go.camera(*cam))
    r1, rs, _ = go.pyrlk_init(a, b, pp[0, :n], g, *gc.LK)
    assert np.array_equal(st[0, :n], rs.ravel())
    ok = st[0, :n] == 1
    assert ok.sum() > 0.5 * n
    assert np.abs(pn[0, :n][ok] - r1.reshape(-1, 2)[ok]).max() <= 2e-4
    x, u = co.calibrate(pn[0, :n][ok], pp[0, :n][ok], cam)
    v = vo.solve_lgs(x, u, mo["d"], mo["n"], mo["w"], variant="node")[0]
    assert relerr(res["v"][0], v) <= 1e-6


def test_frame_pairs_with_fb_check(ofb200, ctx):
    """prediction + forward-backward check against the composition forward from g, backward from p1 + (p0 - g) (the C
    oracle; cv2 live when installed): no status differs except for points within 0.05 px of T"""
    try:
        import cv2
    except ImportError:
        cv2 = None
    T = 1.0
    names = list(gc.ROTATIONS)
    scenes = [gc.rotation_scene(n) for n in names]
    prev = np.stack([s[0] for s in scenes]); nxt = np.stack([s[1] for s in scenes])
    imu = scene_imu(ofb200, [s[2] for s in scenes])
    cfg = scene_cfg(ofb200)
    res, pp, pn, st = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx, gyro_prediction=True, fb_threshold=T)
    _, _, pn0, _ = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx, gyro_prediction=True)
    assert np.array_equal(pn, pn0)                      # the forward results are the check's input, unchanged
    covered = total = 0
    for i, (a, b, w) in enumerate(scenes):
        n = int(res["n_features"][i])
        p0 = pp[i, :n]
        g = go.predict(p0, w, scene_model())
        lks = [go.pyrlk_init]
        if cv2:
            lks.append(lambda a_, b_, p_, g_, *r: cv2.calcOpticalFlowPyrLK(
                a_, b_, np.asarray(p_, np.float32).reshape(-1, 1, 2), np.asarray(g_, np.float32).reshape(-1, 1, 2).copy(),
                winSize=r[0], maxLevel=r[1], criteria=r[2], flags=cv2.OPTFLOW_USE_INITIAL_FLOW))
        for lk in lks:
            p1, s1, _ = lk(a, b, p0, g, *gc.LK)
            p1 = np.asarray(p1, np.float32).reshape(-1, 2)
            p0r, s0, _ = lk(b, a, p1, p1 + (p0 - g), *gc.LK)
            gst, gfb = fb_oracle.fb_check(p0, p1, s1, p0r, s0, T)
            near = np.abs(gfb.astype(np.float64) - T) <= 0.05
            diff = st[i, :n] != gst
            assert not (diff & ~near).any(), names[i]
            covered += int((diff & near).sum()); total += n
        assert (st[i, :n] == 1).sum() > 0.7 * n
    assert covered <= 0.01 * total


# ---- tracker ----------------------------------------------------------------------------------------------------
W_STEP = np.array([0.004, -0.006, 0.003])           # rad per frame (the tracker cases' flow_scale = scaling: dt = 1)


def gyro_imu(im, k):
    im = dict(im)
    im["w"] = W_STEP * (1 + 0.3 * np.sin(k))
    return im


@pytest.mark.parametrize("seed,camera", [(21, False), (22, False), (24, True)])
def test_tracker_vs_oracle(ofb200, ctx, seed, camera):
    """random_case sequences teacher-forced on TrackerOracle / CameraTrackerOracle with the gyro engine (and the
    forward-backward check on one seed): the same counts step by step, the fp64 solve on the GPU's kept tracks"""
    frames, imus, kw = tc.random_case(seed)
    T = 0.3 if seed == 22 else 0.0
    okw = {k: v for k, v in kw.items() if k != "bgr"}
    if camera:
        cam = cam_for(kw)
        eng = go.GyroEngine(tracker_oracle.Engine(), go.camera(*cam), T)
        orc = co.CameraTrackerOracle(tc.W, tc.H, cam, engine=eng, **okw)
    else:
        cam = None
        c = vo.pix_trans((tc.W, tc.H))
        eng = go.GyroEngine(tracker_oracle.Engine(), go.pinhole(c[0], c[1], kw["scaling"], kw["scaling"]), T)
        orc = tracker_oracle.TrackerOracle(tc.W, tc.H, engine=eng, **okw)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, camera=cam, fb_threshold=T or None, gyro_prediction=True, **kw)
    solved = 0
    try:
        for k in range(len(frames[0])):
            im = gyro_imu(imus[0][k], k)
            eng.w = im["w"]
            trk.set_points(orc.pts)
            o = orc.step(frames[0][k], im["d"], im["n"], im["w"], im["t"], im["v_prior"])
            res, kp, kn = trk.step(frames[0][k], imu_records(ofb200, [im]), v_prior=im["v_prior"][None], want_kept=True)
            for key in ("n_prev", "n_tracked", "n_kept"):
                assert int(res[key][0]) == int(o[key]), (seed, k, key)
            if res["flags"][0] & 1:
                solved += 1
                if camera:
                    x, u = co.calibrate(kn[0], kp[0], cam)
                else:
                    x = (kn[0].astype(np.float64) - vo.pix_trans((tc.W, tc.H))) * kw["scaling"]
                    u = (kn[0] - kp[0]).astype(np.float64) * kw["scaling"]
                v = vo.solve_lgs(x, u, im["d"], im["n"], im["w"], None if kw["variant"] == "node" else im["t"], kw["variant"])[0]
                assert relerr(res["v"][0], v) <= 1e-9, (seed, k)
                assert relerr(res["v"][0], o["v"]) <= 2e-3, (seed, k)
    finally:
        trk.close()
    assert solved >= 2


SWITCH = {3: True, 6: False, 9: True}


def run_switching(ofb200, kw, frames, imus, mode, monkeypatch, camera=None, switch=SWITCH, start=False, zero_w=False):
    """as tests/test_gpu_fb.run_switching, switching the gyro prediction"""
    import torch
    monkeypatch.setenv("OFB_TRACKER_GRAPH", "0" if mode == "plain" else "1")
    monkeypatch.setenv("OFB_TRACKER_SPLIT_SOLVE", "0" if mode == "nosplit" else "1")
    ctx = ofb200.Context(0)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, camera=camera, gyro_prediction=start, **kw)
    order = list(range(len(frames))) + list(range(len(frames) - 2, -1, -1))
    out = []
    dev = mode in ("split", "nosplit")
    d_res = torch.zeros(C.sizeof(ofb200._lib.TrackResult), dtype=torch.uint8, device="cuda") if dev else None
    try:
        for j, k in enumerate(order):
            if j in switch:
                trk.set_gyro_prediction(switch[j])
            s = gyro_imu(imus[k], k)
            if zero_w:
                s["w"] = np.zeros(3)
            im = imu_records(ofb200, [s])
            if dev:
                fr = torch.from_numpy(frames[k]).cuda()
                d_imu = torch.from_numpy(im.view(np.uint8).copy()).cuda()
                ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, ofb200._lib.ptr(fr), tc.W, tc.W * tc.H, ofb200._lib.ptr(d_imu),
                                                           None, ofb200._lib.ptr(d_res), None, None, None, None))
                ctx.sync()
                out.append(d_res.cpu().numpy().view(ofb200._lib.TRACK_RESULT_DTYPE).copy())
            else:
                out.append(trk.step(frames[k], im).copy())
        graph_steps = trk.graph_steps()
    finally:
        trk.close()
        ctx.close()
    return out, graph_steps, order


@pytest.mark.parametrize("scenario,camera", [("exp", False), ("node", True)])
def test_tracker_switch_identical_in_every_mode(ofb200, monkeypatch, scenario, camera):
    """on / off / on mid-sequence: graph replay, the split solve and one kernel for filter and solve give the records of
    plain launches"""
    frames, imus, kw = tc.build(scenario)
    frames, imus = frames[0], imus[0]
    cam = cam_for(kw) if camera else None
    ref, _, order = run_switching(ofb200, kw, frames, imus, "plain", monkeypatch, cam)
    for mode in ("graph", "split", "nosplit"):
        got, graph_steps, _ = run_switching(ofb200, kw, frames, imus, mode, monkeypatch, cam)
        if mode == "graph":
            assert graph_steps >= 6, graph_steps
        for j in range(len(order)):
            assert same_record(got[j][0], ref[j][0]), (mode, j)


def test_tracker_zero_rate_is_no_prediction(ofb200, monkeypatch):
    frames, imus, kw = tc.build("node")
    frames, imus = frames[0], imus[0]
    for mode in ("graph", "split"):
        off, _, order = run_switching(ofb200, kw, frames, imus, mode, monkeypatch, switch={}, zero_w=True)
        on, _, _ = run_switching(ofb200, kw, frames, imus, mode, monkeypatch, switch={}, start=True, zero_w=True)
        for j in range(len(order)):
            assert same_record(off[j][0], on[j][0]), (mode, j)


def test_fleet_tracker_gyro(ofb200, ctx):
    frames, imus, kw = tc.build("module")
    fleet = ofb200.FleetTracker(2, tc.W, tc.H, ctx=ctx, gyro_prediction=True, **kw)
    ref = ofb200.StreamTracker(tc.W, tc.H, n_streams=2, ctx=ctx, gyro_prediction=True, **kw)
    try:
        for k in range(4):
            if k == 2:
                fleet.set_gyro_prediction(False); ref.set_gyro_prediction(False)
            samples = [gyro_imu(imus[s][k], k + s) for s in range(2)]
            fr = np.stack([frames[s][k] for s in range(2)])
            pri = np.stack([s["v_prior"] for s in samples])
            a = fleet.step(fr, imu_records(ofb200, samples), v_prior=pri)
            r = ref.step(fr, imu_records(ofb200, samples), v_prior=pri)
            assert all(same_record(a[s], r[s]) for s in range(2))
    finally:
        fleet.close()
        ref.close()
