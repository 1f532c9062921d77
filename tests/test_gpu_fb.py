"""GPU side of the forward-backward check (include/ofb200.h `ofb_pyrlk_fb`, `ofb_frame_pairs_fb`,
`ofb_tracker_set_fb_check`): the fused kernel against the composition of two LK calls and the NumPy fold, bit for bit;
against cv2 4.13 (golden file and live); the frame-pair routes, the camera and the solve; the tracker against
TrackerOracle with oracle/fb_oracle.FBEngine, graph replay, switching and the split solve; the outlier scene; and
the argument checks."""
import ctypes as C

import numpy as np
import pytest

import fb_cases
import synth
import tracker_cases as tc
from oracle import camera_oracle as co
from oracle import fb_oracle, tracker_oracle
from oracle import velocity_oracle as vo
from test_gpu_camera import cam_for, pair_setup, relerr
from test_gpu_tracker import imu_records, same_record
from test_host_fb import compare_to_golden, golden, golden_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ofb200():
    import ofb200
    return ofb200


def composition(ofb200, ctx, a, b, p0, T, **lk):
    """two calcOpticalFlowPyrLK calls on the GPU and the NumPy fold"""
    p1, st, err = ofb200.calcOpticalFlowPyrLK(a, b, p0, None, ctx=ctx, **lk)
    if len(p1) == 0:
        return p1, st, err, np.zeros(0, np.float32)
    p0r, st0, _ = ofb200.calcOpticalFlowPyrLK(b, a, p1, None, ctx=ctx, **lk)
    status, fb = fb_oracle.fb_check(p0, p1, st, p0r, st0, T)
    return p1, status.reshape(-1, 1), err, fb


def assert_fused_is_composition(ofb200, ctx, a, b, p0, T, **lk):
    got = ofb200.track_forward_backward(a, b, p0, threshold=T, ctx=ctx, **lk)
    ref = composition(ofb200, ctx, a, b, p0, T, **lk)
    for x, y, name in zip(got, ref, ("nextPts", "status", "err", "fbErr")):
        assert x.shape == y.shape and x.dtype == y.dtype and np.array_equal(x, y), name
    return got


@pytest.mark.parametrize("win", [(15, 15), (9, 13), (16, 15), (21, 21)])
@pytest.mark.parametrize("T", [0.25, 1.0, 5.0])
def test_fused_equals_composition(ofb200, ctx, win, T):
    a, b, _ = synth.make_pair(480, 640, 1, 3)
    p0 = ofb200.goodFeaturesToTrack(a, 400, 0.01, 8, blockSize=7, ctx=ctx)
    got = assert_fused_is_composition(ofb200, ctx, a, b, p0, T, winSize=win, maxLevel=3, criteria=(3, 20, 0.03))
    assert 0 < int(got[1].sum()) <= len(p0)


@pytest.mark.parametrize("win", [(15, 15), (21, 21)])
def test_fused_equals_composition_generic_kernel(ofb200, ctx, monkeypatch, win):
    monkeypatch.setenv("OFB_LK_GENERIC", "1")
    a, b = synth.affine_pair(241, 323, 4, shift=(3.2, 2.1), rot=-0.02)
    p0 = ofb200.goodFeaturesToTrack(a, 200, 0.01, 8, blockSize=7, ctx=ctx)
    for T in (0.25, 1.0):
        assert_fused_is_composition(ofb200, ctx, a, b, p0, T, winSize=win, maxLevel=3, criteria=(3, 20, 0.03))


def test_fused_border_points_and_empty_set(ofb200, ctx, monkeypatch):
    a, b, pts = fb_cases.border_scene()
    for generic in ("0", "1"):
        monkeypatch.setenv("OFB_LK_GENERIC", generic)
        got = assert_fused_is_composition(ofb200, ctx, a, b, pts, 1.0, winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
        assert np.isinf(got[3]).any() and (got[1] == 1).any()
    out = ofb200.track_forward_backward(a, b, np.zeros((0, 1, 2), np.float32), ctx=ctx)
    assert [x.shape for x in out] == [(0, 1, 2), (0, 1), (0, 1), (0,)]
    # T = 0: the plain forward call, no distance
    p1, st, err, fb = ofb200.track_forward_backward(a, b, pts, threshold=0, ctx=ctx, winSize=(15, 15))
    q1, qst, qerr = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, winSize=(15, 15), ctx=ctx)
    assert np.array_equal(p1, q1) and np.array_equal(st, qst) and np.array_equal(err, qerr) and np.isinf(fb).all()


def test_fused_vs_cv2_golden(ofb200, ctx):
    g = golden()
    covered, total = 0, 0
    for tag, a, b, p0, (win, ml, crit), T in golden_cases(g):
        p1, st, err, fb = ofb200.track_forward_backward(a, b, p0, threshold=T, winSize=win, maxLevel=ml, criteria=crit, ctx=ctx)
        covered += compare_to_golden(g, tag, st, fb)
        total += len(st)
    print("near-threshold exception covered %d of %d points" % (covered, total))
    assert covered <= 0.01 * total


@pytest.mark.parametrize("shape", [(720, 1280, 500), (1080, 1920, 1000)])
def test_fused_vs_cv2_live(ofb200, ctx, shape):
    cv2 = pytest.importorskip("cv2")
    h, w, K = shape
    a, b, _ = synth.make_pair(h, w, 2, 7)
    p0 = cv2.goodFeaturesToTrack(a, K, 0.01, 10, blockSize=7)
    lk = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
    p1, st, _ = cv2.calcOpticalFlowPyrLK(a, b, p0, None, **lk)
    p0r, st0, _ = cv2.calcOpticalFlowPyrLK(b, a, p1, None, **lk)
    gst, gfb = fb_oracle.fb_check(p0, p1, st, p0r, st0, 1.0)
    _, got, _, fb = ofb200.track_forward_backward(a, b, p0, threshold=1.0, ctx=ctx, **lk)
    near = np.abs(gfb.astype(np.float64) - 1.0) <= 0.05
    assert not ((got.ravel() != gst) & ~near).any()
    fin = np.isfinite(gfb) & np.isfinite(fb)
    assert np.abs(fb[fin] - gfb[fin]).max() <= 0.1
    print("%dx%d: near-threshold exception covered %d of %d" % (w, h, int(((got.ravel() != gst) & near).sum()), len(gst)))


# ---- frame pairs ------------------------------------------------------------------------------------------------
def test_frame_pairs_fb_counts_and_solve(ofb200, ctx):
    prev, nxt, imu, cfg, mo = pair_setup(ofb200)
    T = 0.25
    res, pp, pn, st = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx, fb_threshold=T)
    plain, _, pn0, st0 = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx)
    rejected = 0
    for i in range(len(prev)):
        n = int(res["n_features"][i])
        _, kst, _, _ = ofb200.track_forward_backward(prev[i], nxt[i], pp[i, :n], threshold=T, winSize=(15, 15), maxLevel=3,
                                                    criteria=(3, 20, 0.03), ctx=ctx)
        assert np.array_equal(st[i, :n], kst.ravel()) and np.array_equal(pn[i, :n], pn0[i, :n])
        ok = st[i, :n] == 1
        assert int(res["n_tracked"][i]) == int(ok.sum()) > 20
        rejected += int(plain["n_tracked"][i]) - int(ok.sum())
        x = (pn[i, :n][ok].astype(np.float64) - [cfg.cx, cfg.cy]) * cfg.pos_scale
        u = (pn[i, :n][ok] - pp[i, :n][ok]).astype(np.float64) * cfg.flow_scale
        v = vo.solve_lgs(x, u, imu["d"][i], imu["n"][i], imu["w"][i], variant="node")[0]
        assert relerr(res["v"][i], v) <= 1e-4
    assert rejected > 0


def test_frame_pairs_fb_routes_identical(ofb200, ctx):
    """resident single pass, resident twin chunks, host-frame pipeline, sequence layout: one result"""
    import torch
    h, w, n = 240, 320, 12
    frames = np.stack([synth.make_pair(h, w, 3, k, max_disp=5.0)[0 if k == 0 else 1] for k in range(n + 1)])
    imu = np.zeros(n, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"][:, 2], imu["w"][:, 0] = 2.0, 1.0, 0.01
    cfg = ofb200.make_pair_cfg(w, h, 150, 0.01, 8, 7, (15, 15), 3, (3, 20, 0.03), variant="node", pos_scale=1 / 256.0,
                               flow_scale=1 / 8.0)
    T = 0.5
    host = ofb200.frame_pairs(frames[:-1].copy(), frames[1:].copy(), imu, cfg, want_tracks=True, ctx=ctx, fb_threshold=T)
    seq = ofb200.frame_sequence(frames, imu, cfg, want_tracks=True, ctx=ctx, fb_threshold=T)
    d = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    twin = ofb200.frame_pairs(d[:-1].contiguous(), d[1:].contiguous(), imu, cfg, want_tracks=True, ctx=ctx, fb_threshold=T)
    ofb200._lib.check(ctx.lib.ofb_ctx_set_profile(ctx.h, 1))          # stage timing: the resident single pass
    try:
        single = ofb200.frame_pairs(d[:-1].contiguous(), d[1:].contiguous(), imu, cfg, want_tracks=True, ctx=ctx, fb_threshold=T)
    finally:
        ofb200._lib.check(ctx.lib.ofb_ctx_set_profile(ctx.h, 0))
    for other in (seq, twin, single):
        assert all(same_record(host[0][i], other[0][i]) for i in range(n))
        for x, y in zip(host[1:], other[1:]):
            assert np.array_equal(x, y)
    plain = ofb200.frame_pairs(frames[:-1], frames[1:], imu, cfg, ctx=ctx)
    assert (host[0]["n_tracked"] <= plain["n_tracked"]).all()


def test_frame_pairs_fb_with_camera(ofb200, ctx):
    prev, nxt, imu, cfg, mo = pair_setup(ofb200)
    K = np.array([[mo["f"] * 1.01, 0.0, mo["cx"] + 1.5], [0.0, mo["f"], mo["cy"] - 0.5], [0.0, 0.0, 1.0]])
    cam = (K, [-0.2, 0.05, 0.001, -0.002], 1.0 / mo["dt"], 20)
    T = 0.25
    res, pp, pn, st = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx, camera=cam, fb_threshold=T)
    _, pp0, pn0, st0 = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx, fb_threshold=T)
    assert np.array_equal(pp, pp0) and np.array_equal(pn, pn0) and np.array_equal(st, st0)
    for i in range(len(prev)):
        n = int(res["n_features"][i])
        ok = st[i, :n] == 1
        x, u = co.calibrate(pn[i, :n][ok], pp[i, :n][ok], cam)
        v = vo.solve_lgs(x, u, imu["d"][i], imu["n"][i], imu["w"][i], variant="node")[0]
        assert int(res["n_tracked"][i]) == int(ok.sum()) and relerr(res["v"][i], v) <= 1e-4


# ---- tracker ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [21, 22, 23, 24])
def test_tracker_fb_vs_oracle(ofb200, ctx, seed):
    """random_case sequences, teacher-forced on the oracle's point sets: the check keeps the same points as
    TrackerOracle(engine=FBEngine(...)), and every velocity is the fp64 solve on the GPU's kept tracks."""
    frames, imus, kw = tc.random_case(seed)
    T = 0.3
    okw = {k: v for k, v in kw.items() if k != "bgr"}
    orc = tracker_oracle.TrackerOracle(tc.W, tc.H, engine=fb_oracle.FBEngine(tracker_oracle.Engine(), T), **okw)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, fb_threshold=T, **kw)
    solved = 0
    try:
        for k in range(len(frames[0])):
            im = imus[0][k]
            trk.set_points(orc.pts)
            o = orc.step(frames[0][k], im["d"], im["n"], im["w"], im["t"], im["v_prior"])
            res, kp, kn = trk.step(frames[0][k], imu_records(ofb200, [im]), v_prior=im["v_prior"][None], want_kept=True)
            for key in ("n_prev", "n_tracked", "n_kept"):
                assert int(res[key][0]) == int(o[key]), (seed, k, key)
            if res["flags"][0] & 1:
                solved += 1
                x = (kn[0].astype(np.float64) - vo.pix_trans((tc.W, tc.H))) * kw["scaling"]
                u = (kn[0] - kp[0]).astype(np.float64) * kw["scaling"]
                v = vo.solve_lgs(x, u, im["d"], im["n"], im["w"], None if kw["variant"] == "node" else im["t"], kw["variant"])[0]
                assert relerr(res["v"][0], v) <= 1e-9, (seed, k)
                assert relerr(res["v"][0], o["v"]) <= 2e-3, (seed, k)
    finally:
        trk.close()
    assert solved >= 3


@pytest.mark.parametrize("seed", [22, 24])
def test_tracker_fb_with_camera_vs_oracle(ofb200, ctx, seed):
    """the check and a calibrated camera together, teacher-forced on CameraTrackerOracle(engine=FBEngine(...)): the same
    points pass the check and the gate, and every velocity is the fp64 solve on the calibrated kept tracks"""
    frames, imus, kw = tc.random_case(seed)
    T = 0.3
    cam = cam_for(kw)
    okw = {k: v for k, v in kw.items() if k != "bgr"}
    orc = co.CameraTrackerOracle(tc.W, tc.H, cam, engine=fb_oracle.FBEngine(tracker_oracle.Engine(), T), **okw)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, camera=cam, fb_threshold=T, **kw)
    solved = 0
    try:
        for k in range(len(frames[0])):
            im = imus[0][k]
            trk.set_points(orc.pts)
            o = orc.step(frames[0][k], im["d"], im["n"], im["w"], im["t"], im["v_prior"])
            res, kp, kn = trk.step(frames[0][k], imu_records(ofb200, [im]), v_prior=im["v_prior"][None], want_kept=True)
            for key in ("n_prev", "n_tracked", "n_kept"):
                assert int(res[key][0]) == int(o[key]), (seed, k, key)
            if res["flags"][0] & 1:
                solved += 1
                x, u = co.calibrate(kn[0], kp[0], cam)
                v = vo.solve_lgs(x, u, im["d"], im["n"], im["w"], None if kw["variant"] == "node" else im["t"], kw["variant"])[0]
                assert relerr(res["v"][0], v) <= 1e-9, (seed, k)
                assert relerr(res["v"][0], o["v"]) <= 2e-3, (seed, k)
    finally:
        trk.close()
    assert solved >= 3


SWITCH = {3: 0.0, 6: 0.4, 10: None}          # step -> threshold set before it (the run starts with 0.25)


def run_switching(ofb200, kw, frames, imus, mode, monkeypatch, camera=None, switch=SWITCH, start=0.25):
    """as tests/test_gpu_camera.run_switching, switching the check instead of the camera"""
    import torch
    monkeypatch.setenv("OFB_TRACKER_GRAPH", "0" if mode == "plain" else "1")
    monkeypatch.setenv("OFB_TRACKER_SPLIT_SOLVE", "0" if mode == "nosplit" else "1")
    ctx = ofb200.Context(0)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, camera=camera, fb_threshold=start, **kw)
    order = list(range(len(frames))) + list(range(len(frames) - 2, -1, -1))
    out = []
    dev = mode in ("split", "nosplit")
    d_res = torch.zeros(C.sizeof(ofb200._lib.TrackResult), dtype=torch.uint8, device="cuda") if dev else None
    try:
        for j, k in enumerate(order):
            if j in switch:
                trk.set_fb_threshold(switch[j])
            im = imu_records(ofb200, [imus[k]])
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
def test_tracker_fb_switch_identical_in_every_mode(ofb200, monkeypatch, scenario, camera):
    """on / off / on / off mid-sequence: graph replay, the split solve and one kernel for filter and solve give the
    records of plain launches; with the check, with a camera and with the masked top-up ("node")"""
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


def test_tracker_fb_switch_matches_oracle(ofb200, ctx):
    """the same switches on the oracle (FBEngine with the threshold in force): the same counts step by step"""
    frames, imus, kw = tc.build("exp")
    frames, imus = frames[0], imus[0]
    okw = {k: v for k, v in kw.items() if k != "bgr"}
    eng = fb_oracle.FBEngine(tracker_oracle.Engine(), 0.25)
    orc = tracker_oracle.TrackerOracle(tc.W, tc.H, engine=eng, **okw)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, fb_threshold=0.25, **kw)
    try:
        for k in range(len(frames)):
            if k in (2, 4, 6):
                T = {2: 0.0, 4: 0.4, 6: None}[k]
                trk.set_fb_threshold(T); eng.T = T or 0.0
            trk.set_points(orc.pts)
            o = orc.step(frames[k], imus[k]["d"], imus[k]["n"], imus[k]["w"], imus[k]["t"])
            r = trk.step(frames[k], imu_records(ofb200, [imus[k]]))
            for key in ("n_prev", "n_tracked", "n_kept"):
                assert int(r[key][0]) == int(o[key]), (k, key)
    finally:
        trk.close()


def test_tracker_threshold_zero_is_no_check(ofb200, monkeypatch):
    frames, imus, kw = tc.build("node")
    frames, imus = frames[0], imus[0]
    for mode in ("graph", "split"):
        never, _, order = run_switching(ofb200, kw, frames, imus, mode, monkeypatch, switch={}, start=None)
        zero, _, _ = run_switching(ofb200, kw, frames, imus, mode, monkeypatch, switch={1: 0.0, 5: 0.0}, start=0.0)
        for j in range(len(order)):
            assert same_record(never[j][0], zero[j][0]), (mode, j)


def test_fleet_tracker_fb(ofb200, ctx):
    frames, imus, kw = tc.build("module")
    fleet = ofb200.FleetTracker(2, tc.W, tc.H, ctx=ctx, fb_threshold=0.3, **kw)
    ref = ofb200.StreamTracker(tc.W, tc.H, n_streams=2, ctx=ctx, fb_threshold=0.3, **kw)
    try:
        for k in range(4):
            if k == 2:
                fleet.set_fb_threshold(None); ref.set_fb_threshold(0)
            samples = [imus[s][k] for s in range(2)]
            fr = np.stack([frames[s][k] for s in range(2)])
            pri = np.stack([s["v_prior"] for s in samples])
            a = fleet.step(fr, imu_records(ofb200, samples), v_prior=pri)
            r = ref.step(fr, imu_records(ofb200, samples), v_prior=pri)
            assert all(same_record(a[s], r[s]) for s in range(2))
    finally:
        fleet.close()
        ref.close()


# ---- what the check is for --------------------------------------------------------------------------------------
def test_outlier_scene(ofb200, ctx):
    rej, far_kept, e_plain, e_fb = [], [], [], []
    win, ml, crit = fb_cases.OCCLUDER_LK
    for k in fb_cases.OCCLUDER_SEEDS:
        a, b, mo, patch = fb_cases.occluder_scene(k)
        p0 = ofb200.goodFeaturesToTrack(a, 500, 0.01, 10, blockSize=7, ctx=ctx)
        p1, good, _, _ = ofb200.track_forward_backward(a, b, p0, threshold=fb_cases.OCCLUDER_T, winSize=win, maxLevel=ml,
                                                       criteria=crit, ctx=ctx)
        _, st, _ = ofb200.calcOpticalFlowPyrLK(a, b, p0, None, winSize=win, maxLevel=ml, criteria=crit, ctx=ctx)
        st, good = st.ravel() == 1, good.ravel() == 1
        inside, far = fb_cases.patch_masks(p0, patch)
        rej.append(1 - (inside & good).sum() / (inside & st).sum())
        far_kept.append((far & good).sum() / (far & st).sum())
        e_plain.append(fb_cases.velocity_error(p0, p1, st, mo))
        e_fb.append(fb_cases.velocity_error(p0, p1, good, mo))
    print("rejected inside", np.round(rej, 3), "kept far", np.round(far_kept, 3), "error", np.round(e_plain, 3), np.round(e_fb, 3))
    assert min(rej) >= 0.70 and min(far_kept) >= 0.97
    assert np.mean(e_fb) < 0.5 * np.mean(e_plain)


# ---- errors -----------------------------------------------------------------------------------------------------
def test_invalid_thresholds_rejected(ofb200, ctx):
    lib = ctx.lib
    prev, nxt, imu, cfg, mo = pair_setup(ofb200, n=1)
    res = np.zeros(1, ofb200._lib.RESULT_DTYPE)
    pyr = ofb200.Pyramid(prev[0], 3, ctx)
    pts = np.array([[100.0, 100.0]], np.float32)
    out, st, er, fb = np.zeros((1, 2), np.float32), np.zeros(1, np.uint8), np.zeros(1, np.float32), np.zeros(1, np.float32)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx)
    P = ofb200._lib.ptr
    try:
        for bad in (-1.0, -1e-300, float("nan"), float("-inf")):
            assert lib.ofb_pyrlk_fb(ctx.h, pyr.h, 0, pyr.h, 0, P(pts), 1, 15, 15, 3, 20, 0.03, 1e-4, bad, P(out), P(st), P(er),
                                    P(fb)) == ofb200._lib.OFB_E_INVALID
            assert lib.ofb_frame_pairs_fb(ctx.h, C.byref(cfg), None, bad, 1, P(prev), P(nxt), cfg.width, cfg.width * cfg.height,
                                          P(imu), None, None, P(res), None, None, None) == ofb200._lib.OFB_E_INVALID
            assert lib.ofb_tracker_set_fb_check(trk.h, bad) == ofb200._lib.OFB_E_INVALID
        assert lib.ofb_tracker_set_fb_check(None, 1.0) == ofb200._lib.OFB_E_INVALID
        # still usable
        assert lib.ofb_pyrlk_fb(ctx.h, pyr.h, 0, pyr.h, 0, P(pts), 1, 15, 15, 3, 20, 0.03, 1e-4, float("inf"), P(out), P(st),
                                P(er), P(fb)) == ofb200._lib.OFB_OK
        assert st[0] == 1 and fb[0] == 0.0
        trk.set_fb_threshold(1.0)
        trk.set_fb_threshold(None)
    finally:
        trk.close()
        pyr.close()
