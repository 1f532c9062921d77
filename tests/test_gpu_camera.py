"""GPU side of the calibrated camera (include/ofb200.h `ofb_camera`, csrc/camera.cuh): the standalone undistortion
against cv2 4.13 (golden file and live) and oracle/camera_oracle.py, the frame-pair and tracker velocity paths against
the fp64 NumPy solve on the oracle's calibrated x, u of the GPU's own tracks, camera switches in every tracker mode,
the velocity of a pair rendered through a wide-angle lens, and the argument checks."""
import ctypes as C

import numpy as np
import pytest

import synth
import tracker_cases as tc
from oracle import camera_oracle as co
from oracle import velocity_oracle as vo
from test_gpu_tracker import imu_records, same_record
from test_host_camera import golden_cases

pytestmark = pytest.mark.gpu

K_WIDE = np.array([[512.0, 0.0, 320.0], [0.0, 512.0, 240.0], [0.0, 0.0, 1.0]])
D_WIDE = np.array([-0.3, 0.1, 0.0, 0.0, -0.02])


@pytest.fixture(scope="module")
def ofb200():
    import ofb200
    return ofb200


def relerr(a, b):
    return np.abs(np.asarray(a) - b).max() / max(np.abs(b).max(), 1e-300)


# ---- standalone undistortion ------------------------------------------------------------------------------------
def test_undistort_points_equals_cv2_golden(ofb200, ctx):
    _, cases = golden_cases()
    for c in cases:
        if c["iterations"] == 5:
            got = ofb200.undistortPoints(c["src"].reshape(-1, 1, 2), c["K"], c["D"], R=c["R"], P=c["P"], ctx=ctx)
        else:
            got = ofb200.undistortPointsIter(c["src"], c["K"], c["D"], c["R"], c["P"], (ofb200.TERM_CRITERIA_COUNT, c["iterations"], 0),
                                             ctx=ctx)
        assert got.shape == (len(c["src"]), 1, 2) and got.dtype == c["out"].dtype, c["tag"]
        got = got.reshape(-1, 2)
        if got.dtype == np.float32:
            ulp = np.spacing(np.abs(c["out"]).astype(np.float32))
            assert np.all(np.abs(got - c["out"]) <= ulp), c["tag"]
        else:
            assert np.abs(got - c["out"]).max() <= 1e-14, c["tag"]
            ref = co.undistort(c["src"], c["K"], c["D"], c["iterations"], co.rectification(c["R"], c["P"]))
            assert np.abs(got - ref).max() <= 1e-14, c["tag"]


def test_undistort_points_large_and_live_cv2(ofb200, ctx):
    rng = np.random.default_rng(9)
    src = np.stack([rng.uniform(-100, 1380, 100000), rng.uniform(-100, 820, 100000)], axis=1)
    K = np.array([[900.0, 0.0, 640.0], [0.0, 900.0, 360.0], [0.0, 0.0, 1.0]])
    D = np.array([-0.3, 0.12, 0.001, -0.0005, -0.02, 0.05, 0.01, 0.002])
    P = np.array([[800.0, 0.0, 640.0, 5.0], [0.0, 800.0, 360.0, 0.0], [0.0, 0.0, 1.0, 0.0]])
    R = np.array([[1.0, 0.0, 0.0], [0.0, np.cos(0.02), -np.sin(0.02)], [0.0, np.sin(0.02), np.cos(0.02)]])
    for d in (None, D[:4], D[:5], D):
        got = ofb200.undistortPointsIter(src, K, d, R, P, (ofb200.TERM_CRITERIA_COUNT, 20, 0), ctx=ctx).reshape(-1, 2)
        assert np.abs(got - co.undistort(src, K, d, 20, co.rectification(R, P))).max() <= 1e-14 * 1000
        got = ofb200.undistortPoints(src, K, d, ctx=ctx).reshape(-1, 2)
        assert np.abs(got - co.undistort(src, K, d, 5)).max() <= 1e-14
    try:
        import cv2
    except ImportError:
        return
    for d in (None, D[:5], D):
        ref = cv2.undistortPoints(src.reshape(-1, 1, 2), K, d, R=R, P=P)
        got = ofb200.undistortPoints(src.reshape(-1, 1, 2), K, d, R=R, P=P, ctx=ctx)
        assert np.abs(got - ref).max() <= 1e-14 * 1000
        s32 = src.astype(np.float32)
        ref, got = cv2.undistortPoints(s32, K, d), ofb200.undistortPoints(s32, K, d, ctx=ctx)
        assert got.dtype == np.float32 and np.all(np.abs(got - ref) <= np.spacing(np.abs(ref)))


def test_undistort_points_device_arrays_and_empty(ofb200, ctx):
    import torch
    src = np.array([[10.0, 20.0], [640.0, 360.0], [1270.0, 700.0]])
    K = np.array([[900.0, 0.0, 640.0], [0.0, 900.0, 360.0], [0.0, 0.0, 1.0]])
    cam = ofb200.make_camera(K, D_WIDE, 1.0, 5)
    d_in = torch.from_numpy(src).cuda()
    d_out = torch.empty_like(d_in)
    ofb200._lib.check(ctx.lib.ofb_undistort_points(ctx.h, C.byref(cam), ofb200._lib.ptr(d_in), 3, None, ofb200._lib.ptr(d_out)))
    ctx.sync()
    assert np.abs(d_out.cpu().numpy() - co.undistort(src, K, D_WIDE, 5)).max() <= 1e-14
    ofb200._lib.check(ctx.lib.ofb_undistort_points(ctx.h, C.byref(cam), None, 0, None, None))
    assert ofb200.undistortPoints(np.zeros((0, 2)), K, D_WIDE, ctx=ctx).shape == (0, 1, 2)


# ---- frame pairs ------------------------------------------------------------------------------------------------
def pair_setup(ofb200, n=3, h=240, w=320):
    prev, nxt, imu = [], [], np.zeros(n, ofb200._lib.IMU_DTYPE)
    mos = []
    for i in range(n):
        a, b, mo = synth.make_pair(h, w, i, 10 + i, max_disp=6.0)
        prev.append(a); nxt.append(b); mos.append(mo)
        imu["d"][i], imu["n"][i], imu["w"][i] = mo["d"], mo["n"], mo["w"]
    mo = mos[0]
    cfg = ofb200.make_pair_cfg(w, h, 150, 0.01, 8, 7, (15, 15), 3, (3, 20, 0.03), variant="node",
                               principal=(mo["cx"], mo["cy"]), pos_scale=1.0 / mo["f"], flow_scale=1.0 / (mo["f"] * mo["dt"]))
    return np.stack(prev), np.stack(nxt), imu, cfg, mo


@pytest.mark.parametrize("D", [None, [-0.2, 0.05, 0.001, -0.002], list(D_WIDE), [-0.3, 0.1, 0.001, 0.0, -0.02, 0.04, 0.01, 0.0]])
def test_frame_pairs_camera_equals_fp64_solve(ofb200, ctx, D):
    prev, nxt, imu, cfg, mo = pair_setup(ofb200)
    K = np.array([[mo["f"] * 1.01, 0.0, mo["cx"] + 1.5], [0.0, mo["f"], mo["cy"] - 0.5], [0.0, 0.0, 1.0]])
    cam = (K, D, 1.0 / mo["dt"], 20)
    res, pp, pn, st = ofb200.frame_pairs(prev, nxt, imu, cfg, want_tracks=True, ctx=ctx, camera=cam)
    seq = ofb200.frame_sequence(np.concatenate([prev[:1], nxt[:1]]), imu[:1], cfg, ctx=ctx, camera=cam)
    assert same_record(seq[0], res[0])
    for i in range(len(prev)):
        n = int(res["n_features"][i])
        ok = st[i, :n] == 1
        x, u = co.calibrate(pn[i, :n][ok], pp[i, :n][ok], cam)
        v, r, rank, s = vo.solve_lgs(x, u, imu["d"][i], imu["n"][i], imu["w"][i], variant="node")
        assert int(res["n_tracked"][i]) == int(ok.sum()) > 20
        assert relerr(res["v"][i], v) <= 1e-9, (i, res["v"][i], v)
        assert int(res["rank"][i]) == int(rank) and np.allclose(res["s"][i], s, rtol=1e-7)


def test_frame_pairs_camera_without_distortion_is_the_pinhole(ofb200, ctx):
    """n_dist = 0, fx = fy = 1/pos_scale, rate = flow_scale/pos_scale. The scales are powers of two (f = 256 px, rate 32)
    so that 1/fx and rate carry no rounding of their own: the camera path's x and u are then the pinhole's exactly. The
    pinhole kernel, however, lets nvcc fuse `ux = dx * flow_scale` into the next addition (one FMA), so the solves see
    inputs one rounding apart, and the least well-conditioned pair of this set amplifies that to 1.5e-9 (measured on a
    B200): the bar is 1e-8."""
    prev, nxt, imu, cfg, mo = pair_setup(ofb200, n=10)          # > 8 host pairs: the pipelined sub-batch path too
    assert mo["f"] == 256.0
    cfg.pos_scale, cfg.flow_scale = 1.0 / 256.0, 32.0 / 256.0
    K = np.array([[1.0 / cfg.pos_scale, 0.0, cfg.cx], [0.0, 1.0 / cfg.pos_scale, cfg.cy], [0.0, 0.0, 1.0]])
    ref = ofb200.frame_pairs(prev, nxt, imu, cfg, ctx=ctx)
    got = ofb200.frame_pairs(prev, nxt, imu, cfg, ctx=ctx, camera=(K, None, cfg.flow_scale / cfg.pos_scale))
    for i in range(len(prev)):
        assert got["n_tracked"][i] == ref["n_tracked"][i]
        assert relerr(got["v"][i], ref["v"][i]) <= 1e-8


# ---- tracker ----------------------------------------------------------------------------------------------------
def cam_for(kw, D=D_WIDE):
    f = 1.0 / kw["scaling"]
    K = np.array([[f, 0.0, tc.W / 2 + 0.5], [0.0, f * 0.995, tc.H / 2 - 1.0], [0.0, 0.0, 1.0]])
    return (K, np.asarray(D), 30.0, 20)


@pytest.mark.parametrize("seed", [22, 24, 26])
def test_tracker_camera_vs_oracle(ofb200, ctx, seed):
    """random_case sequences with the r_tilde gate, teacher-forced on the oracle's point sets: the gate keeps the same
    points, and every velocity equals the fp64 solve on the oracle's calibrated x, u of the GPU's kept tracks."""
    frames, imus, kw = tc.random_case(seed)
    assert kw["gate"] is not None
    cam = cam_for(kw)
    okw = {k: v for k, v in kw.items() if k != "bgr"}
    orc = co.CameraTrackerOracle(tc.W, tc.H, cam, **okw)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, camera=cam, **kw)
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


def test_tracker_module_variant_with_camera(ofb200, ctx):
    """variant="module": the per-point distances (4-argument r_tilde from the prior) come from calibrated x, u (the gate
    keeps every point here, as in tests/test_gpu_round2.py; the gated random cases above cover the gate)."""
    h, w = 240, 320
    a, b, mo = synth.make_pair(h, w, 3, 5, max_disp=4.0)
    imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
    K = np.array([[mo["f"], 0.0, mo["cx"]], [0.0, mo["f"], mo["cy"]], [0.0, 0.0, 1.0]])
    cam = (K, [-0.1, 0.02, 0.0, 0.0, 0.0], 1.0 / mo["dt"], 20)
    v_prior = np.asarray(mo["v"], dtype=np.float64) * 1.1 + 0.01
    trk = ofb200.StreamTracker(w, h, max_features=60, min_features=10, topup="module", variant="module", gate=("ge", -2.0),
                               min_solve=4, camera=cam, ctx=ctx)
    try:
        trk.step(a, imu)
        r, kp, kn = trk.step(b, imu, v_prior=v_prior[None], want_kept=True)
    finally:
        trk.close()
    assert r["flags"][0] & 1 and r["n_kept"][0] >= 20
    x, u = co.calibrate(kn[0], kp[0], cam)
    xh = np.hstack([x, np.ones((len(x), 1))]); uh = np.hstack([u, np.zeros((len(u), 1))])
    _, dist = vo.r_tilde(xh, uh, mo["n"], v_prior)
    v_ref, _, rank, _ = vo.solve_lgs_module(xh, uh, mo["n"], dist)
    assert rank == 3 and relerr(r["v"][0], v_ref) <= 1e-9


SWITCH = {5: "B", 9: None, 12: "A"}          # step -> camera set before it


def run_switching(ofb200, kw, frames, imus, mode, monkeypatch):
    """One stream through the sequence forwards and backwards, switching cameras at the SWITCH steps. mode: "graph"
    (host frames: graph replay from the fourth step), "plain" (OFB_TRACKER_GRAPH=0), "kept" (host frames with the kept
    tracks read back), "split" / "nosplit" (device frames, IMU samples and result records: split solve default on,
    OFB_TRACKER_SPLIT_SOLVE=0)."""
    import torch
    monkeypatch.setenv("OFB_TRACKER_GRAPH", "0" if mode == "plain" else "1")
    monkeypatch.setenv("OFB_TRACKER_SPLIT_SOLVE", "0" if mode == "nosplit" else "1")
    cams = {"A": cam_for(kw), "B": cam_for(kw, [0.05, -0.01, 0.002, 0.001, 0.0, 0.02, 0.0, 0.001])}
    ctx = ofb200.Context(0)                 # a context that owns its stream: the tracker may use its side streams
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, camera=cams["A"], **kw)
    order = list(range(len(frames))) + list(range(len(frames) - 2, -1, -1))
    out, kept = [], []
    dev = mode in ("split", "nosplit")
    d_res = torch.zeros(C.sizeof(ofb200._lib.TrackResult), dtype=torch.uint8, device="cuda") if dev else None
    try:
        for j, k in enumerate(order):
            if j in SWITCH:
                trk.set_camera(None if SWITCH[j] is None else cams[SWITCH[j]])
            im = imu_records(ofb200, [imus[k]])
            if dev:
                fr = torch.from_numpy(frames[k]).cuda()
                d_imu = torch.from_numpy(im.view(np.uint8).copy()).cuda()
                ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, ofb200._lib.ptr(fr), tc.W, tc.W * tc.H, ofb200._lib.ptr(d_imu),
                                                           None, ofb200._lib.ptr(d_res), None, None, None, None))
                ctx.sync()
                out.append(d_res.cpu().numpy().view(ofb200._lib.TRACK_RESULT_DTYPE).copy())
            elif mode == "kept":
                r, kp, kn = trk.step(frames[k], im, want_kept=True)
                out.append(r.copy()); kept.append((kp[0], kn[0]))
            else:
                out.append(trk.step(frames[k], im).copy())
        graph_steps = trk.graph_steps()
    finally:
        trk.close()
        ctx.close()
    return out, kept, graph_steps, cams, order


def test_camera_switch_identical_in_every_mode(ofb200, monkeypatch):
    frames, imus, kw = tc.build("exp")
    frames, imus = frames[0], imus[0]
    kw = dict(kw, gate=("le", 0.0), v_init=[0.1, -0.05, 0.0])
    ref, kept, _, cams, order = run_switching(ofb200, kw, frames, imus, "kept", monkeypatch)
    # the kept run is the reference: its velocities are the fp64 solve under the camera in force at each step
    cur, solved = cams["A"], 0
    for j, k in enumerate(order):
        if j in SWITCH:
            cur = None if SWITCH[j] is None else cams[SWITCH[j]]
        if not ref[j]["flags"][0] & 1:
            continue
        solved += 1
        kp, kn = kept[j]
        if cur is None:
            x = (kn.astype(np.float64) - vo.pix_trans((tc.W, tc.H))) * kw["scaling"]
            u = (kn - kp).astype(np.float64) * kw["scaling"]
        else:
            x, u = co.calibrate(kn, kp, cur)
        im = imus[k]
        v = vo.solve_lgs(x, u, im["d"], im["n"], im["w"], im["t"], kw["variant"])[0]
        assert relerr(ref[j]["v"][0], v) <= 1e-9, j
    assert solved >= 8
    for mode in ("graph", "plain", "split", "nosplit"):
        got, _, graph_steps, _, _ = run_switching(ofb200, kw, frames, imus, mode, monkeypatch)
        if mode == "graph":
            assert graph_steps >= len(order) - 3 - 1, graph_steps
        for j in range(len(order)):
            assert same_record(got[j][0], ref[j][0]), (mode, j)


# ---- what the feature is for ------------------------------------------------------------------------------------
def render_lens_pair(w, h, K, D, mo, seed=7):
    """Two frames of a textured plane seen through OpenCV's lens model: every distorted pixel is sent to its
    undistorted normalised coordinates by the inverse lens model iterated to convergence (200 fixed-point steps; the
    round trip through the forward model is exact to 1e-9 px here), the second frame moved by the flow model of
    simulation.py:7-12 (backward warp, fixed point)."""
    f = K[0, 0]
    pad = w
    big = synth.texture(h + 2 * pad, w + 2 * pad, seed).astype(np.float64)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    und = co.undistort(np.stack([xx.ravel(), yy.ravel()], 1), K, D, iterations=200)
    x, y = und[:, 0], und[:, 1]
    a = synth.bilinear_sample(big, x * f + K[0, 2] + pad, y * f + K[1, 2] + pad).reshape(h, w)
    sx, sy = x.copy(), y.copy()
    for _ in range(6):
        ux, uy = synth.flow_model(sx, sy, mo["v"], mo["w"], mo["d"], mo["n"])
        sx, sy = x - ux * mo["dt"], y - uy * mo["dt"]
    b = synth.bilinear_sample(big, sx * f + K[0, 2] + pad, sy * f + K[1, 2] + pad).reshape(h, w)
    q = lambda im: np.clip(np.round(im), 0, 255).astype(np.uint8)
    return q(a), q(b)


def test_wide_angle_lens_velocity(ofb200, ctx):
    """A 640x480 frame pair through a k1 = -0.3 lens (fx = 512 px) with known (v, w, d, n): the calibrated path recovers
    v within 4 % (relative norm), the pinhole path on the same frames misses it by more than three times that."""
    w, h = 640, 480
    n = np.array([0.03, -0.02, 1.0])
    mo = dict(v=np.array([0.6, -0.35, 0.15]), w=np.array([0.02, -0.015, 0.03]), d=2.0, n=n / np.linalg.norm(n), dt=1 / 30.0)
    a, b = render_lens_pair(w, h, K_WIDE, D_WIDE, mo)
    roundtrip = co.undistort(np.array([[0.0, 0.0], [639.0, 479.0]]), K_WIDE, D_WIDE, 200)
    r2 = (roundtrip ** 2).sum(1)
    assert np.abs(roundtrip[:, 0] * (1 + (D_WIDE[0] + (D_WIDE[1] + D_WIDE[4] * r2) * r2) * r2) * 512 + 320 - [0, 639]).max() < 1e-9
    imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
    f = K_WIDE[0, 0]
    cfg = ofb200.make_pair_cfg(w, h, 300, 0.01, 10, 7, (15, 15), 3, (3, 20, 0.03), variant="node", principal=(w / 2, h / 2),
                               pos_scale=1.0 / f, flow_scale=1.0 / (f * mo["dt"]))
    pin = ofb200.frame_pairs(a[None], b[None], imu, cfg, ctx=ctx)
    cal = ofb200.frame_pairs(a[None], b[None], imu, cfg, ctx=ctx, camera=(K_WIDE, D_WIDE, 1.0 / mo["dt"]))
    err = lambda r: np.linalg.norm(r["v"][0] - mo["v"]) / np.linalg.norm(mo["v"])
    e_pin, e_cal = err(pin), err(cal)
    print("wide-angle lens: relative velocity error pinhole %.4f, calibrated %.4f (v = %s, truth %s)"
          % (e_pin, e_cal, np.round(cal["v"][0], 4), mo["v"]))
    assert int(cal["n_tracked"][0]) > 200
    assert e_cal <= 0.04 and e_pin >= 3 * e_cal


# ---- errors -----------------------------------------------------------------------------------------------------
def bad_cameras(ofb200):
    good = ofb200.make_camera(K_WIDE, D_WIDE, 30.0, 20)
    out = []
    for field, value in (("fx", 0.0), ("fy", -1.0), ("cx", float("nan")), ("n_dist", 3), ("n_dist", 12), ("iterations", 0),
                         ("iterations", 1001), ("rate", 0.0), ("rate", float("inf"))):
        c = ofb200._lib.Camera.from_buffer_copy(good)
        setattr(c, field, value)
        out.append(c)
    c = ofb200._lib.Camera.from_buffer_copy(good)
    c.dist[1] = float("nan")
    out.append(c)
    return out


def test_invalid_cameras_rejected_and_context_stays_usable(ofb200, ctx):
    lib = ctx.lib
    pts = np.zeros((4, 2))
    out = np.zeros((4, 2))
    prev, nxt, imu, cfg, mo = pair_setup(ofb200, n=1)
    res = np.zeros(1, ofb200._lib.RESULT_DTYPE)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx)
    try:
        for cam in bad_cameras(ofb200):
            assert lib.ofb_undistort_points(ctx.h, C.byref(cam), ofb200._lib.ptr(pts), 4, None, ofb200._lib.ptr(out)) == ofb200._lib.OFB_E_INVALID
            assert lib.ofb_last_error()
            rc = lib.ofb_frame_pairs_cam(ctx.h, C.byref(cfg), C.byref(cam), 1, ofb200._lib.ptr(prev), ofb200._lib.ptr(nxt), cfg.width,
                                         cfg.width * cfg.height, ofb200._lib.ptr(imu), None, None, ofb200._lib.ptr(res), None, None, None)
            assert rc == ofb200._lib.OFB_E_INVALID
            assert lib.ofb_tracker_set_camera(trk.h, C.byref(cam)) == ofb200._lib.OFB_E_INVALID
        bad_h = np.eye(3).ravel().copy(); bad_h[4] = np.nan
        good = ofb200.make_camera(K_WIDE, D_WIDE, 30.0, 5)
        assert lib.ofb_undistort_points(ctx.h, C.byref(good), ofb200._lib.ptr(pts), 4, ofb200._lib.ptr(bad_h), ofb200._lib.ptr(out)) == ofb200._lib.OFB_E_INVALID
        assert lib.ofb_undistort_points(ctx.h, C.byref(good), ofb200._lib.ptr(pts), -1, None, ofb200._lib.ptr(out)) == ofb200._lib.OFB_E_INVALID
        assert lib.ofb_undistort_points(ctx.h, None, ofb200._lib.ptr(pts), 4, None, ofb200._lib.ptr(out)) == ofb200._lib.OFB_E_INVALID
        assert lib.ofb_tracker_set_camera(None, C.byref(good)) == ofb200._lib.OFB_E_INVALID
        with pytest.raises(ValueError):
            trk.set_camera((K_WIDE, [0.1, 0.2, 0.3], 30.0))
        # still usable: the same calls with valid arguments
        ref = ofb200.frame_pairs(prev, nxt, imu, cfg, ctx=ctx)
        got = ofb200.frame_pairs(prev, nxt, imu, cfg, ctx=ctx, camera=(np.array([[mo["f"], 0, mo["cx"]], [0, mo["f"], mo["cy"]], [0, 0, 1.0]]),
                                                                          None, 1.0 / mo["dt"]))
        assert relerr(got["v"][0], ref["v"][0]) <= 1e-9
        trk.set_camera(good)
        trk.set_camera(None)
        assert np.abs(ofb200.undistortPoints(pts, K_WIDE, D_WIDE, ctx=ctx).reshape(-1, 2) - co.undistort(pts, K_WIDE, D_WIDE, 5)).max() <= 1e-14
    finally:
        trk.close()


def test_fleet_tracker_camera(ofb200, ctx):
    frames, imus, kw = tc.build("module")
    cam = cam_for(kw)
    fleet = ofb200.FleetTracker(2, tc.W, tc.H, ctx=ctx, camera=cam, **kw)
    ref = ofb200.StreamTracker(tc.W, tc.H, n_streams=2, ctx=ctx, camera=cam, **kw)
    try:
        for k in range(3):
            if k == 2:
                fleet.set_camera(None); ref.set_camera(None)
            samples = [imus[s][k] for s in range(2)]
            fr = np.stack([frames[s][k] for s in range(2)])
            pri = np.stack([s["v_prior"] for s in samples])
            a = fleet.step(fr, imu_records(ofb200, samples), v_prior=pri)
            r = ref.step(fr, imu_records(ofb200, samples), v_prior=pri)
            assert all(same_record(a[s], r[s]) for s in range(2))
    finally:
        fleet.close()
        ref.close()
