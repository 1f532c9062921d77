"""Ego-motion solve on the GPU (include/ofb200.h `ofb_solve_ego_motion*`, `ofb_frame_pairs_ego`,
`ofb_tracker_set_ego_motion`, `ofb_tracker_step_ego`) against the literal 3N x 6 lstsq of oracle/ego_oracle.py, the
motion truth of the synthetic pairs, and the records of the paths with ego-motion off."""
import ctypes as C
import os

import numpy as np
import pytest

import synth
import tracker_cases as tc
from conftest import GOLDEN
from oracle import camera_oracle as co
from oracle import ego_oracle as eo
from oracle import velocity_oracle as vo
from test_gpu_camera import cam_for
from test_gpu_tracker import imu_records, same_record

pytestmark = pytest.mark.gpu
VARIANTS = ["node", "exp", "sim"]


@pytest.fixture(scope="module")
def ofb200():
    import ofb200
    return ofb200


def flow_scene(seed, spread, n_pts=300, noise=2e-4, x=None):
    rng = np.random.default_rng(seed)
    if x is None:
        x = rng.uniform(-spread, spread, (n_pts, 2))
    v = rng.uniform(-1, 1, 3)
    w = rng.normal(0, 0.3, 3)
    n = np.array([rng.normal(0, 0.1), rng.normal(0, 0.1), 1.0])
    n /= np.linalg.norm(n)
    d, t = rng.uniform(0.5, 5.0), rng.normal(0, 0.1, 3)
    u = vo.generate_test_data(x, v, w, d, n, t) + rng.normal(0, noise, x.shape)
    return x, u, d, n, t


def check_against_oracle(got, x, u, d, n, t, variant):
    """v, w, rank, s and res of a device record against lstsq on the stacked system"""
    ve, we, res, rank, s = eo.solve_ego_motion(x, u, d, n, t, variant)
    A, _ = eo.build_system(x, u, d, n, variant)
    sv = np.zeros(6)
    if len(x):
        sv[:min(A.shape)] = np.linalg.svd(A, compute_uv=False)         # a 1-point system has 3 singular values
    cond = sv[0] / sv[5] if sv[5] > 0 else np.inf
    assert int(got["rank"]) == rank
    tol = 1e-9 if cond <= 300 else 1e-14 * cond ** 2
    if rank == 6:
        for a, b in ((got["v"], ve), (got["w"], we)):
            assert np.abs(a - b).max() <= tol * max(np.abs(b).max(), 1e-300), (variant, cond)
        np.testing.assert_allclose(got["res"], res[0] if res.size else got["res"], rtol=1e-6, atol=1e-18)
    s_ref = np.zeros(6)
    s_ref[:len(s)] = s
    smax = max(s_ref[0], 1e-300)
    bound = 1e-13 * smax ** 2 / np.maximum(s_ref, 1e-300 * smax) + 1e-13 * smax
    assert (np.abs(got["s"] - s_ref) <= bound).all(), (got["s"], s_ref)
    return cond


# ---- standalone solve -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("spread", [0.6, 0.3, 0.05])
@pytest.mark.parametrize("lever", [False, True])
def test_standalone_vs_oracle(ofb200, ctx, variant, spread, lever):
    x, u, d, n, t = flow_scene(int(spread * 100) + len(variant), spread)
    tt = t if lever else None
    v, w, res, rank, s = ofb200.solve_ego_motion(x, u, d, n, tt, variant=variant, ctx=ctx)
    rec = np.zeros(1, ofb200._lib.EGO_RESULT_DTYPE)[0]
    rec["v"], rec["w"], rec["rank"], rec["s"] = v, w, rank, s
    rec["res"] = res[0] if res.size else 0.0
    check_against_oracle(rec, x, u, d, n, tt, variant)
    assert res.shape == ((1,) if rank == 6 else (0,))


@pytest.mark.parametrize("variant", VARIANTS)
def test_golden_points_and_device_pointers(ofb200, ctx, variant):
    import torch
    pts = np.load(os.path.join(GOLDEN, "points.npy")).reshape(-1, 2).astype(np.float64)
    x = (pts - pts.mean(0)) / (2 * np.abs(pts - pts.mean(0)).max())      # normalised, about +-0.5
    x, u, d, n, t = flow_scene(40, 0.0, x=x)
    host = ofb200.solve_ego_motion(x, u, d, n, t, variant=variant, ctx=ctx)
    rec = np.zeros(1, ofb200._lib.EGO_RESULT_DTYPE)
    dx, du = torch.from_numpy(x).cuda(), torch.from_numpy(u).cuda()
    dn, dt = torch.from_numpy(n).cuda(), torch.from_numpy(t).cuda()
    drec = torch.zeros(rec.nbytes, dtype=torch.uint8, device="cuda")
    ofb200._lib.check(ctx.lib.ofb_solve_ego_motion(ctx.h, ofb200._lib.VARIANTS[variant], ofb200._lib.ptr(dx), ofb200._lib.ptr(du),
                                                   len(x), d, ofb200._lib.ptr(dn), ofb200._lib.ptr(dt), ofb200._lib.ptr(drec)))
    ctx.sync()
    dev = drec.cpu().numpy().view(ofb200._lib.EGO_RESULT_DTYPE)[0]
    assert np.array_equal(dev["v"], host[0]) and np.array_equal(dev["w"], host[1]) and dev["rank"] == host[3]
    assert dev["flags"] == ofb200._lib.EGO_SOLVED
    check_against_oracle(dev, x, u, d, n, t, variant)
    # the fixed-rate identity through the gyro-based solve
    vg = ofb200.solve_lgs(x, u, d, n, dev["w"], t, variant=variant, ctx=ctx)[0]
    np.testing.assert_allclose(vg, dev["v"], rtol=0, atol=1e-9 * np.abs(dev["v"]).max())


def test_batched_with_empty_frames_and_device_offsets(ofb200, ctx):
    import torch
    frames = [flow_scene(50 + k, [0.6, 0.3, 0.05, 0.6][k % 4], n_pts=[200, 0, 3, 150, 1, 90][k]) if k not in (1,) else None
              for k in range(6)]
    xs, us, offs, ds, ns, ts = [], [], [0], [], [], []
    for f in frames:
        x, u, d, n, t = f if f is not None else (np.zeros((0, 2)), np.zeros((0, 2)), 1.0, np.array([0, 0, 1.0]), np.zeros(3))
        xs.append(x); us.append(u); offs.append(offs[-1] + len(x)); ds.append(d); ns.append(n); ts.append(t)
    X, U = np.concatenate(xs), np.concatenate(us)
    for variant in VARIANTS:
        recs = ofb200.solve_ego_motion_batched(X, U, offs, np.array(ds), np.stack(ns), np.stack(ts), variant=variant, ctx=ctx)
        for k in range(len(frames)):
            r = recs[k]
            assert r["flags"] == ofb200._lib.EGO_SOLVED
            if offs[k + 1] == offs[k]:
                assert r["rank"] == 0 and not r["v"].any() and not r["w"].any() and not r["s"].any()
                continue
            check_against_oracle(r, xs[k], us[k], ds[k], ns[k], ts[k], variant)
            one = ofb200.solve_ego_motion(xs[k], us[k], ds[k], ns[k], ts[k], variant=variant, ctx=ctx)
            assert np.array_equal(one[0], r["v"]) and np.array_equal(one[1], r["w"])
    d_off = torch.from_numpy(np.asarray(offs, np.int32)).cuda()
    out = np.zeros(len(frames), ofb200._lib.EGO_RESULT_DTYPE)
    dd, dn, dt = np.array(ds), np.ascontiguousarray(np.stack(ns)), np.ascontiguousarray(np.stack(ts))
    ofb200._lib.check(ctx.lib.ofb_solve_ego_motion_batched(ctx.h, 2, ofb200._lib.ptr(X), ofb200._lib.ptr(U), ofb200._lib.ptr(d_off),
                                                           len(frames), ofb200._lib.ptr(dd), ofb200._lib.ptr(dn), ofb200._lib.ptr(dt),
                                                           ofb200._lib.ptr(out)))
    assert all(same_record(a, b) for a, b in zip(out, recs))


# ---- frame pairs ------------------------------------------------------------------------------------------------
def pair_batch(ofb200, n=4, h=240, w=320):
    pairs = [synth.make_pair(h, w, k, k, max_disp=6.0) for k in range(n)]
    prev, nxt = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    imu = np.zeros(n, ofb200._lib.IMU_DTYPE)
    for k, (_, _, mo) in enumerate(pairs):
        imu["d"][k], imu["n"][k], imu["w"][k] = mo["d"], mo["n"], mo["w"]
        imu["t"][k] = [0.02, -0.01, 0.05]
    f, dt = pairs[0][2]["f"], pairs[0][2]["dt"]
    return prev, nxt, imu, f, dt, [p[2] for p in pairs]


@pytest.mark.parametrize("camera", [False, True])
@pytest.mark.parametrize("fb", [None, 0.5])
@pytest.mark.parametrize("gyro", [False, True])
def test_frame_pairs_ego_vs_oracle(ofb200, ctx, camera, fb, gyro):
    prev, nxt, imu, f, dt, mos = pair_batch(ofb200)
    h, w = prev.shape[1:]
    cfg = ofb200.make_pair_cfg(w, h, 200, 0.01, 8, 7, (15, 15), 3, (3, 20, 0.03), variant="exp", pos_scale=1 / f,
                               flow_scale=1 / (f * dt))
    cam = None
    if camera:
        K = np.array([[f, 0.0, mos[0]["cx"] + 0.5], [0.0, f * 0.998, mos[0]["cy"] - 0.5], [0.0, 0.0, 1.0]])
        cam = (K, np.array([-0.02, 0.004, 0.0003, -0.0002, 0.0]), 1.0 / dt, 20)
    kw = dict(want_tracks=True, ctx=ctx, camera=cam, fb_threshold=fb, gyro_prediction=gyro)
    base = ofb200.frame_pairs(prev, nxt, imu, cfg, **kw)
    res, pp, pn, st, ego = ofb200.frame_pairs(prev, nxt, imu, cfg, ego_motion=True, **kw)
    assert all(same_record(a, b) for a, b in zip(base[0], res))
    for x_, y_ in zip(base[1:], (pp, pn, st)):
        assert np.array_equal(x_, y_)
    for k in range(len(prev)):
        nf = int(res["n_features"][k])
        ok = st[k, :nf] == 1
        p0, p1 = pp[k, :nf][ok], pn[k, :nf][ok]
        if camera:
            x, u = co.calibrate(p1, p0, cam)
        else:
            x = (p1.astype(np.float64) - [cfg.cx, cfg.cy]) * cfg.pos_scale
            u = (p1 - p0).astype(np.float64) * cfg.flow_scale                 # the fp32 difference, as TrackLoader forms it
        assert ego["flags"][k] == ofb200._lib.EGO_SOLVED
        check_against_oracle(ego[k], x, u, imu["d"][k], imu["n"][k], imu["t"][k], "exp")


def test_frame_pairs_ego_routes_and_sequence(ofb200, ctx):
    """host pipeline, resident twin chunks and the sequence layout give one set of ego records"""
    import torch
    h, w, n = 240, 320, 12
    frames = np.stack([synth.make_pair(h, w, 3, k, max_disp=5.0)[0 if k == 0 else 1] for k in range(n + 1)])
    imu = np.zeros(n, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"][:, 2] = 2.0, 1.0
    cfg = ofb200.make_pair_cfg(w, h, 150, 0.01, 8, 7, (15, 15), 3, (3, 20, 0.03), variant="node", pos_scale=1 / 256.0,
                               flow_scale=1 / 8.0)
    host = ofb200.frame_pairs(frames[:-1].copy(), frames[1:].copy(), imu, cfg, ctx=ctx, ego_motion=True)
    seq = ofb200.frame_sequence(frames, imu, cfg, ctx=ctx, ego_motion=True)
    d = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    twin = ofb200.frame_pairs(d[:-1].contiguous(), d[1:].contiguous(), imu, cfg, ctx=ctx, ego_motion=True)
    for other in (seq, twin):
        assert all(same_record(host[0][i], other[0][i]) for i in range(n))
        assert all(same_record(host[1][i], other[1][i]) for i in range(n))


def test_frame_pairs_ego_truth_720p(ofb200, ctx):
    """|w_hat - w| f dt <= 0.5 px on synth.make_pair motions at 1280 x 720 (no gyro sample is used). The least squares
    has no outlier rejection: without the forward-backward check a few status-1 tracks that are 5-17 px off move w_hat
    by up to 0.84 px on these pairs (cv2 4.13 gives the same tracks); with it every pair is within 0.15 px."""
    h, w, n = 720, 1280, 6
    pairs = [synth.make_pair(h, w, 20 + k, 20 + k) for k in range(n)]
    prev, nxt = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    mo0 = pairs[0][2]
    f, dt = mo0["f"], mo0["dt"]
    imu = np.zeros(n, ofb200._lib.IMU_DTYPE)
    for k, (_, _, mo) in enumerate(pairs):
        imu["d"][k], imu["n"][k] = mo["d"], mo["n"]
        imu["w"][k] = [0.3, -0.2, 0.1]                                         # a wrong gyro: it must not matter
    cfg = ofb200.make_pair_cfg(w, h, 400, 0.01, 10, 7, (21, 21), 3, (3, 30, 0.01), variant="node", pos_scale=1 / f,
                               flow_scale=1 / (f * dt))
    res, ego = ofb200.frame_pairs(prev, nxt, imu, cfg, ctx=ctx, fb_threshold=0.5, ego_motion=True)
    errs = [np.abs(ego["w"][k] - pairs[k][2]["w"]).max() * f * dt for k in range(n)]
    print("ego rate error (px):", np.round(errs, 3))
    assert (ego["rank"] == 6).all()
    assert max(errs) <= 0.5, errs


# ---- tracker ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scenario,camera", [("exp", False), ("node", False), ("module", False), ("exp", True)])
def test_tracker_ego_vs_oracle(ofb200, ctx, scenario, camera):
    frames, imus, kw = tc.build(scenario)
    S = len(frames)
    cam = cam_for(kw) if camera else None
    trk = ofb200.StreamTracker(tc.W, tc.H, n_streams=S, ctx=ctx, camera=cam, ego_motion=True, **kw)
    ref = ofb200.StreamTracker(tc.W, tc.H, n_streams=S, ctx=ctx, camera=cam, **kw)
    solved = 0
    try:
        for k in range(len(frames[0])):
            samples = [imus[s][k] for s in range(S)]
            fr = np.stack([frames[s][k] for s in range(S)])
            pri = None if samples[0]["v_prior"] is None else np.stack([s["v_prior"] for s in samples])
            res, kp, kn, ego = trk.step(fr, imu_records(ofb200, samples), v_prior=pri, want_kept=True, want_ego=True)
            r0, kp0, kn0 = ref.step(fr, imu_records(ofb200, samples), v_prior=pri, want_kept=True)
            assert all(same_record(a, b) for a, b in zip(res, r0))
            assert all(np.array_equal(a, b) for a, b in zip(kp + kn, kp0 + kn0))
            for s in range(S):
                if not res["flags"][s] & ofb200._lib.TRACK_SOLVED:
                    assert ego["flags"][s] == 0 and not ego["v"][s].any()
                    continue
                solved += 1
                assert ego["flags"][s] == ofb200._lib.EGO_SOLVED
                if camera:
                    x, u = co.calibrate(kn[s], kp[s], cam)
                else:
                    x = (kn[s].astype(np.float64) - vo.pix_trans((tc.W, tc.H))) * kw["scaling"]
                    u = (kn[s] - kp[s]).astype(np.float64) * kw["scaling"]
                im = samples[s]
                check_against_oracle(ego[s], x, u, im["d"], im["n"], im["t"], kw["variant"])
    finally:
        trk.close()
        ref.close()
    assert solved >= 2


SWITCH = {3: True, 6: False, 9: True}


def run_modes(ofb200, kw, frames, imus, mode, monkeypatch, switch, start):
    """as tests/test_gpu_gyro.run_switching, switching ego-motion; -> per step (record, ego record or None)"""
    import torch
    monkeypatch.setenv("OFB_TRACKER_GRAPH", "0" if mode == "plain" else "1")
    monkeypatch.setenv("OFB_TRACKER_SPLIT_SOLVE", "0" if mode == "nosplit" else "1")
    ctx = ofb200.Context(0)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, ego_motion=start, **kw)
    order = list(range(len(frames))) + list(range(len(frames) - 2, -1, -1))
    out = []
    L = ofb200._lib
    dev = mode in ("split", "nosplit")
    d_res = torch.zeros(C.sizeof(L.TrackResult), dtype=torch.uint8, device="cuda") if dev else None
    d_ego = torch.zeros(C.sizeof(L.EgoResult), dtype=torch.uint8, device="cuda") if dev else None
    try:
        on = start
        for j, k in enumerate(order):
            if j in switch:
                trk.set_ego_motion(switch[j])
                on = switch[j]
            im = imu_records(ofb200, [imus[k]])
            if dev:
                fr = torch.from_numpy(frames[k]).cuda()
                d_imu = torch.from_numpy(im.view(np.uint8).copy()).cuda()
                L.check(ctx.lib.ofb_tracker_step_ego(trk.h, L.ptr(fr), tc.W, tc.W * tc.H, L.ptr(d_imu), None, L.ptr(d_res),
                                                     None, None, None, None, L.ptr(d_ego) if on else None))
                ctx.sync()
                out.append((d_res.cpu().numpy().view(L.TRACK_RESULT_DTYPE).copy(),
                            d_ego.cpu().numpy().view(L.EGO_RESULT_DTYPE).copy() if on else None))
            elif mode == "kept":
                r = trk.step(frames[k], im, want_kept=True, want_ego=on)
                out.append((r[0], r[3] if on else None))
            else:
                r = trk.step(frames[k], im, want_ego=on)
                out.append((r[0], r[1]) if on else (r, None))
        graph_steps = trk.graph_steps()
    finally:
        trk.close()
        ctx.close()
    return out, graph_steps, order


def test_tracker_modes_and_switching(ofb200, monkeypatch):
    """graph / plain / kept / split / nosplit: the standard records equal a tracker without ego-motion, the ego records
    are one set in every mode, and switching it on mid-run gives the records of a tracker built with it on"""
    frames, imus, kw = tc.build("exp")
    frames, imus = frames[0], imus[0]
    off, _, order = run_modes(ofb200, kw, frames, imus, "plain", monkeypatch, {}, False)
    full, _, _ = run_modes(ofb200, kw, frames, imus, "plain", monkeypatch, {}, True)
    assert any(e["flags"][0] for _, e in full)
    for mode in ("graph", "plain", "kept", "split", "nosplit"):
        got, graph_steps, _ = run_modes(ofb200, kw, frames, imus, mode, monkeypatch, SWITCH, False)
        if mode == "graph":
            assert graph_steps >= 6, graph_steps
        for j in range(len(order)):
            assert same_record(got[j][0][0], off[j][0][0]), (mode, j)
            if got[j][1] is not None:
                assert same_record(got[j][1][0], full[j][1][0]), (mode, j)
    # graph replay with ego-motion on from the start
    got, graph_steps, _ = run_modes(ofb200, kw, frames, imus, "graph", monkeypatch, {}, True)
    assert graph_steps >= 6
    assert all(same_record(got[j][1][0], full[j][1][0]) for j in range(len(order)))


def test_fleet_tracker_ego(ofb200, ctx):
    frames, imus, kw = tc.build("module")
    fleet = ofb200.FleetTracker(2, tc.W, tc.H, ctx=ctx, ego_motion=True, **kw)
    ref = ofb200.StreamTracker(tc.W, tc.H, n_streams=2, ctx=ctx, ego_motion=True, **kw)
    try:
        for k in range(4):
            samples = [imus[s][k] for s in range(2)]
            fr = np.stack([frames[s][k] for s in range(2)])
            pri = np.stack([s["v_prior"] for s in samples])
            a = fleet.step(fr, imu_records(ofb200, samples), v_prior=pri, want_ego=True)
            r = ref.step(fr, imu_records(ofb200, samples), v_prior=pri, want_ego=True)
            assert all(same_record(a[1][s], r[1][s]) for s in range(2))
    finally:
        fleet.close()
        ref.close()


# ---- errors -----------------------------------------------------------------------------------------------------
def test_errors_leave_the_context_usable(ofb200, ctx):
    x, u, d, n, t = flow_scene(60, 0.5)
    L = ofb200._lib
    rec = np.zeros(1, L.EGO_RESULT_DTYPE)
    with pytest.raises(ValueError):
        L.check(ctx.lib.ofb_solve_ego_motion(ctx.h, L.VARIANT_MODULE, L.ptr(x), L.ptr(u), len(x), d, L.ptr(n), None, L.ptr(rec)))
    with pytest.raises(ValueError):
        L.check(ctx.lib.ofb_solve_ego_motion(ctx.h, 0, None, L.ptr(u), len(x), d, L.ptr(n), None, L.ptr(rec)))
    with pytest.raises(ValueError):
        L.check(ctx.lib.ofb_solve_ego_motion(ctx.h, 0, L.ptr(x), L.ptr(u), len(x), d, None, None, L.ptr(rec)))
    with pytest.raises(ValueError):
        L.check(ctx.lib.ofb_solve_ego_motion_batched(ctx.h, 0, L.ptr(x), L.ptr(u), L.ptr(np.array([0, 5, 2], np.int32)), 2,
                                                     L.ptr(np.ones(2)), L.ptr(np.tile(n, 2)), None, L.ptr(np.zeros(2, L.EGO_RESULT_DTYPE))))
    frames, imus, kw = tc.build("exp")
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, **kw)
    mod = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, **dict(kw, variant="module"))
    try:
        with pytest.raises(ValueError):
            trk.step(frames[0][0], imu_records(ofb200, [imus[0][0]]), want_ego=True)
        with pytest.raises(ValueError):
            L.check(ctx.lib.ofb_tracker_step_ego(trk.h, L.ptr(frames[0][0]), tc.W, tc.W * tc.H, L.ptr(imu_records(ofb200, [imus[0][0]])),
                                                 None, L.ptr(np.zeros(1, L.TRACK_RESULT_DTYPE)), None, None, None, None, L.ptr(rec)))
        with pytest.raises(ValueError):
            mod.set_ego_motion(True)
        with pytest.raises(ValueError):
            trk.set_ego_motion(1)
    finally:
        trk.close()
        mod.close()
    v, w, res, rank, s = ofb200.solve_ego_motion(x, u, d, n, t, variant="sim", ctx=ctx)
    assert rank == 6 and res.shape == (1,)
    check = eo.solve_ego_motion(x, u, d, n, t, "sim")
    np.testing.assert_allclose(w, check[1], rtol=1e-8, atol=1e-12)
