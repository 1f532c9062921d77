"""Robust velocity solve on the GPU (include/ofb200.h `ofb_solve_velocity_robust*`, `ofb_frame_pairs_robust`,
`ofb_tracker_set_robust`, `ofb_tracker_step_robust`) against oracle/robust_oracle.py, the plain solve, the motion truth
of an image scene with a moving object, and the records of the paths with the robust solve off."""
import ctypes as C

import numpy as np
import pytest

import robust_cases as rc
import synth
import tracker_cases as tc
from oracle import camera_oracle as co
from oracle import robust_oracle as ro
from oracle import velocity_oracle as vo
from test_gpu_camera import cam_for
from test_gpu_ego import pair_batch
from test_gpu_tracker import imu_records, same_record

pytestmark = pytest.mark.gpu
VARIANTS = ["node", "exp", "sim"]


@pytest.fixture(scope="module")
def ofb200():
    import ofb200
    return ofb200


def flow_scene(seed, spread, n_pts=300, noise=2e-4, frac=0.2):
    """the plane's flow with a share `frac` of the points moving with a velocity of their own"""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-spread, spread, (n_pts, 2))
    v = rng.uniform(-1, 1, 3)
    w = rng.normal(0, 0.3, 3)
    n = np.array([rng.normal(0, 0.1), rng.normal(0, 0.1), 1.0])
    n /= np.linalg.norm(n)
    d, t = rng.uniform(0.5, 5.0), rng.normal(0, 0.1, 3)
    u = vo.generate_test_data(x, v, w, d, n, t) + rng.normal(0, noise, x.shape)
    k = int(frac * n_pts)
    u[:k] = vo.generate_test_data(x[:k], v + rng.uniform(-3, 3, 3), w, d, n, t) + rng.normal(0, noise, (k, 2))
    return x, u, d, n, w, t


def check_against_oracle(got, x, u, d, n, w, t, variant, c=4.0, K=10, weights=None):
    """A device record (and weights) against the oracle. v within 1e-9 relative where the last weighted system has
    cond <= 300; n_inliers, iterations and scale exact unless some rho_i lies within 1e-9 relative of tau (a point at the
    cut-off may then fall on either side).
    A single point is fitted exactly: its residual, and so the scale, is rounding noise that differs between the device
    and NumPy. The iteration still runs, and the point's weight is (1 - (rho/tau)^2)^2 with rho/tau = rho / (c (float)rho),
    i.e. 1/c up to the fp32 rounding of the key (2^-24 relative). The weighted system is the plain one times that weight,
    so the solution does not depend on it and s is the plain solve's times sqrt(weight): equal to the oracle's within
    ~1e-7 relative instead of the eigen-solver's resolution. The scale itself is not compared there."""
    ref = ro.solve_velocity_robust(x, u, d, n, w, t, variant, c, K)
    exact = len(x) == 1
    near = ref["iterations"] > 0 and np.any(np.abs(ref["rho_w"] - ref["tau"]) <= 1e-9 * ref["tau"])
    near = near or exact
    if not near:
        assert int(got["iterations"]) == ref["iterations"] and int(got["n_inliers"]) == ref["n_inliers"]
        assert got["scale"] == ref["scale"]
    assert int(got["rank"]) == ref["rank"]
    s_ref = ref["s"]
    cond = s_ref[0] / s_ref[2] if s_ref[2] > 0 else np.inf
    if ref["rank"] == 3:
        tol = 1e-9 if cond <= 300 else 1e-14 * cond ** 2
        assert np.abs(got["v"] - ref["v"]).max() <= tol * max(np.abs(ref["v"]).max(), 1e-300), (variant, cond)
        np.testing.assert_allclose(got["res"], ref["res"], rtol=1e-6, atol=1e-18)
    smax = max(s_ref[0], 1e-300)
    bound = 1e-13 * smax ** 2 / np.maximum(s_ref, 1e-300 * smax) + 1e-13 * smax
    if exact:
        bound = 1e-6 * s_ref + 1e-13 * smax
    assert (np.abs(got["s"] - s_ref) <= bound).all(), (got["s"], s_ref)
    if weights is not None and not near:
        np.testing.assert_allclose(weights, ref["weights"], rtol=0, atol=1e-9)
    return ref


# ---- standalone solve -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("spread", [0.6, 0.3, 0.05])
@pytest.mark.parametrize("lever", [False, True])
def test_standalone_vs_oracle(ofb200, ctx, variant, spread, lever):
    x, u, d, n, w, t = flow_scene(int(spread * 100) + len(variant), spread)
    tt = t if lever else None
    rec, wts = ofb200.solve_velocity_robust(x, u, d, n, w, tt, variant=variant, want_weights=True, ctx=ctx)
    assert rec["flags"] == ofb200._lib.ROBUST_SOLVED
    ref = check_against_oracle(rec, x, u, d, n, w, tt, variant, weights=wts)
    assert ref["iterations"] >= 1


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("lever", [False, True])
def test_zero_iterations_is_the_plain_solve_bit_for_bit(ofb200, ctx, variant, lever):
    for seed, spread in ((1, 0.6), (2, 0.05), (3, 0.3)):
        x, u, d, n, w, t = flow_scene(seed, spread)
        tt = t if lever else None
        rec, wts = ofb200.solve_velocity_robust(x, u, d, n, w, tt, variant=variant, iterations=0, want_weights=True, ctx=ctx)
        v, res, rank, s = ofb200.solve_full(x, u, d, n, w, tt, variant=variant, ctx=ctx)
        assert np.array_equal(rec["v"], v) and np.array_equal(rec["s"], s) and rec["rank"] == rank
        assert res.size == 0 or rec["res"] == res[0]
        assert rec["iterations"] == 0 and rec["scale"] == 0.0 and rec["n_inliers"] == len(x)
        assert np.array_equal(wts, np.ones(len(x)))


def test_device_pointers_and_determinism(ofb200, ctx):
    import torch
    L = ofb200._lib
    x, u, d, n, w, t = flow_scene(40, 0.5, n_pts=2000)
    host, hw = ofb200.solve_velocity_robust(x, u, d, n, w, t, variant="sim", want_weights=True, ctx=ctx)
    dx, du, dn, dw, dt = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (x, u, n, w, t))
    drec = torch.zeros(C.sizeof(L.RobustResult), dtype=torch.uint8, device="cuda")
    dwts = torch.zeros(len(x), dtype=torch.float64, device="cuda")
    cfg = L.RobustCfg(4.0, 10)
    L.check(ctx.lib.ofb_solve_velocity_robust(ctx.h, L.VARIANTS["sim"], L.ptr(dx), L.ptr(du), len(x), d, L.ptr(dn), L.ptr(dw),
                                              L.ptr(dt), C.byref(cfg), L.ptr(drec), L.ptr(dwts)))
    ctx.sync()
    dev = drec.cpu().numpy().view(L.ROBUST_RESULT_DTYPE)[0]
    assert same_record(dev, host) and np.array_equal(dwts.cpu().numpy(), hw)
    again, aw = ofb200.solve_velocity_robust(x, u, d, n, w, t, variant="sim", want_weights=True, ctx=ctx)
    assert host.tobytes() == again.tobytes() and np.array_equal(hw, aw)
    check_against_oracle(host, x, u, d, n, w, t, "sim", weights=hw)


def test_batched_with_empty_frames_and_device_offsets(ofb200, ctx):
    import torch
    L = ofb200._lib
    sizes = [200, 0, 3, 150, 1, 90, 2]
    frames = [flow_scene(50 + k, [0.6, 0.3, 0.05][k % 3], n_pts=m) for k, m in enumerate(sizes)]
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    X, U = np.concatenate([f[0] for f in frames]), np.concatenate([f[1] for f in frames])
    ds = np.array([f[2] for f in frames])
    ns, ws, ts = (np.ascontiguousarray(np.stack([f[i] for f in frames])) for i in (3, 4, 5))
    for variant in VARIANTS:
        recs, wts = ofb200.solve_velocity_robust_batched(X, U, offs, ds, ns, ws, ts, variant=variant, c=3.0, iterations=6,
                                                         want_weights=True, ctx=ctx)
        for k, f in enumerate(frames):
            r = recs[k]
            assert r["flags"] == L.ROBUST_SOLVED
            if sizes[k] == 0:                         # v' = 0; EXP and SIM still remove the lever arm, as the plain solve does
                assert r["rank"] == 0 and r["iterations"] == 0 and r["n_inliers"] == 0 and not r["s"].any()
                lever = np.zeros(3) if variant == "node" else -np.cross(f[4], f[5])
                np.testing.assert_allclose(r["v"], lever, rtol=1e-15, atol=1e-18)
                continue
            one, ow = ofb200.solve_velocity_robust(f[0], f[1], f[2], f[3], f[4], f[5], variant=variant, c=3.0, iterations=6,
                                                   want_weights=True, ctx=ctx)
            assert same_record(one, r) and np.array_equal(ow, wts[offs[k]:offs[k + 1]])
            check_against_oracle(r, *f, variant, c=3.0, K=6, weights=ow)
    d_off = torch.from_numpy(offs).cuda()
    out = np.zeros(len(frames), L.ROBUST_RESULT_DTYPE)
    cfg = L.RobustCfg(3.0, 6)
    L.check(ctx.lib.ofb_solve_velocity_robust_batched(ctx.h, L.VARIANTS["sim"], L.ptr(X), L.ptr(U), L.ptr(d_off), len(frames),
                                                      L.ptr(ds), L.ptr(ns), L.ptr(ws), L.ptr(ts), C.byref(cfg), L.ptr(out), None))
    assert all(same_record(a, b) for a, b in zip(out, recs))


def test_no_cap_on_the_point_count(ofb200, ctx):
    x, u, d, n, w, t = flow_scene(77, 0.5, n_pts=200_000, frac=0.3)
    rec, wts = ofb200.solve_velocity_robust(x, u, d, n, w, t, variant="exp", want_weights=True, ctx=ctx)
    check_against_oracle(rec, x, u, d, n, w, t, "exp", weights=wts)
    assert rec["n_inliers"] < 0.8 * len(x) and rec["iterations"] >= 1


# ---- frame pairs ------------------------------------------------------------------------------------------------
def pair_points(cfg, pp, pn, st, k, nf, cam):
    ok = st[k, :nf] == 1
    p0, p1 = pp[k, :nf][ok], pn[k, :nf][ok]
    if cam is not None:
        return co.calibrate(p1, p0, cam)
    return (p1.astype(np.float64) - [cfg.cx, cfg.cy]) * cfg.pos_scale, (p1 - p0).astype(np.float64) * cfg.flow_scale


@pytest.mark.parametrize("camera", [False, True])
@pytest.mark.parametrize("fb", [None, 0.5])
@pytest.mark.parametrize("gyro", [False, True])
def test_frame_pairs_robust_vs_oracle(ofb200, ctx, camera, fb, gyro):
    prev, nxt, imu, f, dt, mos = pair_batch(ofb200)
    h, w = prev.shape[1:]
    cfg = ofb200.make_pair_cfg(w, h, 200, 0.01, 8, 7, (15, 15), 3, (3, 20, 0.03), variant="exp", pos_scale=1 / f,
                               flow_scale=1 / (f * dt))
    cam = None
    if camera:
        K = np.array([[f, 0.0, mos[0]["cx"] + 0.5], [0.0, f * 0.998, mos[0]["cy"] - 0.5], [0.0, 0.0, 1.0]])
        cam = (K, np.array([-0.02, 0.004, 0.0003, -0.0002, 0.0]), 1.0 / dt, 20)
    kw = dict(want_tracks=True, ctx=ctx, camera=cam, fb_threshold=fb, gyro_prediction=gyro)
    base = ofb200.frame_pairs(prev, nxt, imu, cfg, ego_motion=True, **kw)
    res, pp, pn, st, ego, rob = ofb200.frame_pairs(prev, nxt, imu, cfg, ego_motion=True, robust=True, **kw)
    assert base[0].tobytes() == res.tobytes() and base[4].tobytes() == ego.tobytes()
    for a, b in zip(base[1:4], (pp, pn, st)):
        assert np.array_equal(a, b)
    alone = ofb200.frame_pairs(prev, nxt, imu, cfg, robust=(3.0, 5), **kw)
    assert alone[0].tobytes() == res.tobytes()
    for k in range(len(prev)):
        x, u = pair_points(cfg, pp, pn, st, k, int(res["n_features"][k]), cam)
        assert rob["flags"][k] == ofb200._lib.ROBUST_SOLVED
        check_against_oracle(rob[k], x, u, imu["d"][k], imu["n"][k], imu["w"][k], imu["t"][k], "exp")
        check_against_oracle(alone[4][k], x, u, imu["d"][k], imu["n"][k], imu["w"][k], imu["t"][k], "exp", c=3.0, K=5)


def test_frame_pairs_robust_routes_and_sequence(ofb200, ctx):
    """host pipeline, resident twin chunks and the sequence layout give one set of robust records, and the standard
    records equal those with the robust solve off"""
    import torch
    h, w, n = 240, 320, 12
    frames = np.stack([synth.make_pair(h, w, 3, k, max_disp=5.0)[0 if k == 0 else 1] for k in range(n + 1)])
    imu = np.zeros(n, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"][:, 2] = 2.0, 1.0
    cfg = ofb200.make_pair_cfg(w, h, 150, 0.01, 8, 7, (15, 15), 3, (3, 20, 0.03), variant="node", pos_scale=1 / 256.0,
                               flow_scale=1 / 8.0)
    off = ofb200.frame_pairs(frames[:-1].copy(), frames[1:].copy(), imu, cfg, ctx=ctx)
    host = ofb200.frame_pairs(frames[:-1].copy(), frames[1:].copy(), imu, cfg, ctx=ctx, robust=True)
    assert off.tobytes() == host[0].tobytes()
    seq = ofb200.frame_sequence(frames, imu, cfg, ctx=ctx, robust=True)
    d = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    twin = ofb200.frame_pairs(d[:-1].contiguous(), d[1:].contiguous(), imu, cfg, ctx=ctx, robust=True)
    for other in (seq, twin):
        assert host[0].tobytes() == other[0].tobytes() and host[1].tobytes() == other[1].tobytes()
    assert (host[1]["flags"] == ofb200._lib.ROBUST_SOLVED).all()


def test_moving_object_scene(ofb200, ctx, capsys):
    """A textured patch of 10-25 % of the frame moves by (9, -7) px on its own. Its features track with status 1 and
    pass the forward-backward check, so the plain solve (check on) follows them part of the way; the robust solve stays
    near the ground's velocity. Measured on an NVIDIA B200 (1000 W): plain relative error 0.25 / 0.68 / 0.74 / 1.13,
    robust 0.0034 / 0.0061 / 0.0020 / 0.0020 (patch share of the kept tracks 9-28 %); the bounds keep a margin of 1.7x
    (plain) and 8x (robust)."""
    h, w = 480, 640
    plain_err, rob_err, patch_share = [], [], []
    for k, frac in enumerate([0.10, 0.15, 0.20, 0.25]):
        a, b, mo, box = rc.moving_patch_pair(h, w, 30 + k, frac)
        imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
        imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
        cfg = ofb200.make_pair_cfg(w, h, 400, 0.01, 10, 7, (21, 21), 3, (3, 30, 0.01), variant="node",
                                   principal=(mo["cx"], mo["cy"]), pos_scale=1 / mo["f"], flow_scale=1 / (mo["f"] * mo["dt"]))
        res, pp, pn, st, rob = ofb200.frame_pairs(a[None], b[None], imu, cfg, want_tracks=True, ctx=ctx, fb_threshold=0.5,
                                                  robust=True)
        nf = int(res["n_features"][0])
        ok = st[0, :nf] == 1
        inside = rc.in_patch(pp[0, :nf], box)
        assert (ok & inside).sum() >= 10                           # the object's features are tracked and kept
        patch_share.append((ok & inside).sum() / ok.sum())
        scale = np.abs(mo["v"]).max()
        plain_err.append(np.abs(res["v"][0] - mo["v"]).max() / scale)
        rob_err.append(np.abs(rob["v"][0] - mo["v"]).max() / scale)
    with capsys.disabled():
        print("\nmoving object: share of kept tracks", np.round(patch_share, 3), "plain rel. error", np.round(plain_err, 3),
              "robust rel. error", np.round(rob_err, 4))
    assert min(plain_err) > 0.15
    assert max(rob_err) < 0.05
    assert all(r < 0.1 * p for r, p in zip(rob_err, plain_err))


# ---- tracker ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scenario,camera", [("exp", False), ("node", False), ("exp", True)])
def test_tracker_robust_vs_oracle(ofb200, ctx, scenario, camera):
    frames, imus, kw = tc.build(scenario)
    S = len(frames)
    cam = cam_for(kw) if camera else None
    trk = ofb200.StreamTracker(tc.W, tc.H, n_streams=S, ctx=ctx, camera=cam, robust=True, ego_motion=True, **kw)
    ref = ofb200.StreamTracker(tc.W, tc.H, n_streams=S, ctx=ctx, camera=cam, ego_motion=True, **kw)
    solved = 0
    try:
        for k in range(len(frames[0])):
            samples = [imus[s][k] for s in range(S)]
            fr = np.stack([frames[s][k] for s in range(S)])
            pri = None if samples[0]["v_prior"] is None else np.stack([s["v_prior"] for s in samples])
            res, kp, kn, ego, rob = trk.step(fr, imu_records(ofb200, samples), v_prior=pri, want_kept=True, want_ego=True,
                                             want_robust=True)
            r0, kp0, kn0, ego0 = ref.step(fr, imu_records(ofb200, samples), v_prior=pri, want_kept=True, want_ego=True)
            assert all(same_record(a, b) for a, b in zip(res, r0)) and ego.tobytes() == ego0.tobytes()
            assert all(np.array_equal(a, b) for a, b in zip(kp + kn, kp0 + kn0))
            for s in range(S):
                if not res["flags"][s] & ofb200._lib.TRACK_SOLVED:
                    assert rob[s].tobytes() == np.zeros(1, ofb200._lib.ROBUST_RESULT_DTYPE).tobytes()
                    continue
                solved += 1
                assert rob["flags"][s] == ofb200._lib.ROBUST_SOLVED
                if camera:
                    x, u = co.calibrate(kn[s], kp[s], cam)
                else:
                    x = (kn[s].astype(np.float64) - vo.pix_trans((tc.W, tc.H))) * kw["scaling"]
                    u = (kn[s] - kp[s]).astype(np.float64) * kw["scaling"]
                im = samples[s]
                check_against_oracle(rob[s], x, u, im["d"], im["n"], im["w"], im["t"], kw["variant"])
    finally:
        trk.close()
        ref.close()
    assert solved >= 2


SWITCH = {3: True, 6: False, 9: True}


def run_modes(ofb200, kw, frames, imus, mode, monkeypatch, switch, start):
    """as tests/test_gpu_ego.run_modes, switching the robust solve; -> per step (record, robust record or None)"""
    import torch
    monkeypatch.setenv("OFB_TRACKER_GRAPH", "0" if mode == "plain" else "1")
    monkeypatch.setenv("OFB_TRACKER_SPLIT_SOLVE", "0" if mode == "nosplit" else "1")
    ctx = ofb200.Context(0)
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, robust=start, **kw)
    order = list(range(len(frames))) + list(range(len(frames) - 2, -1, -1))
    out = []
    L = ofb200._lib
    dev = mode in ("split", "nosplit")
    d_res = torch.zeros(C.sizeof(L.TrackResult), dtype=torch.uint8, device="cuda") if dev else None
    d_rob = torch.zeros(C.sizeof(L.RobustResult), dtype=torch.uint8, device="cuda") if dev else None
    try:
        on = start
        for j, k in enumerate(order):
            if j in switch:
                trk.set_robust(switch[j])
                on = switch[j]
            im = imu_records(ofb200, [imus[k]])
            if dev:
                fr = torch.from_numpy(frames[k]).cuda()
                d_imu = torch.from_numpy(im.view(np.uint8).copy()).cuda()
                L.check(ctx.lib.ofb_tracker_step_robust(trk.h, L.ptr(fr), tc.W, tc.W * tc.H, L.ptr(d_imu), None, L.ptr(d_res),
                                                        None, None, None, None, None, L.ptr(d_rob) if on else None))
                ctx.sync()
                out.append((d_res.cpu().numpy().view(L.TRACK_RESULT_DTYPE).copy(),
                            d_rob.cpu().numpy().view(L.ROBUST_RESULT_DTYPE).copy() if on else None))
            elif mode == "kept":
                r = trk.step(frames[k], im, want_kept=True, want_robust=on)
                out.append((r[0], r[3] if on else None))
            else:
                r = trk.step(frames[k], im, want_robust=on)
                out.append((r[0], r[1]) if on else (r, None))
        graph_steps = trk.graph_steps()
    finally:
        trk.close()
        ctx.close()
    return out, graph_steps, order


def test_tracker_modes_and_switching(ofb200, monkeypatch):
    """graph / plain / kept / split / nosplit: the standard records equal a tracker without the robust solve, the robust
    records are one set in every mode, and switching it on mid-run gives the records of a tracker built with it on"""
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
                assert got[j][1].tobytes() == full[j][1].tobytes(), (mode, j)
    got, graph_steps, _ = run_modes(ofb200, kw, frames, imus, "graph", monkeypatch, {}, True)
    assert graph_steps >= 6
    assert all(got[j][1].tobytes() == full[j][1].tobytes() for j in range(len(order)))
    # a new setting while on also reaches the replayed graphs
    monkeypatch.setenv("OFB_TRACKER_GRAPH", "1")
    c2 = ofb200.Context(0)
    a = ofb200.StreamTracker(tc.W, tc.H, ctx=c2, robust=True, **kw)
    b = ofb200.StreamTracker(tc.W, tc.H, ctx=c2, robust=(2.0, 3), **kw)
    try:
        for j, k in enumerate(order):
            if j == 7:
                a.set_robust((2.0, 3))
            ra = a.step(frames[k], imu_records(ofb200, [imus[k]]), want_robust=True)
            rb = b.step(frames[k], imu_records(ofb200, [imus[k]]), want_robust=True)
            if j >= 7:
                assert ra[1].tobytes() == rb[1].tobytes(), j
        assert a.graph_steps() >= 4
    finally:
        a.close()
        b.close()
        c2.close()


# ---- errors -----------------------------------------------------------------------------------------------------
def test_errors_leave_the_context_usable(ofb200, ctx):
    x, u, d, n, w, t = flow_scene(60, 0.5)
    L = ofb200._lib
    rec = np.zeros(1, L.ROBUST_RESULT_DTYPE)
    good = L.RobustCfg(4.0, 10)

    def call(variant=0, cfg=good, xp=x):
        return L.check(ctx.lib.ofb_solve_velocity_robust(ctx.h, variant, L.ptr(xp), L.ptr(u), len(x), d, L.ptr(n), L.ptr(w),
                                                         None, C.byref(cfg) if cfg is not None else None, L.ptr(rec), None))
    for bad in (dict(variant=L.VARIANT_MODULE), dict(cfg=None), dict(cfg=L.RobustCfg(1.4, 10)),
                dict(cfg=L.RobustCfg(float("nan"), 10)), dict(cfg=L.RobustCfg(float("inf"), 10)), dict(cfg=L.RobustCfg(4.0, 65)),
                dict(cfg=L.RobustCfg(4.0, -1)), dict(xp=None)):
        with pytest.raises(ValueError):
            call(**bad)
    with pytest.raises(ValueError):
        L.check(ctx.lib.ofb_solve_velocity_robust_batched(ctx.h, 0, L.ptr(x), L.ptr(u), L.ptr(np.array([0, 5, 2], np.int32)), 2,
                                                          L.ptr(np.ones(2)), L.ptr(np.tile(n, 2)), L.ptr(np.tile(w, 2)), None,
                                                          C.byref(good), L.ptr(np.zeros(2, L.ROBUST_RESULT_DTYPE)), None))
    prev, nxt, imu, f, dt, _ = pair_batch(ofb200, n=1)
    hh, ww = prev.shape[1:]
    cfg = ofb200.make_pair_cfg(ww, hh, 50, variant="node", pos_scale=1 / f, flow_scale=1 / (f * dt))
    with pytest.raises(ValueError):                         # robust records without a setting
        L.check(ctx.lib.ofb_frame_pairs_robust(ctx.h, C.byref(cfg), None, 0.0, 0, 1, L.ptr(prev), L.ptr(nxt), ww, ww * hh,
                                               L.ptr(imu), None, None, L.ptr(np.zeros(1, L.RESULT_DTYPE)), None, None,
                                               L.ptr(np.zeros(1, L.ROBUST_RESULT_DTYPE)), None, None, None))
    with pytest.raises(ValueError):
        ofb200.frame_pairs(prev, nxt, imu, cfg, ctx=ctx, robust=(1.0, 3))
    frames, imus, kw = tc.build("exp")
    trk = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, **kw)
    mod = ofb200.StreamTracker(tc.W, tc.H, ctx=ctx, **dict(kw, variant="module"))
    try:
        with pytest.raises(ValueError):
            trk.step(frames[0][0], imu_records(ofb200, [imus[0][0]]), want_robust=True)
        with pytest.raises(ValueError):
            L.check(ctx.lib.ofb_tracker_step_robust(trk.h, L.ptr(frames[0][0]), tc.W, tc.W * tc.H,
                                                    L.ptr(imu_records(ofb200, [imus[0][0]])), None,
                                                    L.ptr(np.zeros(1, L.TRACK_RESULT_DTYPE)), None, None, None, None, None,
                                                    L.ptr(rec)))
        with pytest.raises(ValueError):
            mod.set_robust(True)
        with pytest.raises(ValueError):
            trk.set_robust((4.0, 65))
        with pytest.raises(ValueError):
            L.check(ctx.lib.ofb_tracker_set_robust(trk.h, C.byref(L.RobustCfg(0.5, 3))))
        assert trk.robust is None
    finally:
        trk.close()
        mod.close()
    rec2 = ofb200.solve_velocity_robust(x, u, d, n, w, t, variant="sim", ctx=ctx)
    check_against_oracle(rec2, x, u, d, n, w, t, "sim")
