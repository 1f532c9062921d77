"""GPU parity for the pieces added in round 2, all through the C ABI:
  * solve variant MODULE -- the inline system of optical_flow_experiments/of_module.py:136-146 -- against the
    reference's own statements (golden) and inside the tracker's "module" mode;
  * the time-evolution sweep (simulation.py:472-501): device-side trajectory vs the reference's, statistics vs the
    reference's of_simulation on the traced points;
  * the sorting study (simulation.py:604-894), live section 753-779 against the reference run;
  * detector overflow reported by ofb_frame_pairs; contexts on two devices in one process; the r_tilde gate without
    a prior; offset validation of the batched solve."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import velocity_oracle as vo
import synth

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4


@pytest.fixture(scope="module")
def g2():
    return np.load(os.path.join(GOLDEN, "velocity_golden_r2.npz"))


def relerr(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300)


# ---- variant MODULE ---------------------------------------------------------------------------------------------
def test_module_variant_against_reference_statements(ctx, g2):
    import ofb200
    worst = 0.0
    for c in range(int(g2["module_n_cases"])):
        k = lambda s: g2["module%d_%s" % (c, s)]
        # distances given (the reference's feasible_dist) ...
        v, res, rank, s = ofb200.solve_lgs_module(k("x"), k("u"), k("n"), dist=k("dist"), ctx=ctx)
        worst = max(worst, relerr(v, k("v")))
        assert rank == int(k("rank"))
        np.testing.assert_allclose(s, k("s"), rtol=1e-8)
        assert res.shape == k("res").shape
        if res.size:
            np.testing.assert_allclose(res, k("res"), rtol=1e-5, atol=1e-16)
        # ... and derived on the device from the prior velocity, as the 4-argument r_tilde does (of_module.py:125)
        v2, _, _, _ = ofb200.solve_lgs_module(k("x"), k("u"), k("n"), v_prior=k("v_prior"), ctx=ctx)
        worst = max(worst, relerr(v2, k("v")))
        # (N,2) rows are the same problem
        v3, _, _, _ = ofb200.solve_lgs_module(k("x")[:, :2], k("u")[:, :2], k("n"), dist=k("dist"), ctx=ctx)
        assert np.array_equal(v3, v)
    assert worst <= REL_TOL, worst
    with pytest.raises(ValueError):
        ofb200.solve_lgs_module(g2["module0_x"], g2["module0_u"], g2["module0_n"], ctx=ctx)


def test_tracker_module_mode_solves_the_module_system(ctx):
    """StreamTracker(variant="module", gate=("ge", T)): the kept (old, new) pairs of a step, pushed through the oracle's
    restatement of of_module.py:125-146 (4-argument r_tilde distances from the prior, per-point-distance lstsq), give
    the tracker's velocity."""
    import ofb200
    h, w = 240, 320
    a, b, mo = synth.make_pair(h, w, 3, 5, max_disp=4.0)
    imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
    ps, fs = 1.0 / mo["f"], 1.0 / (mo["f"] * mo["dt"])
    v_prior = np.asarray(mo["v"], dtype=np.float64) * 1.1 + 0.01
    trk = ofb200.StreamTracker(w, h, max_features=60, min_features=10, topup="module", variant="module", gate=("ge", -2.0),
                               principal=(mo["cx"], mo["cy"]), scaling=ps, flow_scaling=fs, min_solve=4, ctx=ctx)
    trk.step(a, imu)
    r, kp, kn = trk.step(b, imu, v_prior=v_prior[None], want_kept=True)
    trk.close()
    assert r["flags"][0] & 1 and r["n_kept"][0] >= 20
    x = (kn[0].astype(np.float64) - np.array([mo["cx"], mo["cy"]])) * ps
    u = (kn[0] - kp[0]).astype(np.float64) * fs
    xh = np.hstack([x, np.ones((len(x), 1))]); uh = np.hstack([u, np.zeros((len(u), 1))])
    _, dist = vo.r_tilde(xh, uh, mo["n"], v_prior)
    v_ref, _, rank, _ = vo.solve_lgs_module(xh, uh, mo["n"], dist)
    assert rank == 3
    assert relerr(r["v"][0], v_ref) <= REL_TOL, (r["v"][0], v_ref)


# ---- time-evolution sweep ---------------------------------------------------------------------------------------
def test_time_evolution_trajectory_on_device(ctx, g2):
    import ofb200
    sim = ofb200.simulation
    pos, flow, hs = sim.advect_points(g2["te_pos"][0], [1, 1, 1], [1, 1, 1], 1.0, [0, 0, 1], [0.02, 0, 0.205], 100, ctx=ctx)
    np.testing.assert_allclose(hs, g2["te_heights"], rtol=0, atol=0)
    np.testing.assert_allclose(pos, g2["te_pos"], rtol=1e-11, atol=1e-8)
    for s in (0, 13, 99):
        np.testing.assert_allclose(flow[s], vo.generate_test_data(pos[s], [1, 1, 1], [1, 1, 1], hs[s], [0, 0, 1], [0.02, 0, 0.205]),
                                   rtol=1e-11, atol=1e-12)


def test_time_evolution_sweep_statistics(ctx, g2, points200):
    """build_sweep("time_evolution") = simulation.py:472-501; per-step statistics within the SURVEY 8d bands of the
    reference's own of_simulation (400 trials, golden) on the same traced points."""
    import ofb200
    sim = ofb200.simulation
    steps, pos, flow = sim.build_sweep("time_evolution", points200)
    assert len(steps) == 100 and pos.shape == (100 * 200, 2)
    np.testing.assert_allclose(pos.reshape(100, 200, 2), g2["te_pos"], rtol=1e-11, atol=1e-8)
    assert [s.height for s in steps] == list(g2["te_heights"])
    n_ref = int(g2["te_ref_trials"])
    mean, std, mR, n = sim.run_sweep(steps, pos, flow, 20_000, seed=4, precision="fp64", ctx=ctx)
    for s in (0, 7, 60):
        rm, rs = g2["te_ref_mean_%d" % s], g2["te_ref_std_%d" % s]
        assert np.all(np.abs(mean[s] - rm) <= 4 * rs / np.sqrt(n_ref)), (s, mean[s], rm, rs)
        assert np.all(np.abs(std[s] / rs - 1) <= 4 / np.sqrt(2 * n_ref)), (s, std[s], rs)
    flat, _ = sim.run_named_sweep("time_evolution", points200, trials=200, seed=1, ctx=ctx)
    assert flat.shape == (600,)


# ---- sorting study ----------------------------------------------------------------------------------------------
def test_sorting_live_section_against_reference_run(ctx, g2, points200):
    """simulation.py:753-779, the reference's only live section. Same RandomState seed => the same rotation angles, so
    the scenario is the reference's to rounding; the six per-point means agree within the reference's own
    seed-to-seed scatter (two golden runs of 300 trials), and the two printed fractions are reproduced."""
    import ofb200
    sim = ofb200.simulation
    rng = np.random.RandomState(int(g2["live_seed"]))
    sc = sim.sorting_scenario("moving_and_plane", points200, minang=float(g2["live_minang"]), rng=rng)
    np.testing.assert_allclose(sc["data"], g2["live_data"], atol=1e-13)
    np.testing.assert_allclose(sc["true_flow"], g2["live_true_flow"], rtol=1e-10, atol=1e-11)
    np.testing.assert_allclose(sc["linear_velocity"], g2["live_velocity"], rtol=1e-15)
    out = sim.sorting_study("moving_and_plane", points200, iterations=20_000, seed=int(g2["live_seed"]),
                            minang=float(g2["live_minang"]), ctx=ctx)
    third = 66
    for m in sim.METRICS:
        ra, rb = g2["live_%s_a" % m], g2["live_%s_b" % m]
        # groups 0 and 2 (static points) share their flow field between the two reference seeds: their difference is
        # the reference's sampling noise at 300 trials; the GPU mean (20000 trials) must sit within 5 sigma of run a
        # (medians: the distance metrics are ratios with heavy tails). Expected ratio of the two medians: 0.71.
        stat = np.r_[0:40, 132:200]
        dev = np.abs(out[m][stat] - ra[stat])
        assert np.median(dev) <= 2.0 * np.median(np.abs(ra[stat] - rb[stat])) + 1e-12, (m, np.median(dev))
        # the moving points' values are set by their rotation angles (identical here: same seed), not by the noise
        mov = slice(40, 132)
        assert np.corrcoef(out[m][mov], ra[mov])[0, 1] >= 0.9, m
    ref_fwd = np.sum(g2["live_forward_para_a"][third:2 * third] > 0.88) / float(third)
    ref_bwd = np.sum(g2["live_backward_para_a"][third:2 * third] > 0.88) / float(third)
    assert abs(out["sorted_out_forward"] - ref_fwd) <= 0.08 and abs(out["sorted_out_backward"] - ref_bwd) <= 0.08
    # Python-2 default: minang = 0 (10/360 is integer division in the interpreter the reference ran under)
    sc0 = sim.sorting_scenario("moving_and_plane", points200)
    assert sc0["true_flow"].shape == (200, 2) and set(sc0["groups"]) == {"static_2m", "moving_1m", "static_1m"}


def test_sorting_other_scenarios(ctx, points200):
    import ofb200
    sim = ofb200.simulation
    out = sim.sorting_study("planes", points200, iterations=2000, seed=3, ctx=ctx)
    # three planes at 3, 2, 1 m, forward distance metric clusters around the true plane heights (simulation.py:630-639)
    fd, gs = out["forward_dist"], out["groups"]
    med = [float(np.median(fd[gs[k]])) for k in ("3m", "2m", "1m")]
    assert med[0] > med[1] > med[2] > 0 and abs(med[0] / med[2] - 3.0) < 0.5
    assert np.all(np.diff(out["sorted_distance"]) >= 0) and len(out["distance_diff"]) == 199
    out = sim.sorting_study("moving", points200, iterations=2000, seed=3, ctx=ctx)
    st, mv = out["forward_para"][out["groups"]["static"]], out["forward_para"][out["groups"]["moving"]]
    assert np.median(st) > 0.95 and np.median(mv) < np.median(st)
    cur = sim.sorting_study("dynamic", points200, iterations=100, seed=5, k=6, ctx=ctx)
    assert set(cur) == {"%s_overlap_%s" % (g, m) for g in ("mov", "plane") for m in sim.METRICS} | {"velocity_scale"}
    assert cur["mov_overlap_forward_para"].shape == (6,)
    for name, c in cur.items():                 # an overlap is a count of histogram entries of the smaller group
        if name != "velocity_scale":
            assert np.all(c >= 0) and np.all(c <= 67), (name, c)
    # host restatement of simulation.py:124-136 on the same per-point means (the curve itself is overlap of those)
    sc = sim.sorting_scenario("dynamic", points200, rng=np.random.RandomState(5), velocity_scale=0.0)
    assert np.allclose(sc["linear_velocity"], 0.0) and sc["height"] == 1.0
    lit = sim.sorting_study("dynamic", points200, iterations=50, seed=5, k=3, cumulative=True, ctx=ctx)
    assert np.all(np.isfinite(lit["plane_overlap_backward_dist"]))


# ---- correctness hazards of round 1 -----------------------------------------------------------------------------
def test_frame_pairs_reports_detector_overflow(ctx):
    """A checkerboard of 2x2 blocks seen through a 4x4 window (one period) is one big lambda_min plateau: the exact
    integer window sums are identical at every interior pixel, so every pixel is a 3x3 local maximum above the quality
    threshold -- 75 k candidates (cv2 agrees) against the w*h/4 + 1024 = 20 k slots of ofb_frame_pairs. The pair must
    say so."""
    import ofb200
    h, w = 240, 320
    yy, xx = np.mgrid[0:h, 0:w]
    a = ((((xx >> 1) + (yy >> 1)) & 1) * 200 + 20).astype(np.uint8)
    imu = np.zeros(1, ofb200._lib.IMU_DTYPE); imu["d"], imu["n"] = 1.0, [0, 0, 1]
    cfg = ofb200.make_pair_cfg(w, h, 100, quality=0.01, min_distance=10, block_size=4, max_level=2, pos_scale=0.01, flow_scale=0.01)
    res = ofb200.frame_pairs(a[None], a[None], imu, cfg, ctx=ctx, on_overflow="ignore")
    assert res["flags"][0] & ofb200._lib.PAIR_OVERFLOW
    with pytest.raises(ofb200.OfbError):
        ofb200.frame_pairs(a[None], a[None], imu, cfg, ctx=ctx)
    # the single-image entry point already refused such an image (it sizes its list for every pixel, so here: fine)
    pts = ofb200.goodFeaturesToTrack(a, 100, 0.01, 10, blockSize=4, ctx=ctx)
    assert pts is not None and len(pts) == 100
    # a textured frame does not raise the flag
    b, c, mo = synth.make_pair(h, w, 0, 0, max_disp=3.0)
    res = ofb200.frame_pairs(b[None], c[None], imu, cfg, ctx=ctx)
    assert res["flags"][0] == 0 and res["n_features"][0] > 50


def test_contexts_on_two_devices_in_one_process():
    """cudaFuncAttributeMaxDynamicSharedMemorySize is per device: the > 48 KB kernels (lambda_min marching kernel,
    1024-thread selection, generic LK) must launch on a second device of the same process."""
    import torch
    import ofb200
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    a, b, mo = synth.make_pair(240, 320, 1, 2, max_disp=3.0)
    outs = []
    for dev in (0, 1):
        c = ofb200.Context(dev)
        pts = ofb200.goodFeaturesToTrack(a, 600, 0.01, 5, blockSize=7, ctx=c)              # march kernel + select<1024>
        nxt, st, err = ofb200.calcOpticalFlowPyrLK(a, b, pts, None, winSize=(21, 21), maxLevel=2, ctx=c)   # generic LK (smem)
        e = ofb200.cornerMinEigenVal(a, 5, ctx=c)                                            # tile kernel
        outs.append((pts, nxt, st, e))
        c.close()
    for x, y in zip(outs[0], outs[1]):
        assert np.array_equal(x, y)


def test_r_tilde_gate_without_prior(ctx):
    """ADVICE r1: with gate=("le", T<1) and no prior velocity r_tilde is 1 for every point, which used to drop all points
    forever. No prior => no gate; v_init (node:183) provides one."""
    import ofb200
    h, w = 240, 320
    a, b, mo = synth.make_pair(h, w, 2, 9, max_disp=4.0)
    imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
    kw = dict(max_features=80, min_features=10, topup="node", variant="node", gate=("le", 0.0), principal=(mo["cx"], mo["cy"]),
              scaling=1.0 / mo["f"], flow_scaling=1.0 / (mo["f"] * mo["dt"]), ctx=ctx)
    trk = ofb200.StreamTracker(w, h, **kw)
    trk.step(a, imu)
    r = trk.step(b, imu)
    assert r["n_kept"][0] == r["n_tracked"][0] > 20 and r["flags"][0] & 1        # gate skipped, velocity solved
    r2 = trk.step(a, imu)                                                        # now the solved velocity is the prior
    assert r2["n_kept"][0] <= r2["n_tracked"][0]
    trk.close()
    # a seeded prior gates from the first tracked frame on: the reference's convention r = -1 for consistent points
    trk = ofb200.StreamTracker(w, h, v_init=mo["v"], **kw)
    trk.step(a, imu)
    r, kp, kn = trk.step(b, imu, want_kept=True)
    x = (kn[0].astype(np.float64) - np.array([mo["cx"], mo["cy"]])) / mo["f"]
    u = (kn[0] - kp[0]).astype(np.float64) / (mo["f"] * mo["dt"])
    rr, _ = vo.r_tilde(x, u, mo["n"], mo["v"], mo["d"])
    assert np.all(rr <= 0.0) and 0 < r["n_kept"][0] <= r["n_tracked"][0]
    trk.close()


def test_batched_solve_rejects_bad_offsets(ctx):
    import ofb200
    x = np.random.default_rng(0).uniform(-0.5, 0.5, (10, 2)); u = x * 0.1
    for off in ([0, 6, 4, 10], [-1, 5, 10], [0, 5, 12]):
        with pytest.raises(ValueError):
            ofb200.solve_lgs_batched(x, u, off, 1.0, [0, 0, 1], [0, 0, 0], ctx=ctx)
    import ctypes as C
    lib = ctx.lib
    offs = np.array([0, 6, 4, 10], np.int32); d = np.ones(3); n3 = np.tile([0.0, 0, 1], (3, 1)); w3 = np.zeros((3, 3)); v = np.zeros((3, 3))
    rc = lib.ofb_solve_velocity_batched(ctx.h, 0, ofb200._lib.ptr(x), ofb200._lib.ptr(u), ofb200._lib.ptr(offs), 3, ofb200._lib.ptr(d),
                                        ofb200._lib.ptr(n3), ofb200._lib.ptr(w3), None, ofb200._lib.ptr(v), None, None, None)
    assert rc == ofb200._lib.OFB_E_INVALID and b"non-decreasing" in lib.ofb_last_error()


def test_mc_sweep_over_several_contexts_of_one_process(ctx, points200):
    """ofb_mc_sweep_multi: the library shards the trial range over the contexts it is given and merges the sums itself
    (no torch.distributed). Two contexts on one device, and -- where the box has them -- one context per device, must
    reproduce the one-context sums up to fp64 summation order; uneven and tiny trial counts included."""
    import torch
    import ofb200
    sim = ofb200.simulation
    steps, pos, flow = sim.build_sweep("flow_errors", points200[:50], k=7)
    extra = [ofb200.Context(0), ofb200.Context(0)]
    if torch.cuda.device_count() >= 2:
        extra.append(ofb200.Context(1))
    try:
        for trials in (1, 2, 1001, 40_000):
            whole = sim.run_steps(steps, pos, flow, trials, seed=5, trial_begin=77, ctx=ctx)
            for group in ([ctx], [ctx, extra[0]], [ctx] + extra):
                got = sim.run_steps_multi(steps, pos, flow, trials, group, seed=5, trial_begin=77)
                assert np.array_equal(got["n"], whole["n"])
                np.testing.assert_allclose(got.view(np.float64), whole.view(np.float64), rtol=1e-10, atol=1e-9)
        again = sim.run_steps_multi(steps, pos, flow, 40_000, [ctx] + extra, seed=5, trial_begin=77)
        assert np.array_equal(again.view(np.float64), got.view(np.float64))          # fixed merge order: bit-reproducible
    finally:
        for c in extra:
            c.close()


@pytest.mark.parametrize("shape", [(4, 4), (5, 7), (33, 37), (64, 128), (67, 131), (240, 320), (241, 323), (480, 640), (720, 1280)])
def test_bgr_fused_pyramid_is_bit_exact(ctx, shape):
    """ofb_pyramid_bgr: grey level 0 = cv2's BGR2GRAY rule (oracle), every level = pyrDown of the one below, for tile-
    aligned, odd, tiny and multi-image inputs, unaligned row pitches included (widths that are not multiples of 16)."""
    import ofb200
    from oracle import image_oracle as io
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    frames = rng.integers(0, 256, (3,) + shape + (3,), dtype=np.uint8)
    frames[1, :, :, :] = rng.integers(0, 256, shape + (1,), dtype=np.uint8)          # a grey-valued colour frame
    p = ofb200.Pyramid(frames, 4, ctx=ctx, bgr=True)
    try:
        for i in range(3):
            ref = io.build_pyramid(io.bgr2gray(frames[i]), p.n_levels - 1)
            for l in range(p.n_levels):
                got = p.level(l, i)
                assert got.shape == ref[l].shape and np.array_equal(got, ref[l]), (shape, i, l, np.argwhere(got != ref[l])[:4])
    finally:
        p.close()
    p0 = ofb200.Pyramid(frames[0], 0, ctx=ctx, bgr=True)            # no level 1: plain conversion path
    assert np.array_equal(p0.level(0), io.bgr2gray(frames[0]))
    p0.close()


def test_tracker_bgr_fused_equals_separate_conversion(ctx):
    """The lifecycle on BGR frames: fused conversion + first pyramid step vs the separate conversion kernel
    (OFB_BGR_FUSED=0) vs grey frames converted beforehand -- identical records, points and velocities."""
    import ofb200
    h, w = 240, 320
    a, b, mo = synth.make_pair(h, w, 4, 11, max_disp=4.0)
    rng = np.random.default_rng(3)
    tint = rng.integers(0, 40, (h, w, 3), dtype=np.uint8)
    to_bgr = lambda g: np.clip(np.stack([g, g, g], -1).astype(np.int32) + tint - 20, 0, 255).astype(np.uint8)
    A, B = to_bgr(a), to_bgr(b)
    from oracle import image_oracle as io
    ga, gb = io.bgr2gray(A), io.bgr2gray(B)
    imu = np.zeros(1, ofb200._lib.IMU_DTYPE)
    imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
    kw = dict(max_features=120, min_features=118, topup="node", mask_radius=12, variant="node", principal=(mo["cx"], mo["cy"]),
              scaling=1.0 / mo["f"], flow_scaling=1.0 / (mo["f"] * mo["dt"]), ctx=ctx)

    def run(frames, bgr, env=None):
        if env is not None:
            os.environ["OFB_BGR_FUSED"] = env
        try:
            trk = ofb200.StreamTracker(w, h, bgr=bgr, **kw)
            out = [trk.step(f, imu, want_points=True) for f in frames]
            trk.close()
            return out
        finally:
            os.environ.pop("OFB_BGR_FUSED", None)
    fused = run([A, B, A, B], True)
    separate = run([A, B, A, B], True, env="0")
    grey = run([ga, gb, ga, gb], False)
    for x, y, z in zip(fused, separate, grey):
        for f in ("v", "n_tracked", "n_kept", "n_added", "n_points", "flags"):
            assert np.array_equal(x[0][f], y[0][f]) and np.array_equal(x[0][f], z[0][f]), f
        assert np.array_equal(x[1][0], y[1][0]) and np.array_equal(x[1][0], z[1][0])


def test_tracker_stream_overlap_modes_are_identical(ctx):
    """ofb_tracker_step with device-resident frames / IMU / result records runs the ingest + pyramid on its own stream, the
    fp64 solve on another one beside the next frame's LK. That is scheduling only: the records of every step and the final point sets must equal the single-stream schedule
    (OFB_TRACKER_EARLY_PYR=0), with frequent top-ups (min_features close to max_features), for one stream and a small fleet."""
    import torch
    import ofb200
    P = ofb200._lib.ptr
    h, w = 240, 320
    for S in (1, 3):
        seqs = []
        for s in range(S):
            a, b, mo = synth.make_pair(h, w, s, 5 + s, max_disp=5.0)
            seqs.append((a, b, mo))
        mo = seqs[0][2]
        imu = np.zeros(S, ofb200._lib.IMU_DTYPE)
        for s in range(S):
            imu["d"][s], imu["n"][s], imu["w"][s] = seqs[s][2]["d"], seqs[s][2]["n"], seqs[s][2]["w"]
        fa = torch.from_numpy(np.stack([q[0] for q in seqs])).cuda()
        fb = torch.from_numpy(np.stack([q[1] for q in seqs])).cuda()
        d_imu = torch.from_numpy(imu.view(np.uint8).reshape(-1).copy()).cuda()
        nsteps = 9
        rsz = ofb200._lib.TRACK_RESULT_DTYPE.itemsize
        kw = dict(max_features=150, min_features=140, n_streams=S, topup="node", mask_radius=10, variant="node",
                  principal=(mo["cx"], mo["cy"]), scaling=1.0 / mo["f"], flow_scaling=1.0 / (mo["f"] * mo["dt"]),
                  borrow_frames=True, ctx=ctx)

        def run(early, split="0"):
            os.environ["OFB_TRACKER_EARLY_PYR"] = early
            os.environ["OFB_TRACKER_SPLIT_SOLVE"] = split
            try:
                trk = ofb200.StreamTracker(w, h, **kw)
                d_res = torch.zeros(nsteps * S * rsz, dtype=torch.uint8, device="cuda")
                for k in range(nsteps):
                    f = fb if k & 1 else fa
                    ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, P(f), w, w * h, P(d_imu), None, d_res.data_ptr() + k * S * rsz,
                                                               None, None, None, None))
                # the last step through the host path: it must join whatever is still pending and return the point sets
                last, pts = trk.step((fb if nsteps & 1 else fa), imu, want_points=True)
                ctx.sync()
                res = np.zeros(nsteps * S, ofb200._lib.TRACK_RESULT_DTYPE)
                ctx.memcpy(res, d_res, res.nbytes)
                trk.close()
                return res, last, pts
            finally:
                os.environ.pop("OFB_TRACKER_EARLY_PYR", None); os.environ.pop("OFB_TRACKER_SPLIT_SOLVE", None)
        ref = run("0")
        assert ref[0]["n_added"].sum() > 0, "the case must exercise the top-up"
        # (split: the fp64 solve of a step on its own stream beside the next frame's LK, track_filter_solve_kernel<1> / <2>)
        for early, split in (("1", "0"), ("1", "1")):
            got = run(early, split)
            for f in ("v", "s", "res", "rank", "n_prev", "n_tracked", "n_kept", "n_added", "n_points", "flags"):
                assert np.array_equal(got[0][f], ref[0][f], equal_nan=True), (S, early, split, f)
                assert np.array_equal(got[1][f], ref[1][f], equal_nan=True), (S, early, split, f, "last")
            for s in range(S):
                assert np.array_equal(got[2][s], ref[2][s]), (S, early, split, s)
