"""GPU: the Monte-Carlo stage (csrc/montecarlo.cu) at the shapes and edges where its kernels can go wrong.

* every trial of mc_sweep_kernel against the oracle's of_trial on the replayed Philox stream, for point counts from 2
  to OFB_MC_MAX_POINTS (odd ones run the tail of the unroll-by-two point loop), a multi-step launch with overlapping
  point ranges and its own parameters per step, trial counts around one CTA, a trial range that crosses 2^32 and a
  seed wider than 32 bits, in fp32 and fp64, with and without the error bound R;
* launch-shape invariance past the grid caps of the sweep (16384 CTAs per step) and of the feasibility kernel
  (8 CTAs per SM), where every thread runs several trials;
* mc_feas_kernel per trial for point counts below and above a warp, where every lane of a warp adds into the same
  shared per-point sums;
* ofb_minmax / ofb_histogram / overlap against NumPy on samples that sit exactly on the bin edges, quantised data,
  1..4096 bins, a degenerate range and non-finite input;
* one-point steps are rejected: their 3x3 normal matrix is singular by construction.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import velocity_oracle as vo

pytestmark = pytest.mark.gpu

V, W, T3 = np.ones(3), np.ones(3), np.array([0.02, 0, 0.205])
NRM = np.array([0.1, -0.05, 1.0])                  # not unit length: n and n/|n| both enter a trial
SIG = dict(ang_vel_sig=0.00071, translation_sig=0.005, height_sig=0.01, flow_sig=0.056 * np.sqrt(2) * 1.23,
           position_sig=0.056 * 1.23)
U = {"fp32": 2.0 ** -24, "fp64": 2.0 ** -53}       # unit roundoff of the trial arithmetic
BASE = {"fp32": 5e-4, "fp64": 1e-8}                # relative bars of test_gpu_pairs_mc at 50 points
BIG_SEED = (0x9E3779B97F4A7C15 >> 3) | (1 << 40)   # both 32-bit key words non-zero


def _prm(v=V, w=W, h=1.3, n=NRM, t=T3, **sig):
    s = dict(SIG)
    s.update(sig)
    return dict(v=np.asarray(v, float), w=np.asarray(w, float), h=float(h), n=np.asarray(n, float),
                t=np.asarray(t, float), **s)


def _step(prm, n_points, pos_offset):
    import ofb200
    return ofb200.simulation.make_step(prm["v"], prm["w"], prm["h"], prm["n"], prm["t"], n_points, pos_offset,
                                       prm["ang_vel_sig"], prm["translation_sig"], prm["height_sig"], prm["flow_sig"],
                                       prm["position_sig"], 0.0)


@pytest.fixture(scope="module")
def pool(points200):
    """300 image points: the 200 centred reference points, then 100 uniform ones over the same box; the flow of the
    truth (V, W, h = 1.3, NRM, T3) at every point."""
    import ofb200
    c = ofb200.simulation.centred_points(points200)
    extra = np.random.default_rng(17).uniform(c.min(0), c.max(0), size=(100, 2))
    pos = np.vstack([c, extra])
    return pos, vo.generate_test_data(pos, V, W, 1.3, NRM, T3)


# ---- per-trial reference and its error bound --------------------------------------------------------------------
def replay(prm, pos, tf, seed, step_id, trial_ids):
    """of_trial on the replayed draws of every trial id, and the two per-trial amplification factors of the
    tolerance (see `tolerances`). -> dict of arrays v (K,3), R (K,), amp_v (K,), amp_R (K,), cond (K,)."""
    N = len(pos)
    z = vo.mc_normals(seed, step_id, np.asarray(trial_ids, np.uint64), N)
    n_err = prm["n"] / np.linalg.norm(prm["n"])
    out = {k: [] for k in ("v", "R", "amp_v", "amp_R", "cond")}
    for k in range(len(trial_ids)):
        d_w, d_t = prm["ang_vel_sig"] * z[k, 0, :3], prm["translation_sig"] * z[k, 1, :3]
        d_h = prm["height_sig"] * z[k, 0, 3]
        d_f, d_p = prm["flow_sig"] * z[k, 3:, 0:2], prm["position_sig"] * z[k, 3:, 2:4]
        v, R = vo.of_trial(prm["v"], prm["w"], prm["h"], prm["n"], prm["t"], pos, tf, prm["ang_vel_sig"],
                           prm["translation_sig"], d_w, d_t, d_h, d_f, d_p)
        w_e, t_e, h_e = prm["w"] + d_w, prm["t"] + d_t, prm["h"] + d_h
        A, B = vo.build_system(pos + d_p, tf + d_f, n_err, w_e, "sim")
        lam = np.linalg.eigvalsh(A.T @ A)                       # ascending; M = A^T A is what the kernel forms
        v_hat = (v + np.cross(w_e, t_e)) / h_e                  # the solution of M v_hat = A^T B
        SM = np.linalg.norm(np.abs(A).T @ np.abs(A), 2)
        Sg = np.linalg.norm(np.abs(A).T @ np.abs(B))
        out["v"].append(v); out["R"].append(R)
        out["amp_v"].append(abs(h_e) * (SM * np.linalg.norm(v_hat) + Sg) / lam[0])
        out["amp_R"].append(1.0 + SM / lam[0])
        out["cond"].append(lam[-1] / lam[0])
    return {k: np.array(a) for k, a in out.items()}


def tolerances(ref, n_points, precision):
    """Per-trial bounds on |v_gpu - v_ref|_inf (absolute) and |R_gpu - R_ref| / R_ref.

    The kernel sums M = sum_i A_i^T A_i and g = sum_i A_i^T B_i over the N points in the trial precision T (unit
    roundoff u), from inputs rounded to T, then solves M v_hat = g in fp64; v_obs = h_e v_hat - w_e x t_e. A sum of N
    terms that each carry a few roundings is off by at most gamma = (N + c) u times the sum of the magnitudes of its
    terms (Higham, "Accuracy and Stability of Numerical Algorithms", 2nd ed., sec. 3.1), so elementwise
    |dM| <= gamma S_M and |dg| <= gamma S_g with S_M = sum |A_i|^T |A_i|, S_g = sum |A_i|^T |B_i|. To first order
    dv_hat = M^-1 (dg - dM v_hat), hence
        |dv_obs| <= |h_e| gamma (||S_M|| ||v_hat|| + ||S_g||) / lambda_min(M)  =  gamma amp_v,
    which is cond(M) gamma |v_obs| when the residual is small (||S_M|| = ||M|| when the signs agree). R divides by
    lambda_min(M), whose error is at most ||dM|| <= gamma ||S_M||, and sums N squares:
        |dR| / R <= gamma (1 + ||S_M|| / lambda_min)  =  gamma amp_R.
    c = 16 covers the rounding of the inputs to T and of the noise draws: the fp64 draws are within an ulp, the fp32
    ones use the SFU logarithm, square root and sine/cosine, ~2^-21 absolute on a standard normal, i.e. a few u of a
    point coordinate of the ~0.3 typical here. Where cond(M) is moderate the bound is below the fixed relative bars
    the 50-point test uses (5e-4 fp32, 1e-8 fp64), and those stay the floor.
    Measured on a B200 (1000 W power limit), 2..256 points: the v errors reach at most 2 % of gamma amp_v in fp32 and
    23 % in fp64; fp32 stays within 2e-6 relative wherever cond(M) < 100, and reaches 1.2e-3 (about cond(M) u, above
    the fixed 5e-4) for two clustered points with cond(M) = 2e4."""
    gamma = (n_points + 16) * U[precision]
    tol_v = np.maximum(BASE[precision] * np.maximum(1.0, np.abs(ref["v"]).max(1)), gamma * ref["amp_v"])
    tol_R = np.maximum(max(BASE[precision], 1e-6), gamma * ref["amp_R"])
    return tol_v, tol_R


def check_trials(vd, Rd, ref, n_points, precision, want_R, what):
    tol_v, tol_R = tolerances(ref, n_points, precision)
    err_v = np.abs(vd - ref["v"]).max(1)
    bad = np.flatnonzero(~(err_v <= tol_v))
    assert bad.size == 0, (what, precision, want_R, bad[:5], err_v[bad[:5]], tol_v[bad[:5]], ref["cond"][bad[:5]])
    if want_R:
        err_R = np.abs(Rd - ref["R"]) / ref["R"]
        bad = np.flatnonzero(~(err_R <= tol_R))
        assert bad.size == 0, (what, precision, bad[:5], err_R[bad[:5]], tol_R[bad[:5]], ref["cond"][bad[:5]])
    else:
        assert np.all(Rd == 0), what


def check_sums(sums, vd, Rd, v_true, trials):
    """The per-step sums are the sums of that step's dumped trials."""
    assert sums["n"] == trials
    np.testing.assert_allclose(sums["sum_dv"], (vd - v_true).sum(0), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(sums["sum_dv2"], ((vd - v_true) ** 2).sum(0), rtol=1e-9)
    np.testing.assert_allclose(sums["sum_R"], Rd.sum(), rtol=1e-9, atol=1e-300)


VARIANTS = [(p, r) for p in ("fp32", "fp64") for r in (True, False)]


@pytest.mark.parametrize("n_points", [2, 3, 4, 31, 33, 50, 51, 255, 256])
def test_mc_per_trial_parity_point_counts(ctx, pool, n_points):
    import ofb200
    sim = ofb200.simulation
    pos, tf = pool[0][:n_points], pool[1][:n_points]
    prm = _prm()
    seed, sid, t0, ntr = 31337 + n_points, 7, 123_456_789, 24
    ref = replay(prm, pos, tf, seed, sid, t0 + np.arange(ntr))
    for precision, want_R in VARIANTS:
        sums, vd, Rd = sim.run_steps([_step(prm, n_points, 0)], pos, tf, ntr, seed=seed, step_id_base=sid,
                                     trial_begin=t0, precision=precision, dump=True, want_R=want_R, ctx=ctx)
        check_trials(vd[0], Rd[0], ref, n_points, precision, want_R, n_points)
        check_sums(sums[0], vd[0], Rd[0], prm["v"], ntr)


@pytest.mark.parametrize("n_points", [2, 3])
def test_mc_per_trial_parity_clustered_points(ctx, n_points):
    """Points within 0.02 of each other and little position noise: cond(M) ~ 1e4, where the fp32 bar is the
    cond(M)-scaled bound of `tolerances` rather than the fixed 5e-4."""
    import ofb200
    pos = np.array([0.3, -0.2]) + np.random.default_rng(1).uniform(-0.02, 0.02, (n_points, 2))
    tf = vo.generate_test_data(pos, V, W, 1.3, NRM, T3)
    prm = _prm(position_sig=1e-4, flow_sig=1e-3)
    seed, sid, ntr = 606, 1, 64
    ref = replay(prm, pos, tf, seed, sid, np.arange(ntr))
    assert ref["cond"].min() > 1e3
    for precision, want_R in VARIANTS:
        sums, vd, Rd = ofb200.simulation.run_steps([_step(prm, n_points, 0)], pos, tf, ntr, seed=seed, step_id_base=sid,
                                                   precision=precision, dump=True, want_R=want_R, ctx=ctx)
        check_trials(vd[0], Rd[0], ref, n_points, precision, want_R, n_points)


def test_mc_multi_step_layout(ctx, pool):
    """One launch, five steps with their own point counts, overlapping ranges of one point array, truth and sigmas:
    step s replays with step id step_id_base + s and dumps at (s * trials + k)."""
    import ofb200
    sim = ofb200.simulation
    pos, tf = pool
    layout = [  # (N, pos_offset, parameters)
        (3, 0, _prm()),
        (51, 1, _prm(v=(0.5, -1.0, 2.0), w=(0.3, -0.2, 0.1), h=2.5, flow_sig=0.02, position_sig=0.03)),
        (256, 10, _prm(v=(-1.0, 0.2, 0.7), n=(0.0, 0.2, 1.0), h=0.8, ang_vel_sig=0.01, height_sig=0.05)),
        (2, 40, _prm(v=(2.0, 1.0, -0.5), w=(0.0, 0.0, 0.5), t=(0.1, 0.05, 0.3), translation_sig=0.02)),
        (33, 250, _prm(w=(-1.0, 0.5, 0.2), h=4.0, n=(0.05, 0.0, 1.0), flow_sig=0.2, position_sig=0.01)),
    ]
    seed, base, t0, ntr = 99, 40, 5_000, 24
    steps = [_step(p, n, off) for n, off, p in layout]
    refs = [replay(p, pos[off:off + n], tf[off:off + n], seed, base + s, t0 + np.arange(ntr))
            for s, (n, off, p) in enumerate(layout)]
    for precision, want_R in VARIANTS:
        sums, vd, Rd = sim.run_steps(steps, pos, tf, ntr, seed=seed, step_id_base=base, trial_begin=t0,
                                     precision=precision, dump=True, want_R=want_R, ctx=ctx)
        assert vd.shape == (5, ntr, 3) and Rd.shape == (5, ntr)
        for s, (n, off, p) in enumerate(layout):
            check_trials(vd[s], Rd[s], refs[s], n, precision, want_R, ("step", s))
            check_sums(sums[s], vd[s], Rd[s], p["v"], ntr)


def test_mc_trial_counts_and_counter_words(ctx, pool):
    """Trial counts around one 128-thread CTA, a 64-bit seed, and a trial range whose high counter word changes
    inside the launch (2^32 - 60 .. 2^32 + 59)."""
    import ofb200
    sim = ofb200.simulation
    N = 31
    pos, tf = pool[0][50:50 + N], pool[1][50:50 + N]
    prm = _prm(h=1.7)
    step = _step(prm, N, 0)
    t0 = 3_000_000_000
    ref = replay(prm, pos, tf, BIG_SEED, 11, t0 + np.arange(129))
    for precision in ("fp32", "fp64"):
        for ntr in (1, 127, 128, 129):
            sums, vd, Rd = sim.run_steps([step], pos, tf, ntr, seed=BIG_SEED, step_id_base=11, trial_begin=t0,
                                         precision=precision, dump=True, ctx=ctx)
            sub = {k: a[:ntr] for k, a in ref.items()}
            check_trials(vd[0], Rd[0], sub, N, precision, True, ntr)
            check_sums(sums[0], vd[0], Rd[0], prm["v"], ntr)
    t_wrap = 2 ** 32 - 60
    ref = replay(prm, pos, tf, BIG_SEED, 12, t_wrap + np.arange(120, dtype=np.uint64))
    for precision in ("fp32", "fp64"):
        sums, vd, Rd = sim.run_steps([step], pos, tf, 120, seed=BIG_SEED, step_id_base=12, trial_begin=t_wrap,
                                     precision=precision, dump=True, ctx=ctx)
        check_trials(vd[0], Rd[0], ref, N, precision, True, "2^32")
        check_sums(sums[0], vd[0], Rd[0], prm["v"], 120)
    # the high key word is live: the same launch under the low word alone draws other noise
    other = sim.run_steps([step], pos, tf, 120, seed=BIG_SEED & 0xFFFFFFFF, step_id_base=12, trial_begin=t_wrap,
                          precision="fp64", dump=True, ctx=ctx)[1]
    assert np.abs(other[0] - vd[0]).max() > 1e-3


# ---- launch shape ---------------------------------------------------------------------------------------------------
def test_mc_sweep_past_the_grid_cap_equals_shards(ctx, pool):
    """9e6 trials of one step: the sweep grid is capped at 16384 CTAs x 128 threads, so every thread runs 4 or 5
    trials. The sums must equal those of three 3e6-trial shards (5860 CTAs, at most 4 trials per thread) up to fp64
    summation order, the bar of test_mc_sharding_is_exact_union."""
    import ofb200
    sim = ofb200.simulation
    pos, tf = pool[0][:50], pool[1][:50]
    step = _step(_prm(), 50, 0)
    total = 9_000_000
    assert total > 16384 * 128 * 4
    whole = sim.run_steps([step], pos, tf, total, seed=8, ctx=ctx)
    acc = np.zeros(8)
    for r in range(3):
        b, c = sim.shard_range(total, r, 3)
        assert c <= 16384 * 128 * 4
        acc += sim.run_steps([step], pos, tf, c, seed=8, trial_begin=b, ctx=ctx).view(np.float64)
    assert whole["n"][0] == total
    np.testing.assert_allclose(acc, whole.view(np.float64), rtol=1e-10, atol=1e-9)


def _feas(ofb200, pos, tf, trials, seed, sid, ctx, trial_begin=0):
    return ofb200.simulation.feas_simulation(V, W, 1.3, NRM, T3, pos, SIG["ang_vel_sig"], SIG["translation_sig"],
                                             SIG["height_sig"], SIG["flow_sig"], SIG["position_sig"], 0.0, V,
                                             iterations=trials, true_flow=tf, seed=seed, step_id=sid, normal_sig=0.3,
                                             velocity_sig=0.01, trial_begin=trial_begin, ctx=ctx, return_sums=True)


def test_mc_feas_past_the_grid_cap_equals_shards(ctx, pool):
    """More trials than the feasibility grid (8 CTAs per SM x 128 threads) holds: every thread runs several trials.
    The per-point sums equal those of shards that each fit in one pass of the grid."""
    import ofb200
    import torch
    one_pass = torch.cuda.get_device_properties(ctx.device).multi_processor_count * 8 * 128
    pos, tf = pool[0][:31], pool[1][:31]
    total = 3 * one_pass + 17
    whole = _feas(ofb200, pos, tf, total, 21, 4, ctx)
    acc = np.zeros_like(whole)
    for r in range(4):
        b, c = ofb200.simulation.shard_range(total, r, 4)
        assert c <= one_pass
        acc += _feas(ofb200, pos, tf, c, 21, 4, ctx, trial_begin=b)
    np.testing.assert_allclose(acc, whole, rtol=1e-10, atol=1e-9)


@pytest.mark.parametrize("n_points", [5, 31, 33, 256])
def test_mc_feas_per_trial_warp_contention(ctx, pool, n_points):
    """96 trials = three full warps, each lane adding into the same per-point shared sums; below 32 points the rotated
    start index wraps with %. Sums against the oracle's feas_trial at the bar of the existing 8-trial check."""
    import ofb200
    pos, tf = pool[0][:n_points], pool[1][:n_points]
    seed, sid, ntr = 4242, 3, 96
    sums = _feas(ofb200, pos, tf, ntr, seed, sid, ctx)
    z = vo.mc_normals(seed, sid, np.arange(ntr), n_points)
    acc = np.zeros((6, n_points))
    for k in range(ntr):
        acc += np.array(vo.feas_trial(W, 1.3, NRM, T3, pos, tf, V, SIG["ang_vel_sig"] * z[k, 0, :3],
                                      SIG["translation_sig"] * z[k, 1, :3], SIG["height_sig"] * z[k, 0, 3],
                                      SIG["flow_sig"] * z[k, 3:, 0:2], SIG["position_sig"] * z[k, 3:, 2:4],
                                      0.01 * z[k, 2, :3], 0.3 * 0.3 * z[k, 1, 3], 0.3 * 0.3 * z[k, 2, 3]))
    np.testing.assert_allclose(sums, acc, rtol=1e-7, atol=1e-9)


# ---- one-point steps ------------------------------------------------------------------------------------------------
def test_mc_rejects_one_point_steps(ctx, pool):
    """With one point the SIM normal matrix q^2 (|X|^2 I - X X^T) has X in its null space: every trial would divide by
    a determinant made of rounding noise. Both the Python layer and the C ABI refuse such a step."""
    import ofb200
    sim = ofb200.simulation
    pos, tf = pool[0][:1], pool[1][:1]
    with pytest.raises(ValueError, match="at least 2"):
        _step(_prm(), 1, 0)
    step = _step(_prm(), 2, 0)
    step.n_points = 1                                    # past make_step, straight to the library
    for precision in ("fp32", "fp64"):
        with pytest.raises(ValueError, match="points"):
            sim.run_steps([step], pool[0], pool[1], 8, precision=precision, ctx=ctx)
    with pytest.raises(ValueError):
        ofb200.of_simulation(V, W, 1.3, NRM, T3, pos, 0, 0, 0, 0, 0, 0, iterations=4, true_flow=tf, ctx=ctx)
    with pytest.raises(ValueError):
        _feas(ofb200, pos, tf, 8, 1, 0, ctx)
    sums6 = np.zeros((6, 2))
    rc = ctx.lib.ofb_mc_feas(ctx.h, C.cast(C.byref(step), C.c_void_p), 0, ofb200._lib.ptr(pool[0]),
                             ofb200._lib.ptr(pool[1]), 0, 8, 1, ofb200._lib.ptr(sums6))
    with pytest.raises(ValueError, match="points"):
        ofb200._lib.check(rc)
    # the context is still usable, and two points are fine
    sums = sim.run_steps([_step(_prm(), 2, 0)], pool[0], pool[1], 8, ctx=ctx)
    assert sums["n"][0] == 8 and np.all(np.isfinite(sums["sum_dv"][0]))


# ---- overlap helpers ------------------------------------------------------------------------------------------------
def _hist(ctx, data, lo, hi, bins):
    import ofb200
    data = np.ascontiguousarray(data, dtype=np.float64)
    out = np.zeros(bins, np.uint64)
    ofb200._lib.check(ctx.lib.ofb_histogram(ctx.h, ofb200._lib.ptr(data), len(data), lo, hi, bins,
                                            ofb200._lib.ptr(out)))
    return out.astype(np.int64)


def _minmax(ctx, data):
    import ofb200
    data = np.ascontiguousarray(data, dtype=np.float64)
    lo, hi = C.c_double(), C.c_double()
    ofb200._lib.check(ctx.lib.ofb_minmax(ctx.h, ofb200._lib.ptr(data), len(data), C.byref(lo), C.byref(hi)))
    return lo.value, hi.value


def _on_edges(lo, hi, bins):
    """NumPy's bin edges over [lo, hi] and their neighbouring doubles on both sides, clipped to the range."""
    e = np.linspace(lo, hi, bins + 1)
    return np.clip(np.concatenate([e, np.nextafter(e, -np.inf), np.nextafter(e, np.inf)]), lo, hi)


def test_histogram_on_numpy_bin_edges(ctx):
    """Samples exactly on np.linspace(lo, hi, bins + 1) and one ulp either side, lo and hi themselves: the counts
    equal np.histogram's for 1, 100 and 4096 bins, and overlap equals the reference's, over random ranges."""
    import ofb200
    rng = np.random.default_rng(5)
    for _ in range(25):
        lo = rng.normal(0, 3)
        hi = lo + rng.uniform(1e-3, 20)
        for bins in (1, 100, 4096):
            d = _on_edges(lo, hi, bins)
            d = np.concatenate([d, rng.uniform(lo, hi, 500)])
            assert np.array_equal(_hist(ctx, d, lo, hi, bins), np.histogram(d, bins=bins, range=(lo, hi))[0]), (lo, hi, bins)
        a = _on_edges(lo, hi, 100)                      # pooled range is exactly [lo, hi]
        b = np.concatenate([a[::3], rng.uniform(lo, hi, 200)])
        assert ofb200.overlap(a, b, ctx=ctx) == vo.overlap(a, b), (lo, hi)
        assert ofb200.overlap(a[1::2], a, ctx=ctx) == vo.overlap(a[1::2], a), (lo, hi)


def test_histogram_degenerate_and_quantised(ctx):
    import ofb200
    rng = np.random.default_rng(6)
    # lo == hi: NumPy widens the range to [lo - 0.5, lo + 0.5]
    c = 2.75
    d = np.array([c, c, c - 0.5, c + 0.5, c - 0.25, c + 0.1, c - 0.6, c + 0.6])
    assert np.array_equal(_hist(ctx, d, c, c, 100), np.histogram(d, bins=100, range=(c, c))[0])
    assert ofb200.overlap(np.full(5, c), np.full(3, c), ctx=ctx) == vo.overlap(np.full(5, c), np.full(3, c)) == 3
    # quantised samples land on (or one rounding from) the edges of their own pooled range
    cases = [(rng.integers(-5, 6, 3000).astype(float), rng.integers(-3, 8, 2000).astype(float)),
             (np.round(rng.normal(0, 1, 4000), 1), np.round(rng.normal(0.5, 1.5, 3000), 1)),
             (np.round(rng.uniform(-2, 3, 1000), 2), np.round(rng.uniform(-2, 3, 1000), 1)),
             (rng.integers(0, 101, 5000) * 0.01, rng.integers(0, 101, 5000) * 0.01 + 0.3)]
    for a, b in cases:
        assert ofb200.overlap(a, b, ctx=ctx) == vo.overlap(a, b)
        pooled = np.hstack([a, b])
        lo, hi = pooled.min(), pooled.max()
        for bins in (1, 100, 4096):
            assert np.array_equal(_hist(ctx, pooled, lo, hi, bins), np.histogram(pooled, bins=bins)[0]), bins


def test_minmax_and_non_finite_input(ctx):
    import ofb200
    rng = np.random.default_rng(7)
    for n in (1, 255, 256, 257, 100_003):
        d = rng.normal(0, 1, n)
        assert _minmax(ctx, d) == (d.min(), d.max()), n
        d[rng.integers(n)] = -1e300; d[rng.integers(n)] = 1e300      # extremes anywhere in the array
        assert _minmax(ctx, d) == (d.min(), d.max()), n
    # NumPy refuses a NaN or infinite autodetected range; overlap does the same instead of binning what is left
    a, b = rng.normal(size=300), rng.normal(size=200)
    for bad in (np.nan, np.inf, -np.inf):
        for which in (0, 1):
            xy = [a.copy(), b.copy()]
            xy[which][17] = bad
            with pytest.raises(ValueError):
                vo.overlap(*xy)
            with pytest.raises(ValueError, match="finite"):
                ofb200.overlap(*xy, ctx=ctx)
    # an explicit non-finite range: NumPy raises, and so does the library
    for lo, hi in ((-np.inf, 1.0), (0.0, np.inf), (np.nan, 1.0), (0.0, np.nan)):
        with pytest.raises(ValueError):
            np.histogram(a, bins=100, range=(lo, hi))
        with pytest.raises(ValueError, match="finite"):
            _hist(ctx, a, lo, hi, 100)
    assert ofb200.overlap(a, b, ctx=ctx) == vo.overlap(a, b)
