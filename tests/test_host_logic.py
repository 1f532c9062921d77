"""Host-side logic that needs no GPU: argument checking, sweep construction, shard arithmetic and the
world_size-2 merge of Monte-Carlo sums over torch.distributed (gloo)."""
import os
import socket

import numpy as np
import pytest

from conftest import GOLDEN


def test_pix_trans_and_static_immobile():
    import ofb200.of_library as of
    assert of.pix_trans((320, 240)) == (160, 120)
    assert of.pix_trans((481, 643)) == (241, 322)
    assert of.pix_trans((480, 640)) == (240, 320)            # of_module.py:100 passes (rows, cols)
    new = np.array([[[1.0, 1.0]], [[5.0, 1.0]], [[-7.0, -7.0]]]); old = np.array([[[0.5, 0.8]], [[0.0, 1.0]], [[-7.0, -7.0]]])
    st = of.static_immobile(new, old, 2.0, 1.0, -7.0)
    assert st.ravel().tolist() == [True, False, False]


def test_shard_ranges_cover_exactly():
    from ofb200 import simulation as sim
    for total in (1, 7, 100, 10 ** 8 + 3):
        for world in (1, 2, 3, 8):
            spans = [sim.shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and sum(c for _, c in spans) == total
            for (b0, c0), (b1, _) in zip(spans, spans[1:]):
                assert b0 + c0 == b1
            assert max(c for _, c in spans) - min(c for _, c in spans) <= 1


def test_sweep_construction_matches_reference_parameters():
    from ofb200 import simulation as sim
    from oracle import velocity_oracle as vo
    pts = np.load(os.path.join(GOLDEN, "points.npy"))
    steps, p, f = sim_build("flow_errors", pts)
    assert len(steps) == 100 and p.shape == (100 * 200, 2)
    assert steps[7].flow_sig == pytest.approx(0.007) and steps[7].position_sig == pytest.approx(np.sqrt(2) / 1000 * 7)
    assert steps[7].ang_vel_sig == 0.00071 and steps[7].pos_offset == 7 * 200
    steps, p, f = sim_build("orientation", pts, 10)
    np.testing.assert_allclose(list(steps[5].n), [1.0, 0.0, np.cos(np.pi / 2)], atol=1e-15)
    steps, p, f = sim_build("number_of_points", pts)
    assert len(steps) == 99 and [s.n_points for s in steps[:3]] == [2, 4, 6] and steps[-1].n_points == 198
    assert steps[2].pos_offset == 6
    steps, p, f = sim_build("height", pts)
    assert steps[0].height == pytest.approx(0.4) and steps[-1].height == pytest.approx(7.85)
    with pytest.raises(ValueError):
        sim.build_sweep("nope", pts)
    with pytest.raises(ValueError):
        sim.make_step([1, 1, 1], [1, 1, 1], 1.0, [0, 0, 1], [0, 0, 0], 5, 0, -1.0, 0, 0, 0, 0, 0)
    for n_points in (1, 0):                             # one point: the velocity solve is singular
        with pytest.raises(ValueError, match="at least 2"):
            sim.make_step([1, 1, 1], [1, 1, 1], 1.0, [0, 0, 1], [0, 0, 0], n_points, 0, 0, 0, 0, 0, 0, 0)
    for bad in (np.nan, np.inf):                        # numpy.histogram refuses a non-finite autodetected range
        with pytest.raises(ValueError, match="finite"):
            sim.overlap(np.array([0.0, bad]), np.array([1.0]))
        with pytest.raises(ValueError):
            vo.overlap(np.array([0.0, bad]), np.array([1.0]))
    d = sim.centred_points(pts)
    assert abs(d[:, 0].mean()) < 1e-15 and d[:, 0].std() == pytest.approx(pts[:, 0].std() * 1.27)


def sim_build(name, pts, k=None):
    """build_sweep needs generate_test_data (GPU); substitute the oracle's flow model so that the
    step/point bookkeeping can be checked on the CPU."""
    from ofb200 import simulation as sim
    from oracle import velocity_oracle as vo
    real = sim._vel.generate_test_data
    sim._vel.generate_test_data = lambda x, v, w, d, n, t=None, ctx=None: vo.generate_test_data(x, v, w, d, n, t)
    try:
        return sim.build_sweep(name, pts, k)
    finally:
        sim._vel.generate_test_data = real


def test_stats_from_sums():
    from ofb200 import simulation as sim, _lib
    rng = np.random.default_rng(0)
    v = 1.0 + rng.normal(0, 0.1, (1000, 3)); R = rng.uniform(0, 1, 1000)
    sums = np.zeros(1, _lib.MCSUMS_DTYPE)
    sums["n"] = 1000; sums["sum_dv"] = (v - 1).sum(0); sums["sum_dv2"] = ((v - 1) ** 2).sum(0); sums["sum_R"] = R.sum()
    step = sim.make_step([1, 1, 1], [0, 0, 0], 1.0, [0, 0, 1], [0, 0, 0], 5, 0, 0, 0, 0, 0, 0, 0)
    mean, std, mR, n = sim.stats_from_sums(sums, [step])
    np.testing.assert_allclose(mean[0], v.mean(0), rtol=1e-12)
    np.testing.assert_allclose(std[0], v.std(0), rtol=1e-10)
    assert mR[0] == pytest.approx(R.mean())


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _merge_worker(rank, world, port, q):
    import torch.distributed as dist
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from ofb200 import simulation as sim, _lib
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    total = 1001
    b, c = sim.shard_range(total, rank, world)
    sums = np.zeros(3, _lib.MCSUMS_DTYPE)
    ids = np.arange(b, b + c, dtype=np.float64)
    for s in range(3):
        sums["n"][s] = c
        sums["sum_dv"][s] = [ids.sum() * (s + 1), 0.5 * c, -ids.sum()]
        sums["sum_dv2"][s] = [(ids ** 2).sum(), c, 2.0 * c]
        sums["sum_R"][s] = ids.sum()
    merged = sim.merge_sums(sums)
    q.put((rank, merged.view(np.float64).reshape(3, 8).tolist()))
    dist.destroy_process_group()


def test_merge_sums_world_size_2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_merge_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    ids = np.arange(1001, dtype=np.float64)
    for rank, m in outs:
        m = np.array(m)
        assert m[0, 0] == 1001
        assert m[1, 1] == pytest.approx(ids.sum() * 2) and m[2, 3] == pytest.approx(-ids.sum())
        assert m[0, 4] == pytest.approx((ids ** 2).sum()) and m[0, 7] == pytest.approx(ids.sum())
    assert outs[0][1] == outs[1][1]


def _hist_worker(rank, world, port, q):
    import torch.distributed as dist
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from ofb200 import simulation as sim
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    rng = np.random.default_rng(9)
    d1, d2 = rng.normal(0, 1, 5000), rng.normal(0.7, 1.3, 4000)
    b1, c1 = sim.shard_range(len(d1), rank, world)
    b2, c2 = sim.shard_range(len(d2), rank, world)
    s1, s2 = d1[b1:b1 + c1], d2[b2:b2 + c2]
    lo, hi = sim.merge_range(min(s1.min(), s2.min()), max(s1.max(), s2.max()))
    # numpy's histogram binning over the merged range stands in for ofb_histogram (same contract, GPU-tested)
    h = np.concatenate([np.histogram(s1, bins=100, range=(lo, hi))[0], np.histogram(s2, bins=100, range=(lo, hi))[0]])
    both = sim.merge_counts(h)
    ids = sim.stream_shard(7, rank, world)
    v = sim.gather_stream_velocities(np.array([[i, 2.0 * i, -i] for i in ids], dtype=float), ids, 7)
    q.put((rank, lo, hi, int(np.minimum(both[:100], both[100:]).sum()), v.tolist()))
    dist.destroy_process_group()


def test_overlap_merge_and_stream_gather_world_size_2_gloo():
    """SURVEY 8e: range all-reduce(min/max) then bin-count all-reduce(sum) reproduce the single-process overlap
    (simulation.py:124-136); stream-sharded velocities gather into one table."""
    import torch.multiprocessing as mp
    from oracle import velocity_oracle as vo
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_hist_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    rng = np.random.default_rng(9)
    d1, d2 = rng.normal(0, 1, 5000), rng.normal(0.7, 1.3, 4000)
    expect = vo.overlap(d1, d2)
    for rank, lo, hi, ov, v in outs:
        assert lo == min(d1.min(), d2.min()) and hi == max(d1.max(), d2.max())
        assert ov == expect
        assert np.array_equal(np.array(v), np.array([[i, 2.0 * i, -i] for i in range(7)], dtype=float))


class _FakeTracker:
    """stands in for StreamTracker (which needs a GPU): stream i reports v = (global id, step, -1); odd ids do not solve"""

    def __init__(self, ids):
        self.ids, self.k = ids, 0

    def step(self, frames, imu):
        from ofb200 import _lib
        self.k += 1
        r = np.zeros(len(self.ids), _lib.TRACK_RESULT_DTYPE)
        for j, g in enumerate(self.ids):
            r["v"][j] = [g, self.k, -1.0]
            r["flags"][j] = 0 if g % 2 else 1
        return r

    def close(self):
        pass


def _fleet_worker(rank, world, port, q):
    import torch.distributed as dist
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import ofb200
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    made = {}

    def factory(n_local, **kw):
        made["n"] = n_local
        return _FakeTracker(ofb200.simulation.stream_shard(9, rank, world))
    fleet = ofb200.FleetTracker(9, 64, 48, tracker_factory=factory)
    assert made["n"] == len(fleet.streams) and fleet.select(list(range(100, 109))) == [100 + s for s in fleet.streams]
    fleet.step(None, None)
    fleet.step(None, None)
    q.put((rank, fleet.streams, fleet.gather_velocities().tolist()))
    fleet.close()
    dist.destroy_process_group()


def test_fleet_tracker_shards_and_gathers_world_size_2_gloo():
    """FleetTracker: streams s mod world per rank, one all-reduce merges the last step's velocities; streams that did
    not solve come back as NaN rows on every rank."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_fleet_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert outs[0][1] == [0, 2, 4, 6, 8] and outs[1][1] == [1, 3, 5, 7]
    for _, _, table in outs:
        t = np.array(table)
        assert t.shape == (9, 3)
        for g in range(9):
            if g % 2:
                assert np.isnan(t[g]).all()
            else:
                assert t[g].tolist() == [g, 2.0, -1.0]


def test_fleet_tracker_single_process():
    import ofb200
    fleet = ofb200.FleetTracker(4, 64, 48, tracker_factory=lambda n, **kw: _FakeTracker([0, 1, 2, 3]))
    assert fleet.streams == [0, 1, 2, 3] and fleet.world == 1
    fleet.step(None, None)
    t = fleet.gather_velocities()
    assert t[0].tolist() == [0.0, 1.0, -1.0] and np.isnan(t[1]).all() and t[2].tolist() == [2.0, 1.0, -1.0]
    fleet.close()


def _fleet_edge_worker(rank, world, port, q):
    """a fleet with fewer streams than ranks (rank 1 owns nothing) and a gather before the first step"""
    import torch.distributed as dist
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import ofb200
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    fleet = ofb200.FleetTracker(1, 64, 48, tracker_factory=lambda n, **kw: _FakeTracker(ofb200.simulation.stream_shard(1, rank, world)))
    before = fleet.gather_velocities()            # nothing stepped yet: every row NaN, on every rank
    fleet.step(None, None)
    after = fleet.gather_velocities()
    q.put((rank, fleet.streams, fleet.local is None, before.tolist(), after.tolist()))
    fleet.close()
    dist.destroy_process_group()


def test_fleet_tracker_rank_without_streams_and_gather_before_first_step_gloo():
    """ADVICE r1: a rank that owns no stream still takes part in the (single) all-reduce, and rows of streams that have
    not solved yet are NaN, not zeros."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_fleet_edge_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert outs[0][1] == [0] and outs[1][1] == [] and outs[1][2] is True
    for _, _, _, before, after in outs:
        assert np.isnan(np.array(before)).all() and np.array(before).shape == (1, 3)
        assert np.array(after).tolist() == [[0.0, 1.0, -1.0]]
