"""Pins the numpy oracle (oracle/velocity_oracle.py) to the REFERENCE: against the committed golden
outputs of the reference's own functions (tests/golden/velocity_golden.npz, made by
tools/make_golden.py) and, where OFB_REFERENCE_DIR names a checkout of it, against those functions run live."""
import os
import warnings

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import velocity_oracle as vo
from oracle import ref_loader


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLDEN, "velocity_golden.npz"))


def test_round_trip_known_answers(g):
    # SURVEY 4: solve_lgs(generate_test_data(points.txt, v=w=1, d=1, n=e_z, t)) == [1,1,1]
    pts = g["points"]
    v, w, t = np.ones(3), np.ones(3), np.array([0.02, 0, 0.205])
    tf = vo.generate_test_data(pts, v, w, 1.0, [0, 0, 1], t)
    np.testing.assert_allclose(tf, g["sim_true_flow"], rtol=0, atol=1e-14)
    vv, res, rank, s = vo.solve_lgs(pts, tf, 1.0, [0, 0, 1], w, t, variant="sim")
    np.testing.assert_allclose(vv, [1, 1, 1], atol=1e-12)
    np.testing.assert_allclose(s, g["sim_rt_s"], rtol=1e-12)
    np.testing.assert_allclose(s, [14.763, 14.674, 5.739], atol=2e-3)
    u = vo.generate_test_data(g["node_pts"], [1, 1, 1], [0, 0, 0], 0.75, [0, 0, 1])
    np.testing.assert_allclose(u, g["node_flow"], atol=1e-14)
    vv, res, rank, s = vo.solve_lgs(g["node_pts"], u, 0.75, [0, 0, 1], [0, 0, 0], variant="node")
    np.testing.assert_allclose(vv, [1, 1, 1], atol=1e-12)
    np.testing.assert_allclose(s, g["node_rt_s"], rtol=1e-12)
    assert rank == int(g["node_rt_rank"]) == 3


def test_three_variants_match_reference(g):
    for i in range(int(g["n_cases"])):
        c = {k: g["case%d_%s" % (i, k)] for k in ("x", "u", "d", "n", "w", "t", "v_sim", "s_sim", "res_sim", "v_node",
                                                  "s_node", "res_node", "rank_node", "v_exp", "res_exp")}
        v, res, rank, s = vo.solve_lgs(c["x"], c["u"], c["d"], c["n"], c["w"], c["t"], variant="sim")
        np.testing.assert_allclose(v, c["v_sim"], rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(s, c["s_sim"], rtol=1e-12)
        np.testing.assert_allclose(res, c["res_sim"], rtol=1e-8, atol=1e-20)
        v, res, rank, s = vo.solve_lgs(c["x"], c["u"], c["d"], c["n"], c["w"], variant="node")
        np.testing.assert_allclose(v, c["v_node"], rtol=1e-10, atol=1e-12)
        assert rank == int(c["rank_node"])
        v, res, rank, s = vo.solve_lgs(c["x"], c["u"], c["d"], c["n"], c["w"], c["t"], variant="exp")
        np.testing.assert_allclose(v, c["v_exp"], rtol=1e-10, atol=1e-12)


def test_r_tilde_and_feasibility(g):
    r, d = vo.r_tilde(g["rt5_x"], g["rt5_u"], [0, 0, 1], [0.1, 0.1, 0.1], 0.75)
    np.testing.assert_allclose(r, g["rt5_r"], atol=1e-13)
    np.testing.assert_allclose(d, g["rt5_d"], rtol=1e-12)
    np.testing.assert_allclose(r, -1.0, atol=1e-12)          # of_library.py:363-364: "-1 for properly solved array"
    r, d = vo.r_tilde(g["rt5_x"], g["rt5n_u"], g["rt5n_n"], [0.1, 0.1, 0.1], 0.75)
    np.testing.assert_allclose(r, g["rt5n_r"], atol=1e-13)
    np.testing.assert_allclose(d, g["rt5n_d"], rtol=1e-12)
    r, d = vo.r_tilde(g["rt4_x"], g["rt4_u"], [0, 0, 1], [0.1, 0.1, 0.1])
    np.testing.assert_allclose(r, g["rt4_r"], atol=1e-13)
    np.testing.assert_allclose(d, g["rt4_d"], rtol=1e-12)
    f = vo.feasibility(g["points"][:50], np.ones(3), g["feas_flow"], np.ones(3) + 0.01, [0.02, 0, 0.205], [0, 0, 1])
    np.testing.assert_allclose(f, g["feas_out"], rtol=1e-12, atol=1e-14)


def test_of_simulation_replays_reference_draws(g):
    # same legacy RNG seed -> same Gaussian draws in the same order as simulation.py:40-45
    np.random.seed(777)
    v_obs, R = vo.of_simulation(6, np.random, np.ones(3), np.ones(3), 1.0, np.array([0, 0, 1.0]),
                                np.array([0.02, 0, 0.205]), g["ofsim_pos"], g["ofsim_flow"], 0.00071, 0.005, 0.01,
                                0.056 * np.sqrt(2) * 1.23, 0.056 * 1.23, 0.00065)
    np.testing.assert_allclose(v_obs, g["ofsim_v"], rtol=1e-10)
    np.testing.assert_allclose(R, g["ofsim_R"], rtol=1e-10)


def test_overlap_and_small_helpers(g):
    assert vo.overlap(g["ov_a"], g["ov_b"]) == int(g["ov_out"])
    assert vo.pix_trans((320, 240)) == (160, 120)
    assert vo.pix_trans((481, 643)) == (241, 322)
    R = vo.quat_to_rot(0.1, -0.2, 0.3, np.sqrt(1 - 0.14))
    np.testing.assert_allclose(R @ R.T, np.eye(3), atol=1e-12)
    np.testing.assert_allclose(vo.body_to_world(np.eye(3), [1, 2, 3], [0, 0, 1], [0, 0, 0.1]), [1, 2, 3], atol=1e-15)


def test_philox_known_answer():
    # Random123 known-answer vectors for philox4x32-10
    out = vo.philox4x32_10(np.array([[0, 0, 0, 0]], dtype=np.uint64), np.array([0, 0], dtype=np.uint64))[0]
    assert [int(x) for x in out] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    out = vo.philox4x32_10(np.array([[0xffffffff] * 4], dtype=np.uint64), np.array([0xffffffff] * 2, dtype=np.uint64))[0]
    assert [int(x) for x in out] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    out = vo.philox4x32_10(np.array([[0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]], dtype=np.uint64),
                           np.array([0xa4093822, 0x299f31d0], dtype=np.uint64))[0]
    assert [int(x) for x in out] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    z = vo.mc_normals(1, 0, np.arange(20000), 2)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01


@pytest.mark.skipif(not ref_loader.available(), reason=ref_loader.MISSING)
def test_oracle_against_live_reference():
    sim = ref_loader.simulation()
    node = ref_loader.node()
    rng = np.random.default_rng(3)
    for _ in range(5):
        N = int(rng.integers(3, 60))
        x = rng.uniform(-0.5, 0.5, (N, 2)); u = rng.normal(0, 0.3, (N, 2))
        d = rng.uniform(0.5, 3); n = np.array([0.05, -0.03, 1.0]); w = rng.normal(0, 0.3, 3); t = rng.normal(0, 0.1, 3)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            v_ref, _, s_ref = sim["solve_lgs"](x, u, d, n, w, t)
            vn_ref = node["solve_lgs"](x, u, d, n, w)[0]
        v, _, _, s = vo.solve_lgs(x, u, d, n, w, t, variant="sim")
        np.testing.assert_allclose(v, v_ref, rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(s, s_ref, rtol=1e-12)
        np.testing.assert_allclose(vo.solve_lgs(x, u, d, n, w, variant="node")[0], vn_ref, rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(vo.generate_test_data(x, [1, 2, 3], w, d, n, t),
                                   sim["generate_test_data"](x, np.array([1.0, 2, 3]), w, d, n, t), atol=1e-13)
        np.testing.assert_allclose(vo.feasibility(x, [1, 2, 3], u, w, t, n),
                                   sim["feasibility"](x, np.array([1.0, 2, 3]), u, w, t, n), rtol=1e-12)


# ---- round 2: of_module's inline system, the time-evolution sweep, the live sorting scenario -----------------
@pytest.fixture(scope="module")
def g2():
    return np.load(os.path.join(GOLDEN, "velocity_golden_r2.npz"))


def test_module_system_matches_reference(g2):
    """oracle.solve_lgs_module == the statements of of_module.py:136-146 exec'd unmodified (golden), with the
    distances of the reference's own 4-argument r_tilde."""
    for c in range(int(g2["module_n_cases"])):
        k = lambda s: g2["module%d_%s" % (c, s)]
        r, dist = vo.r_tilde(k("x"), k("u"), k("n"), k("v_prior"))
        np.testing.assert_allclose(dist, k("dist"), rtol=1e-12)
        np.testing.assert_allclose(r, k("feas"), atol=1e-12)
        v, res, rank, s = vo.solve_lgs_module(k("x"), k("u"), k("n"), k("dist"))
        np.testing.assert_allclose(v, k("v"), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(s, k("s"), rtol=1e-10)
        assert rank == int(k("rank"))
        np.testing.assert_allclose(res, k("res"), rtol=1e-6, atol=1e-18)


def test_time_evolution_trajectory_matches_reference(g2):
    """oracle.advect_points == the trajectory the reference's commented time-analysis block (simulation.py:472-499)
    printed when its statements were exec'd."""
    pos, hs = vo.advect_points(g2["te_pos"][0], [1, 1, 1], 1.0, [0, 0, 1], [0.02, 0, 0.205], 100)
    np.testing.assert_allclose(hs, g2["te_heights"], rtol=0, atol=0)
    np.testing.assert_allclose(pos, g2["te_pos"], rtol=1e-12, atol=1e-9)
    last = pos[-1] + vo.generate_test_data(pos[-1], [1, 1, 1], np.zeros(3), hs[-1], [0, 0, 1], [0.02, 0, 0.205])
    np.testing.assert_allclose(last, g2["te_final_pos"], rtol=1e-12, atol=1e-9)


def test_live_sorting_scenario_matches_reference(g2, points200):
    """oracle.sorting_scenario_live == what the live statements simulation.py:753-772 built (points, composite flow)."""
    d, tf, v, h = vo.sorting_scenario_live(points200, [1, 1, 1], [1, 1, 1], [0, 0, 1], [0.02, 0, 0.205], g2["live_angles"])
    np.testing.assert_allclose(d, g2["live_data"], atol=1e-13)
    np.testing.assert_allclose(v, g2["live_velocity"], rtol=1e-15)
    assert h == float(g2["live_height"]) == 2.0
    np.testing.assert_allclose(tf, g2["live_true_flow"], rtol=1e-11, atol=1e-12)


@pytest.mark.skipif(not ref_loader.available(), reason=ref_loader.MISSING)
def test_module_system_live_reference():
    """Where the reference exists: regenerate one module case through the AST-extracted statements and compare."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden_r2", os.path.join(os.path.dirname(GOLDEN), "..", "tools",
                                                                               "make_golden_r2.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    g = {}
    mod.module_golden(g)
    for c in range(int(g["module_n_cases"])):
        v, res, rank, s = vo.solve_lgs_module(g["module%d_x" % c], g["module%d_u" % c], g["module%d_n" % c], g["module%d_dist" % c])
        np.testing.assert_allclose(v, g["module%d_v" % c], rtol=1e-9, atol=1e-12)
