"""Ego-motion solve on the host: the literal 3N x 6 oracle (oracle/ego_oracle.py) against the closed-form normal equations
of include/ofb200.h, the reference's flow model, the gyro-based solve and lstsq's rank; the record layout and the Python
plumbing that needs no device."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import ego_oracle as eo
from oracle import velocity_oracle as vo

VARIANTS = ["node", "exp", "sim"]


def scene(seed, spread=0.6, n_pts=60):
    rng = np.random.default_rng(seed)
    x = rng.uniform(-spread, spread, (n_pts, 2))
    v = rng.uniform(-1, 1, 3)
    w = rng.normal(0, 0.3, 3)
    n = np.array([rng.normal(0, 0.1), rng.normal(0, 0.1), 1.0])
    n /= np.linalg.norm(n)
    t = rng.normal(0, 0.1, 3)
    return x, v, w, rng.uniform(0.5, 5.0), n, t


@pytest.mark.parametrize("variant", VARIANTS)
def test_blocks_equal_the_closed_forms(variant):
    x, v, w, d, n, t = scene(1)
    u = vo.generate_test_data(x, v, w, d, n, t) + np.random.default_rng(2).normal(0, 1e-3, x.shape)
    A, b = eo.build_system(x, u, d, n, variant)
    M, g = eo.normal_blocks(x, u, d, n, variant)
    assert np.abs(A.T @ A - M).max() <= 1e-13 * np.abs(M).max()
    assert np.abs(A.T @ b - g).max() <= 1e-13 * np.abs(g).max()


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("lever", [False, True])
@pytest.mark.parametrize("seed", [3, 4, 5])
def test_round_trip_through_generate_test_data(variant, lever, seed):
    """noiseless flow of the reference's model gives back (v, w); NODE has no lever arm, so it returns v + w x t"""
    x, v, w, d, n, t = scene(seed)
    tt = t if lever else None
    u = vo.generate_test_data(x, v, w, d, n, tt)
    ve, we, res, rank, s = eo.solve_ego_motion(x, u, d, n, tt, variant)
    want = v + np.cross(w, t) if (lever and variant == "node") else v
    assert rank == 6 and res.shape == (1,) and res[0] < 1e-20
    np.testing.assert_allclose(we, w, rtol=0, atol=1e-12)
    np.testing.assert_allclose(ve, want, rtol=0, atol=1e-12)


@pytest.mark.parametrize("variant", VARIANTS)
def test_fixed_rate_identity(variant):
    """the joint minimiser, with omega fixed at its estimate, is the gyro-based solve's minimiser"""
    x, v, w, d, n, t = scene(6)
    u = vo.generate_test_data(x, v, w, d, n, t) + np.random.default_rng(7).normal(0, 2e-3, x.shape)
    ve, we, _, _, _ = eo.solve_ego_motion(x, u, d, n, t, variant)
    vg = vo.solve_lgs(x, u, d, n, we, t, variant)[0]
    np.testing.assert_allclose(vg, ve, rtol=0, atol=1e-12 * max(1.0, np.abs(ve).max()))


def test_residual_is_the_stacked_systems():
    x, v, w, d, n, t = scene(8)
    u = vo.generate_test_data(x, v, w, d, n, t) + np.random.default_rng(9).normal(0, 1e-2, x.shape)
    A, b = eo.build_system(x, u, d, n, "sim")
    sol, res, _, _ = np.linalg.lstsq(A, b, rcond=None)
    assert abs(eo.residual(x, u, d, n, "sim", sol[:3], sol[3:]) - res[0]) <= 1e-10 * res[0]


@pytest.mark.parametrize("variant", VARIANTS)
def test_degenerate_inputs_are_rank_deficient(variant):
    """one point, two points and many points at one X: rank < 6, as lstsq finds it"""
    _, v, w, d, n, _ = scene(10)
    cases = {1: np.array([[0.1, -0.2]]), 2: np.array([[0.1, -0.2], [-0.3, 0.25]]), 3: np.tile([[0.2, 0.1]], (40, 1))}
    for pts in cases.values():
        u = vo.generate_test_data(pts, v, w, d, n)
        A, b = eo.build_system(pts, u, d, n, variant)
        _, _, res, rank, s = eo.solve_ego_motion(pts, u, d, n, None, variant)
        assert rank == np.linalg.matrix_rank(A) < 6 and res.shape == (0,)
    assert eo.solve_ego_motion(cases[1], vo.generate_test_data(cases[1], v, w, d, n), d, n)[3] == 2
    assert eo.solve_ego_motion(cases[2], vo.generate_test_data(cases[2], v, w, d, n), d, n)[3] == 4


def test_module_has_no_rate_to_estimate():
    x, v, w, d, n, _ = scene(11)
    with pytest.raises(ValueError):
        eo.build_system(x, vo.generate_test_data(x, v, w, d, n), d, n, "module")


def test_ego_result_layout_matches_header(tmp_path):
    from ofb200 import _lib
    src = tmp_path / "ego.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ofb200.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %zu %d\\n",'
                   'sizeof(ofb_ego_result),offsetof(ofb_ego_result,v),offsetof(ofb_ego_result,w),offsetof(ofb_ego_result,s),'
                   'offsetof(ofb_ego_result,res),offsetof(ofb_ego_result,rank),offsetof(ofb_ego_result,flags),'
                   'OFB_EGO_SOLVED);return 0;}\n')
    exe = tmp_path / "ego"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    R, D = _lib.EgoResult, _lib.EGO_RESULT_DTYPE
    assert got[:7] == [ctypes.sizeof(R), R.v.offset, R.w.offset, R.s.offset, R.res.offset, R.rank.offset, R.flags.offset]
    assert got[:7] == [D.itemsize] + [D.fields[f][1] for f in ("v", "w", "s", "res", "rank", "flags")]
    assert got[7] == _lib.EGO_SOLVED


def test_fleet_tracker_set_ego_motion_reaches_the_local_tracker():
    import ofb200

    class Fake:
        def __init__(self, n, **kw):
            self.kw, self.calls = kw, []

        def set_ego_motion(self, on):
            self.calls.append(on)

    fleet = ofb200.FleetTracker(3, 64, 48, tracker_factory=lambda n, **kw: Fake(n, **kw), ego_motion=True)
    assert fleet.local.kw["ego_motion"] is True
    fleet.set_ego_motion(False)
    fleet.set_ego_motion(True)
    assert fleet.local.calls == [False, True]
    with pytest.raises(ValueError):
        fleet.set_ego_motion(1)


def test_python_argument_checks_need_no_device():
    import ofb200
    with pytest.raises(ValueError):
        ofb200.solve_ego_motion(np.zeros((3, 2)), np.zeros((3, 2)), 1.0, [0, 0, 1], variant="module")
    with pytest.raises(ValueError):
        ofb200.solve_ego_motion_batched(np.zeros((3, 2)), np.zeros((3, 2)), [0, 2, 1], 1.0, [0, 0, 1])
