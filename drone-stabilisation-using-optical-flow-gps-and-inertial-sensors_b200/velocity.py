"""Stage 4 host mirror: the reference's "TODO move to of_library" functions (velocity_measurment_node:23)
with their positional signatures and return tuples, backed by libofb200.so.

    solve_lgs(x,u,d,n,omega)        velocity_measurment_node:30-42      -> (v, res, rank, s)
    solve_lgs(x,u,d,n,omega,t)      numerical_simulation/simulation.py:15-30 -> (v, res, s)
    solve_lgs(..., variant='exp')   flight_experiments/evaluate_exp.py:18-31 -> (v, res)
    solve_lgs_module(x,u,n,dist)    optical_flow_experiments/of_module.py:136-146 (inline lstsq) -> (v, res, rank, s)
    generate_test_data(x,v,omega,d,n[,t])   node:25-29 / simulation.py:7-12
    feasibility(position,linear_velocity,flow,angular_velocity,translation,normal)  simulation.py:108-120
"""
import ctypes as C

import numpy as np

from . import _lib


def _pts(a, name):
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 3 and a.shape[1] == 1:          # cv2-style (N,1,2), as evaluate_exp.py:113 passes
        a = a.reshape(a.shape[0], a.shape[2])
    if a.ndim != 2 or a.shape[1] < 2:
        raise ValueError("%s must have shape (N,2) or (N,1,2)" % name)
    return np.ascontiguousarray(a[:, :2])


def _vec3(a, name):
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    if a.size != 3:
        raise ValueError("%s must have 3 components" % name)
    return np.ascontiguousarray(a)


def _scalar(d):
    return float(np.asarray(d, dtype=np.float64).reshape(-1)[0])   # simulation.py:42 hands in a shape-(1,) array


def solve_full(x, u, d, n, omega, t=None, variant="node", ctx=None):
    """All outputs of the device solve: v (3,), res (1,)|(0,), rank, s (3,)."""
    ctx = ctx or _lib.default_context()
    x = _pts(x, "x")
    u = _pts(u, "u")
    if len(x) != len(u):
        raise ValueError("x and u must have the same number of rows")
    n3, w3 = _vec3(n, "n"), _vec3(omega, "omega")
    t3 = _vec3(t, "t") if t is not None else None
    v = np.zeros(3)
    s = np.zeros(3)
    res = C.c_double(0.0)
    rank = C.c_int(0)
    _lib.check(ctx.lib.ofb_solve_velocity(ctx.h, _lib.VARIANTS[variant], _lib.ptr(x), _lib.ptr(u), len(x), _scalar(d),
                                          _lib.ptr(n3), _lib.ptr(w3), _lib.ptr(t3), _lib.ptr(v), C.addressof(res),
                                          C.addressof(rank), _lib.ptr(s)))
    # np.linalg.lstsq returns the residual sum only for full-rank over-determined systems
    r = np.array([res.value]) if (rank.value == 3 and 3 * len(x) > 3) else np.array([])
    return v, r, rank.value, s


def solve_lgs(x, u, d, n, omega, t=None, variant=None, ctx=None):
    """Drop-in for the three reference solve_lgs copies; the return tuple follows the variant."""
    if variant is None:
        variant = "node" if t is None else "sim"
    if variant not in _lib.VARIANTS:
        raise ValueError("variant must be one of %s" % sorted(_lib.VARIANTS))
    if variant != "node" and t is None:
        raise TypeError("solve_lgs variant %r needs the lever arm t" % variant)
    v, res, rank, s = solve_full(x, u, d, n, omega, t, variant, ctx)
    if variant == "node":
        return v, res, rank, s
    if variant == "exp":
        return v, res
    return v, res, s


def solve_lgs_module(x, u, n, dist=None, v_prior=None, ctx=None):
    """The inline system of optical_flow_experiments/of_module.py:136-146, `np.linalg.lstsq(A, B)` with
    A_i = [X_i]x / dist_i and B_i = A_i u_i / (n . X_i) -> (v_obs, R, rank, s) as lstsq returns them.
    x, u: (N,2), or the homogeneous (N,3) rows (x, y, 1) / (ux, uy, 0) of of_module.py:96-108. dist: the per-point
    `distance` output of the 4-argument of.r_tilde (of_module.py:125); when omitted it is derived on the device from
    v_prior exactly as that r_tilde does."""
    ctx = ctx or _lib.default_context()
    x = np.asarray(x, dtype=np.float64)
    u = np.asarray(u, dtype=np.float64)
    if x.ndim == 3 and x.shape[1] == 1:
        x = x.reshape(len(x), -1)
        u = u.reshape(len(u), -1)
    if x.ndim != 2 or x.shape[1] not in (2, 3) or u.shape != x.shape:
        raise ValueError("x and u must both have shape (N,2) or (N,3)")
    x, u = np.ascontiguousarray(x), np.ascontiguousarray(u)
    if dist is None and v_prior is None:
        raise ValueError("solve_lgs_module needs the per-point distances or the prior velocity they derive from")
    dd = None
    if dist is not None:
        dd = np.ascontiguousarray(np.asarray(dist, dtype=np.float64).reshape(-1))
        if len(dd) != len(x):
            raise ValueError("one distance per point is required")
    n3 = _vec3(n, "n")
    vp = _vec3(v_prior, "v_prior") if v_prior is not None else None
    v = np.zeros(3)
    s = np.zeros(3)
    res = C.c_double(0.0)
    rank = C.c_int(0)
    _lib.check(ctx.lib.ofb_solve_velocity_module(ctx.h, _lib.ptr(x), _lib.ptr(u), len(x), x.shape[1], _lib.ptr(dd),
                                                 _lib.ptr(n3), _lib.ptr(vp), _lib.ptr(v), C.addressof(res),
                                                 C.addressof(rank), _lib.ptr(s)))
    r = np.array([res.value]) if (rank.value == 3 and 3 * len(x) > 3) else np.array([])
    return v, r, rank.value, s


def solve_lgs_batched(x, u, offsets, d, n, omega, t=None, variant="node", ctx=None):
    """Many frames at once: frame f uses rows offsets[f]:offsets[f+1]. Returns v (F,3), res (F,), rank (F,), s (F,3)."""
    ctx = ctx or _lib.default_context()
    x = _pts(x, "x")
    u = _pts(u, "u")
    offsets = np.ascontiguousarray(offsets, dtype=np.int32)
    F = len(offsets) - 1
    if F < 1 or offsets[0] < 0 or np.any(np.diff(offsets) < 0):
        raise ValueError("offsets must be a non-decreasing sequence of at least two non-negative row indices")
    if len(x) != len(u) or len(x) < offsets[-1]:
        raise ValueError("x and u must have the same number of rows, at least offsets[-1] = %d" % offsets[-1])
    d = np.ascontiguousarray(np.broadcast_to(np.asarray(d, dtype=np.float64).reshape(-1), (F,)))
    n3 = np.ascontiguousarray(np.broadcast_to(np.asarray(n, dtype=np.float64), (F, 3)))
    w3 = np.ascontiguousarray(np.broadcast_to(np.asarray(omega, dtype=np.float64), (F, 3)))
    t3 = None if t is None else np.ascontiguousarray(np.broadcast_to(np.asarray(t, dtype=np.float64), (F, 3)))
    v = np.zeros((F, 3))
    res = np.zeros(F)
    rank = np.zeros(F, np.int32)
    s = np.zeros((F, 3))
    _lib.check(ctx.lib.ofb_solve_velocity_batched(ctx.h, _lib.VARIANTS[variant], _lib.ptr(x), _lib.ptr(u),
                                                  _lib.ptr(offsets), F, _lib.ptr(d), _lib.ptr(n3), _lib.ptr(w3),
                                                  _lib.ptr(t3), _lib.ptr(v), _lib.ptr(res), _lib.ptr(rank), _lib.ptr(s)))
    return v, res, rank, s


def _ego_variant(variant):
    if variant not in _lib.VARIANTS:
        raise ValueError("ego-motion variant must be one of %s (module has no gyro term)" % sorted(_lib.VARIANTS))
    return _lib.VARIANTS[variant]


def solve_ego_motion(x, u, d, n, t=None, variant="node", ctx=None):
    """The angular rate estimated from the flow together with the velocity (include/ofb200.h, ofb_solve_ego_motion):
    np.linalg.lstsq on the 3N x 6 system in (v', omega), v' = v + omega x t. No gyro sample is used.
    Returns (v (3,), omega (3,), res (1,)|(0,), rank, s (6,)); res follows lstsq (only for rank 6 and 3N > 6)."""
    var = _ego_variant(variant)
    x = _pts(x, "x")
    u = _pts(u, "u")
    if len(x) != len(u):
        raise ValueError("x and u must have the same number of rows")
    n3 = _vec3(n, "n")
    t3 = _vec3(t, "t") if t is not None else None
    ctx = ctx or _lib.default_context()
    rec = np.zeros(1, _lib.EGO_RESULT_DTYPE)
    _lib.check(ctx.lib.ofb_solve_ego_motion(ctx.h, var, _lib.ptr(x), _lib.ptr(u), len(x), _scalar(d), _lib.ptr(n3),
                                            _lib.ptr(t3), _lib.ptr(rec)))
    r = rec[0]
    res = np.array([r["res"]]) if (r["rank"] == 6 and 3 * len(x) > 6) else np.array([])
    return r["v"].copy(), r["w"].copy(), res, int(r["rank"]), r["s"].copy()


def solve_ego_motion_batched(x, u, offsets, d, n, t=None, variant="node", ctx=None):
    """Many frames at once, frame f on rows offsets[f]:offsets[f+1] -> _lib.EGO_RESULT_DTYPE records (F,)."""
    var = _ego_variant(variant)
    x = _pts(x, "x")
    u = _pts(u, "u")
    offsets = np.ascontiguousarray(offsets, dtype=np.int32)
    F = len(offsets) - 1
    if F < 1 or offsets[0] < 0 or np.any(np.diff(offsets) < 0):
        raise ValueError("offsets must be a non-decreasing sequence of at least two non-negative row indices")
    if len(x) != len(u) or len(x) < offsets[-1]:
        raise ValueError("x and u must have the same number of rows, at least offsets[-1] = %d" % offsets[-1])
    d = np.ascontiguousarray(np.broadcast_to(np.asarray(d, dtype=np.float64).reshape(-1), (F,)))
    n3 = np.ascontiguousarray(np.broadcast_to(np.asarray(n, dtype=np.float64), (F, 3)))
    t3 = None if t is None else np.ascontiguousarray(np.broadcast_to(np.asarray(t, dtype=np.float64), (F, 3)))
    out = np.zeros(F, _lib.EGO_RESULT_DTYPE)
    ctx = ctx or _lib.default_context()
    _lib.check(ctx.lib.ofb_solve_ego_motion_batched(ctx.h, var, _lib.ptr(x), _lib.ptr(u), _lib.ptr(offsets), F, _lib.ptr(d),
                                                    _lib.ptr(n3), _lib.ptr(t3), _lib.ptr(out)))
    return out


def _robust_args(variant, c, iterations):
    if variant not in _lib.VARIANTS:
        raise ValueError("robust variant must be one of %s (module is not supported)" % sorted(_lib.VARIANTS))
    return _lib.VARIANTS[variant], _lib.robust_cfg((c, iterations))


def solve_velocity_robust(x, u, d, n, omega, t=None, variant="node", c=4.0, iterations=10, want_weights=False, ctx=None):
    """Robust velocity solve (include/ofb200.h, ofb_solve_velocity_robust): iteratively reweighted least squares with
    Tukey's biweight, tau = c x the lower median of the point residual norms, `iterations` reweighted solves after the
    plain one (0 is the plain solve). Returns the _lib.ROBUST_RESULT_DTYPE record, and with want_weights also every
    point's weight in the last solve (N,)."""
    var, cfg = _robust_args(variant, c, iterations)
    x = _pts(x, "x")
    u = _pts(u, "u")
    if len(x) != len(u):
        raise ValueError("x and u must have the same number of rows")
    n3, w3 = _vec3(n, "n"), _vec3(omega, "omega")
    t3 = _vec3(t, "t") if t is not None else None
    ctx = ctx or _lib.default_context()
    rec = np.zeros(1, _lib.ROBUST_RESULT_DTYPE)
    wts = np.zeros(len(x)) if want_weights else None
    _lib.check(ctx.lib.ofb_solve_velocity_robust(ctx.h, var, _lib.ptr(x), _lib.ptr(u), len(x), _scalar(d), _lib.ptr(n3),
                                                 _lib.ptr(w3), _lib.ptr(t3), C.byref(cfg), _lib.ptr(rec), _lib.ptr(wts)))
    return (rec[0], wts) if want_weights else rec[0]


def solve_velocity_robust_batched(x, u, offsets, d, n, omega, t=None, variant="node", c=4.0, iterations=10,
                                  want_weights=False, ctx=None):
    """Many frames at once, frame f on rows offsets[f]:offsets[f+1] -> _lib.ROBUST_RESULT_DTYPE records (F,), and with
    want_weights the weights of every row (rows in no frame get 0)."""
    var, cfg = _robust_args(variant, c, iterations)
    x = _pts(x, "x")
    u = _pts(u, "u")
    offsets = np.ascontiguousarray(offsets, dtype=np.int32)
    F = len(offsets) - 1
    if F < 1 or offsets[0] < 0 or np.any(np.diff(offsets) < 0):
        raise ValueError("offsets must be a non-decreasing sequence of at least two non-negative row indices")
    if len(x) != len(u) or len(x) < offsets[-1]:
        raise ValueError("x and u must have the same number of rows, at least offsets[-1] = %d" % offsets[-1])
    d = np.ascontiguousarray(np.broadcast_to(np.asarray(d, dtype=np.float64).reshape(-1), (F,)))
    n3 = np.ascontiguousarray(np.broadcast_to(np.asarray(n, dtype=np.float64), (F, 3)))
    w3 = np.ascontiguousarray(np.broadcast_to(np.asarray(omega, dtype=np.float64), (F, 3)))
    t3 = None if t is None else np.ascontiguousarray(np.broadcast_to(np.asarray(t, dtype=np.float64), (F, 3)))
    out = np.zeros(F, _lib.ROBUST_RESULT_DTYPE)
    wts = np.zeros(int(offsets[-1])) if want_weights else None
    ctx = ctx or _lib.default_context()
    _lib.check(ctx.lib.ofb_solve_velocity_robust_batched(ctx.h, var, _lib.ptr(x), _lib.ptr(u), _lib.ptr(offsets), F,
                                                         _lib.ptr(d), _lib.ptr(n3), _lib.ptr(w3), _lib.ptr(t3),
                                                         C.byref(cfg), _lib.ptr(out), _lib.ptr(wts if wts is None or len(wts) else None)))
    return (out, wts) if want_weights else out


def generate_test_data(x, v, omega, d, n, t=None, ctx=None):
    ctx = ctx or _lib.default_context()
    x = _pts(x, "x")
    out = np.zeros((len(x), 2))
    v3, w3, n3 = _vec3(v, "v"), _vec3(omega, "omega"), _vec3(n, "n")
    t3 = _vec3(t, "t") if t is not None else None
    _lib.check(ctx.lib.ofb_generate_flow(ctx.h, _lib.ptr(x), len(x), _lib.ptr(v3), _lib.ptr(w3), _scalar(d),
                                         _lib.ptr(n3), _lib.ptr(t3), _lib.ptr(out)))
    return out


def feasibility(position, linear_velocity, flow, angular_velocity, translation, normal, ctx=None):
    ctx = ctx or _lib.default_context()
    x = _pts(position, "position")
    u = _pts(flow, "flow")
    out = np.zeros((2, len(x)))
    # keep the converted vectors alive across the call (ptr() does not hold a reference)
    v3, w3 = _vec3(linear_velocity, "linear_velocity"), _vec3(angular_velocity, "angular_velocity")
    t3, n3 = _vec3(translation, "translation"), _vec3(normal, "normal")
    _lib.check(ctx.lib.ofb_feasibility(ctx.h, _lib.ptr(x), _lib.ptr(v3), _lib.ptr(u), len(x), _lib.ptr(w3), _lib.ptr(t3),
                                       _lib.ptr(n3), _lib.ptr(out)))
    return out


def quaternion_to_rotation(qx, qy, qz, qw):
    """velocity_measurment_node:65-68 / evaluate_exp.py:88-91 (per-frame, 9 numbers: host side)."""
    return np.array([
        [1.0 - 2 * (qy ** 2 + qz ** 2), 2 * (qx * qy - qw * qz), 2 * (qw * qy + qx * qz)],
        [2 * (qx * qy + qw * qz), 1.0 - 2 * (qx ** 2 + qz ** 2), 2 * (qy * qz - qw * qx)],
        [2 * (qx * qz - qw * qy), 2 * (qw * qx + qy * qz), 1.0 - 2 * (qx ** 2 + qy ** 2)]])


def plane_normal(R):
    """velocity_measurment_node:70: n = R . e_z."""
    return np.asarray(R, dtype=np.float64)[:, 2].copy()


def body_to_world(R, v_obs, omega, offset):
    """velocity_measurment_node:258: v_uav = R (v_obs - [omega]x offset)."""
    w = np.asarray(omega, dtype=np.float64)
    return np.asarray(R, dtype=np.float64) @ (np.asarray(v_obs, dtype=np.float64) - np.cross(w, np.asarray(offset, dtype=np.float64)))
