"""CPU ORACLE (test infrastructure, NOT product code) of the robust velocity solve (include/ofb200.h,
ofb_solve_velocity_robust): iteratively reweighted least squares with Tukey's biweight and a median scale.

The stacked 3N x 3 system is velocity_oracle.build_system, built point by point (rows A_i, right-hand side d b_i). Then

    iteration 0:  v'_0 = np.linalg.lstsq(A, d b) -- velocity_oracle.solve_lgs before the lever arm; all weights 1
    k = 1 .. K:   rho_i = |A_i v'_{k-1} - d b_i|,  sigma = np.partition(rho.astype(np.float32), m)[m], m = (N-1)//2,
                  tau = c sigma; tau 0 or not finite: stop (keep v'_{k-1} and its weights);
                  w_i = (1 - (rho_i/tau)^2)^2 for rho_i < tau, else 0;
                  v'_k = np.linalg.lstsq on the sqrt(w_i)-scaled rows of the points with w_i > 0 (rcond=None)
    v = v'_K - omega x t for exp / sim (node has no lever arm), as solve_lgs.
"""
import numpy as np

from .velocity_oracle import build_system, solve_lgs

DEFAULT_C, DEFAULT_ITERATIONS = 4.0, 10


def check_params(c, iterations):
    if not (np.isfinite(c) and c >= 1.5):
        raise ValueError("c must be finite and >= 1.5")
    if not (isinstance(iterations, (int, np.integer)) and 0 <= iterations <= 64):
        raise ValueError("iterations must be an integer in 0..64")


def tukey(rho, tau):
    """(1 - (rho/tau)^2)^2 below tau, 0 at and beyond it."""
    q = rho / tau
    return np.where(rho < tau, (1.0 - q * q) ** 2, 0.0)


def point_norms(A, b, v):
    """|A_i v - b_i| of every point (rows 3i .. 3i+2)."""
    return np.linalg.norm((A @ v - b).reshape(-1, 3), axis=1)


def solve_velocity_robust(x, u, d, n, omega, t=None, variant="node", c=DEFAULT_C, iterations=DEFAULT_ITERATIONS):
    """-> dict(v, s, res, scale, rank, n_inliers, iterations, weights) as the C record defines them, plus v_lever (v'),
    tau of the last solve and rho_w, the norms its weights came from (for tests near the cut-off)."""
    if variant not in ("node", "exp", "sim"):
        raise ValueError("robust variant must be node, exp or sim")
    check_params(c, iterations)
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    N = len(x)
    A, B = build_system(x, u, n, omega, variant)
    d = float(np.asarray(d, dtype=np.float64).reshape(-1)[0])
    b = B * d
    vp, _, rank, s = np.linalg.lstsq(A, b, rcond=None)
    w = np.ones(N)
    scale, done, rho_w = 0.0, 0, np.zeros(N)
    for k in range(1, iterations + 1):
        if N == 0:
            break
        rho = point_norms(A, b, vp)
        m = (N - 1) // 2
        sigma = float(np.partition(rho.astype(np.float32), m)[m])
        tau = c * sigma
        if not (tau > 0 and np.isfinite(tau)):
            break
        w, rho_w = tukey(rho, tau), rho
        keep = np.repeat(w > 0, 3)
        sw = np.repeat(np.sqrt(w), 3)[keep]
        vp, _, rank, s = np.linalg.lstsq(A[keep] * sw[:, None], b[keep] * sw, rcond=None)
        scale, done = sigma, k
    rho = point_norms(A, b, vp) if N else np.zeros(0)
    res = float(np.sum(w * rho ** 2))
    v = vp.copy()
    if t is not None and variant != "node":
        v = vp - np.cross(np.asarray(omega, dtype=np.float64), np.asarray(t, dtype=np.float64))
    s3 = np.zeros(3)
    s3[:len(s)] = s
    return dict(v=v, s=s3, res=res, scale=scale, rank=int(rank), n_inliers=int(np.count_nonzero(w > 0)),
                iterations=done, weights=w, v_lever=vp, tau=c * scale, rho_w=rho_w)


def plain(x, u, d, n, omega, t=None, variant="node"):
    """iteration 0 alone: velocity_oracle.solve_lgs (v, res, rank, s)."""
    return solve_lgs(x, u, d, n, omega, t, variant)
