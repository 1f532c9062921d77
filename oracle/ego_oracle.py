"""CPU ORACLE (test infrastructure, NOT product code) of the ego-motion solve (include/ofb200.h, ofb_solve_ego_motion).

The reference's flow model (SURVEY App. A, velocity_oracle.build_system) with the gyro term moved to the left side:
for X = (x, y, 1), C = [X]x, P = |X|^2 I - X X^T = C^T C, u3 = (ux, uy, 0) and v' = v + w x t, every point gives

    A_i = [ wA C , d wb P ],   b_i = d wb C u3
    sim:        wA = n.X, wb = 1            (simulation.py:19-23)
    node / exp: wA = 1,   wb = 1 / (n.X)    (node:34-38, evaluate_exp.py:22-26)

Built literally, point by point, and solved with np.linalg.lstsq(A, b, rcond=None); then v = v' - w x t for exp / sim
(node has no lever arm, as velocity_oracle.solve_lgs).
"""
import numpy as np

from .velocity_oracle import _hat


def _weights(X, n, variant):
    nx = float(np.dot(n, X))
    if variant == "sim":
        return nx, 1.0
    if variant in ("node", "exp"):
        return 1.0, 1.0 / nx
    raise ValueError("ego-motion variant must be node, exp or sim")


def build_system(x, u, d, n, variant):
    """The stacked (3N x 6) A and (3N,) b."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    u = np.asarray(u, dtype=np.float64).reshape(-1, 2)
    n = np.asarray(n, dtype=np.float64).reshape(3)
    d = float(np.asarray(d, dtype=np.float64).reshape(-1)[0])
    N = len(x)
    A = np.zeros((3 * N, 6))
    b = np.zeros(3 * N)
    for i in range(N):
        X = np.array([x[i, 0], x[i, 1], 1.0])
        C = _hat(X)
        P = np.dot(X, X) * np.eye(3) - np.outer(X, X)
        wA, wb = _weights(X, n, variant)
        A[3 * i:3 * i + 3, :3] = wA * C
        A[3 * i:3 * i + 3, 3:] = d * wb * P
        b[3 * i:3 * i + 3] = d * wb * (C @ np.array([u[i, 0], u[i, 1], 0.0]))
    return A, b


def normal_blocks(x, u, d, n, variant):
    """A^T A and A^T b from the closed forms of the header, summed point by point."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    u = np.asarray(u, dtype=np.float64).reshape(-1, 2)
    n = np.asarray(n, dtype=np.float64).reshape(3)
    d = float(np.asarray(d, dtype=np.float64).reshape(-1)[0])
    M = np.zeros((6, 6))
    g = np.zeros(6)
    for i in range(len(x)):
        X = np.array([x[i, 0], x[i, 1], 1.0])
        C = _hat(X)
        r2 = np.dot(X, X)
        P = r2 * np.eye(3) - np.outer(X, X)
        wA, wb = _weights(X, n, variant)
        u3 = np.array([u[i, 0], u[i, 1], 0.0])
        M[:3, :3] += wA ** 2 * P
        M[:3, 3:] += -wA * d * wb * r2 * C
        M[3:, :3] += (-wA * d * wb * r2 * C).T
        M[3:, 3:] += d ** 2 * wb ** 2 * r2 * P
        g[:3] += wA * d * wb * (P @ u3)
        g[3:] += d ** 2 * wb ** 2 * r2 * (C @ u3)
    return M, g


def solve_ego_motion(x, u, d, n, t=None, variant="node"):
    """-> (v, omega, res, rank, s) as np.linalg.lstsq returns them (res is (1,) or (0,))."""
    A, b = build_system(x, u, d, n, variant)
    sol, res, rank, s = np.linalg.lstsq(A, b, rcond=None)
    vp, w = sol[:3], sol[3:]
    v = vp.copy()
    if t is not None and variant != "node":
        v = vp - np.cross(w, np.asarray(t, dtype=np.float64).reshape(3))
    return v, w, res, int(rank), s


def residual(x, u, d, n, variant, v_lever, omega):
    """sum of squared residuals of the stacked system at (v', omega)."""
    A, b = build_system(x, u, d, n, variant)
    r = A @ np.concatenate([v_lever, omega]) - b
    return float(r @ r)
