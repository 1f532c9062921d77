"""CPU ORACLE (test infrastructure, NOT product code) for stages 4-5 of the hot path.

Plain NumPy restatement of the reference's own arithmetic; every function cites the
reference lines it follows (paths relative to the original project's checkout):

* generate_test_data   numerical_simulation/simulation.py:7-12, velocity_measurment_node:25-29
* solve_lgs (3 variants) simulation.py:15-30 (S), velocity_measurment_node:30-42 (N),
                         flight_experiments/evaluate_exp.py:18-31 (E)
* r_tilde              of_library.py:365-386 (5-arg) and the older 4-arg homogeneous copy
                       sensor_precision_experiments/pixhawk_pure_IMU/of_library.py:365-384
* feasibility          simulation.py:108-120
* of_simulation trial  simulation.py:36-66   (noise is an INPUT here, so the GPU's Philox
                                               stream can be replayed trial by trial)
* feas_simulation trial simulation.py:70-104
* overlap              simulation.py:124-136
* solve_lgs_module     optical_flow_experiments/of_module.py:136-146 (the inline per-point-distance system)
* advect_points        simulation.py:496-499 (time-evolution sweep: points move by their own flow)
* sorting_scenario_live simulation.py:753-772 (the live sorting scenario: static / moving / parallel-plane points)
* pix_trans            of_library.py:31-43
* quaternion -> R, n   velocity_measurment_node:65-70
* body -> world        velocity_measurment_node:258

PARITY PIN: tests/test_oracle_velocity.py runs the reference's functions themselves
(AST-extracted and exec'd where OFB_REFERENCE_DIR names a checkout of it) against this
restatement, and tests/golden/velocity_golden.npz (made by tools/make_golden.py from the
reference functions) pins it everywhere else.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this.
"""
import numpy as np


def pix_trans(img_dim):
    """of_library.py:31-43 (Python-3 semantics: true division)."""
    tx = img_dim[0] / 2 if img_dim[0] % 2 == 0 else (img_dim[0] + 1) / 2
    ty = img_dim[1] / 2 if img_dim[1] % 2 == 0 else (img_dim[1] + 1) / 2
    return tx, ty


def _hat(X):
    """[X]x for X=(x,y,1): literal matrix at simulation.py:20 / node:35 / evaluate_exp.py:23."""
    return np.array([[0.0, -1.0, X[1]], [1.0, 0.0, -X[0]], [-X[1], X[0], 0.0]])


def generate_test_data(x, v, omega, d, n, t=None):
    """Forward flow model. simulation.py:7-12 (with lever arm t); node:25-29 (t=None)."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    v = np.asarray(v, dtype=np.float64)
    omega = np.asarray(omega, dtype=np.float64)
    n = np.asarray(n, dtype=np.float64)
    if t is not None:
        v = v + np.cross(omega, np.asarray(t, dtype=np.float64))
    flow = np.zeros((len(x), 3))
    for i in range(len(x)):
        X = np.array([x[i, 0], x[i, 1], 1.0])
        wx = np.cross(omega, X)
        flow[i] = np.dot(n, X) / d * (v - v[2] * X) + (wx - wx[2] * X)
    return flow[:, :2]


def build_system(x, u, n, omega, variant):
    """Stack the per-point 3x3 blocks exactly as the reference loops do.
    variant 'sim'  : rows (n.X)[X]x, rhs [X]x(u3+[X]x w)            simulation.py:19-23
    variant 'node' : rows [X]x,      rhs [X]x(u3+[X]x w)/(n.X)      node:34-38
    variant 'exp'  : same rows/rhs as 'node'                         evaluate_exp.py:22-26
    """
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    u = np.asarray(u, dtype=np.float64).reshape(-1, 2)
    n = np.asarray(n, dtype=np.float64)
    omega = np.asarray(omega, dtype=np.float64)
    N = len(x)
    A = np.zeros((3 * N, 3))
    B = np.zeros(3 * N)
    for i in range(N):
        X = np.array([x[i, 0], x[i, 1], 1.0])
        xh = _hat(X)
        b_i = xh @ (np.array([u[i, 0], u[i, 1], 0.0]) + xh @ omega)
        nx = float(np.dot(n, X))
        if variant == "sim":
            A[3 * i:3 * i + 3] = xh * nx
            B[3 * i:3 * i + 3] = b_i
        else:
            A[3 * i:3 * i + 3] = xh
            B[3 * i:3 * i + 3] = b_i / nx
    return A, B


def solve_lgs(x, u, d, n, omega, t=None, variant=None):
    """lstsq solve of the stacked system; returns (v, res, rank, s) for every variant
    (the reference returns subsets: node -> all four, exp -> (v,res), sim -> (v,res,s))."""
    if variant is None:
        variant = "node" if t is None else "sim"
    A, B = build_system(x, u, n, omega, variant)
    d = float(np.asarray(d, dtype=np.float64).reshape(-1)[0])
    v, res, rank, s = np.linalg.lstsq(A, B * d, rcond=None)
    if t is not None and variant != "node":
        v = v - np.cross(np.asarray(omega, dtype=np.float64), np.asarray(t, dtype=np.float64))
    return v, res, rank, s


def solve_lgs_module(x, u, n, dist):
    """optical_flow_experiments/of_module.py:136-146: A_i = [X_i]x / dist_i, B_i = A_i u_i / (n . X_i),
    np.linalg.lstsq(A, B) -> (v_obs, R, rank, s). x, u: (N,3) homogeneous rows (x, y, 1) / (ux, uy, 0), or (N,2)."""
    x = np.asarray(x, dtype=np.float64)
    u = np.asarray(u, dtype=np.float64)
    if x.shape[1] == 2:
        x = np.hstack([x, np.ones((len(x), 1))])
        u = np.hstack([u, np.zeros((len(u), 1))])
    n = np.asarray(n, dtype=np.float64)
    A = np.zeros((3 * len(x), 3))
    B = np.zeros(3 * len(x))
    for i in range(len(x)):
        ai = np.array([[0.0, -1.0, x[i, 1]], [1.0, 0.0, -x[i, 0]], [-x[i, 1], x[i, 0], 0.0]]) / dist[i]
        A[3 * i:3 * i + 3] = ai
        B[3 * i:3 * i + 3] = np.dot(ai, u[i]) / np.dot(n, x[i])
    v, res, rank, sv = np.linalg.lstsq(A, B, rcond=None)
    return v, res, rank, sv


def advect_points(data, linear_velocity, height, normal, translation, k):
    """simulation.py:496-499, k steps: data += generate_test_data(data, v, [0,0,0], h, n, t); h += v . n.
    -> (positions (k,N,2), heights (k,)) at the START of every step."""
    d = np.array(data, dtype=np.float64)
    h = float(height)
    pos, hs = [], []
    for _ in range(k):
        pos.append(d.copy()); hs.append(h)
        d = d + generate_test_data(d, linear_velocity, np.zeros(3), h, normal, translation)
        h = h + float(np.dot(linear_velocity, normal))
    return np.array(pos), np.array(hs)


def sorting_scenario_live(data, linear_velocity, angular_velocity, normal, translation, angles):
    """simulation.py:753-772: centred points, h = 2, v x 2.9 h; [0, N/5) static at 2 m, [N/5, 2(N/3)) at 1 m with their
    flows rotated by `angles` (one per row, the reference draws them from U(minang, 2 pi - minang)), [2(N/3), N) at 1 m.
    -> (data, true_flow, linear_velocity, height)."""
    d = np.array(data, dtype=np.float64)
    d[:, 0] = d[:, 0] - np.mean(d[:, 0])
    d[:, 1] = d[:, 1] - np.mean(d[:, 1])
    h = 2.0
    v = np.asarray(linear_velocity, dtype=np.float64) * 2.9 * h
    N = len(d)
    a, b = int(N / 5), 2 * int(N / 3)
    first = generate_test_data(d[:a], v, angular_velocity, h, normal, translation)
    second = generate_test_data(d[a:b], v, angular_velocity, h - 1, normal, translation)
    for i in range(len(second)):
        c, s_ = np.cos(angles[i]), np.sin(angles[i])
        second[i] = np.dot(np.array([[c, -s_], [s_, c]]), second[i])
    third = generate_test_data(d[b:], v, angular_velocity, h - 1, normal, translation)
    return d, np.vstack([first, second, third]), v, h


def r_tilde(x, u, n, v, dist=None):
    """of_library.py:365-386. With dist=None follows the 4-arg homogeneous copy
    (x,u are (N,3); d_i is not divided by dist)."""
    x = np.asarray(x, dtype=np.float64)
    u = np.asarray(u, dtype=np.float64)
    n = np.asarray(n, dtype=np.float64)
    v = np.asarray(v, dtype=np.float64)
    N = len(x)
    r = np.zeros(N)
    dd = np.ones(N)
    for i in range(N):
        if dist is None:
            X = x[i, :3]
            U = u[i, :3]
        else:
            X = np.append(x[i, :2], 1.0)
            U = np.append(u[i, :2], 0.0)
        vc = -np.cross(X, v)
        uc = np.cross(X, U)
        nv = np.linalg.norm(vc)
        nu = np.linalg.norm(uc)
        if dist is not None and nu * nv == 0:      # the 4-arg copy has no zero guard
            r[i] = 1
            continue
        r[i] = np.dot(vc, uc) / nu / nv
        if np.dot(X, n) < 0:
            r[i] = -r[i]
        dd[i] = np.dot(n, X) * nv / nu / (dist if dist is not None else 1.0)
    return r, dd


def feasibility(position, linear_velocity, flow, angular_velocity, translation, normal):
    """simulation.py:108-120 -> array (2,N): parallelity, length."""
    position = np.asarray(position, dtype=np.float64).reshape(-1, 2)
    flow = np.asarray(flow, dtype=np.float64).reshape(-1, 2)
    w = np.asarray(angular_velocity, dtype=np.float64)
    v = np.asarray(linear_velocity, dtype=np.float64)
    t = np.asarray(translation, dtype=np.float64)
    nrm = np.asarray(normal, dtype=np.float64)
    N = len(position)
    par = np.zeros(N)
    length = np.zeros(N)
    for i in range(N):
        X = np.array([position[i, 0], position[i, 1], 1.0])
        f1 = np.cross(X, v - np.cross(w, t))
        f2 = np.cross(X, np.array([flow[i, 0], flow[i, 1], 0.0]) - np.cross(w, X))
        n1 = np.linalg.norm(f1)
        n2 = np.linalg.norm(f2)
        par[i] = np.dot(f1, f2) / (n1 * n2)
        length[i] = n1 / n2 * np.dot(nrm, X)
    return np.array([par, length])


def quat_to_rot(qx, qy, qz, qw):
    """velocity_measurment_node:65-68, evaluate_exp.py:88-91."""
    return np.array([
        [1.0 - 2 * (qy ** 2 + qz ** 2), 2 * (qx * qy - qw * qz), 2 * (qw * qy + qx * qz)],
        [2 * (qx * qy + qw * qz), 1.0 - 2 * (qx ** 2 + qz ** 2), 2 * (qy * qz - qw * qx)],
        [2 * (qx * qz - qw * qy), 2 * (qw * qx + qy * qz), 1.0 - 2 * (qx ** 2 + qy ** 2)]])


def body_to_world(R, v_obs, omega, offset):
    """velocity_measurment_node:258: v_uav = R (v_obs - [w]x offset)."""
    w = np.asarray(omega, dtype=np.float64)
    wx = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    return np.asarray(R) @ (np.asarray(v_obs, dtype=np.float64) - wx @ np.asarray(offset, dtype=np.float64))


def of_trial(linear_velocity, angular_velocity, height, normal, translation, pos, true_flow,
             ang_vel_sig, translation_sig,
             d_omega, d_t, d_h, d_flow, d_pos):
    """One trial of of_simulation (simulation.py:39-64) with the additive noise given
    explicitly (d_* already scaled by their sigmas). The normal-vector noise is drawn but
    discarded by the reference (lines 45-46), so it has no input here. Returns (v_obs, R)."""
    v = np.asarray(linear_velocity, dtype=np.float64)
    w = np.asarray(angular_velocity, dtype=np.float64)
    n = np.asarray(normal, dtype=np.float64)
    t = np.asarray(translation, dtype=np.float64)
    pos = np.asarray(pos, dtype=np.float64)
    true_flow = np.asarray(true_flow, dtype=np.float64)
    w_err = w + d_omega
    t_err = t + d_t
    h_err = height + d_h
    flow_err = true_flow + d_flow
    pos_err = pos + d_pos
    n_err = n / np.linalg.norm(n)
    v_obs, _, _, s = solve_lgs(pos_err, flow_err, h_err, n_err, w_err, t_err, variant="sim")
    part = np.zeros(len(pos))
    for j in range(len(pos)):
        xp = np.array([pos[j, 0], pos[j, 1], 1.0])
        dxp = np.array([pos_err[j, 0], pos_err[j, 1], 1.0]) - xp
        ddotx = np.array([flow_err[j, 0] - true_flow[j, 0], flow_err[j, 1] - true_flow[j, 1], 0.0])
        v_e = (h_err - height) / height * np.dot(n, xp) + np.dot(n_err - n, xp) + np.dot(n, dxp)
        d_e = ddotx + np.cross(dxp, w) + np.cross(xp, w_err - w) + dxp
        part[j] = np.linalg.norm(np.cross(xp, v_e * v + height * d_e)) / np.amin(s)
    R = (np.sqrt(np.sum(part ** 2)) + np.linalg.norm(w) * translation_sig
         + ang_vel_sig * np.linalg.norm(t) + ang_vel_sig * translation_sig)
    return v_obs, float(R)


def of_simulation(iterations, rng, linear_velocity, angular_velocity, height, normal, translation,
                  pos, true_flow, ang_vel_sig, translation_sig, height_sig, flow_sig, position_sig,
                  normal_sig):
    """simulation.py:36-66 with the globals (iterations, true_flow) made explicit and the
    draws taken from `rng` (np.random.Generator or RandomState) in the reference's order."""
    pos = np.asarray(pos, dtype=np.float64)
    v_obs = np.zeros((iterations, 3))
    R = np.zeros(iterations)
    for i in range(iterations):
        d_omega = rng.normal(scale=ang_vel_sig, size=3)
        d_t = rng.normal(scale=translation_sig, size=3)
        d_h = float(rng.normal(scale=height_sig, size=1)[0])
        d_flow = rng.normal(scale=flow_sig, size=(len(pos), 2))
        d_pos = rng.normal(scale=position_sig, size=(len(pos), 2))
        rng.normal(scale=normal_sig, size=3)          # drawn, then discarded (line 45-46)
        v_obs[i], R[i] = of_trial(linear_velocity, angular_velocity, height, normal, translation, pos,
                                  true_flow, ang_vel_sig, translation_sig, d_omega, d_t, d_h, d_flow, d_pos)
    return v_obs, R


def rot_normal(normal, a1, a2):
    """simulation.py:89: Ry(a2) . Rx(a1) . normal."""
    ry = np.array([[np.cos(a2), 0, np.sin(a2)], [0, 1, 0], [-np.sin(a2), 0, np.cos(a2)]])
    rx = np.array([[1, 0, 0], [0, np.cos(a1), -np.sin(a1)], [0, np.sin(a1), np.cos(a1)]])
    return ry @ rx @ np.asarray(normal, dtype=np.float64)


def feas_trial(angular_velocity, height, normal, translation, pos, true_flow, true_vel,
               d_omega, d_t, d_h, d_flow, d_pos, d_vel, a1, a2):
    """One trial of feas_simulation (simulation.py:79-103), noise explicit.
    Returns 6 arrays (N,): backward par, backward dist, forward par, forward dist,
    backward residual norm, forward residual norm."""
    w = np.asarray(angular_velocity, dtype=np.float64)
    t = np.asarray(translation, dtype=np.float64)
    pos = np.asarray(pos, dtype=np.float64)
    w_err = w + d_omega
    t_err = t + d_t
    h_err = height + d_h
    flow_err = np.asarray(true_flow, dtype=np.float64) + d_flow
    pos_err = pos + d_pos
    vel_err = np.asarray(true_vel, dtype=np.float64) + d_vel
    n_err = rot_normal(normal, a1, a2)
    v_obs, _, _, _ = solve_lgs(pos_err, flow_err, h_err, n_err, w_err, t_err, variant="sim")
    bpar, bdist = feasibility(pos_err, v_obs, flow_err, w_err, t_err, n_err)
    fpar, fdist = feasibility(pos_err, vel_err, flow_err, w_err, t_err, n_err)
    N = len(pos)
    bres = np.zeros(N)
    fres = np.zeros(N)
    for j in range(N):
        X = np.array([pos_err[j, 0], pos_err[j, 1], 1.0])
        xh = _hat(X)
        b_i = xh @ (np.array([flow_err[j, 0], flow_err[j, 1], 0.0]) + xh @ w_err)
        Aj = xh * np.dot(n_err, X)
        bres[j] = np.linalg.norm(Aj @ v_obs - b_i)
        fres[j] = np.linalg.norm(Aj @ vel_err - b_i)
    return bpar, bdist, fpar, fdist, bres, fres


def overlap(data1, data2):
    """simulation.py:124-136."""
    binedge = np.histogram(np.hstack((data1, data2)), bins=100)[1]
    h1 = np.histogram(data1, bins=binedge)[0]
    h2 = np.histogram(data2, bins=binedge)[0]
    return np.sum(np.minimum(h1, h2))


# ---- counter-based RNG, restated independently of the CUDA code --------------------------
# Philox4x32-10 (Salmon et al., SC'11) + Box-Muller; the layout of counters is part of the
# product's documented contract (DESIGN.md "Monte-Carlo RNG contract").
_M0, _M1 = 0xD2511F53, 0xCD9E8D57
_W0, _W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32_10(counter, key):
    """counter: (...,4) uint32 array, key: (2,) uint32 -> (...,4) uint32."""
    c = np.array(counter, dtype=np.uint64) & 0xFFFFFFFF
    c0, c1, c2, c3 = [c[..., i].copy() for i in range(4)]
    k0, k1 = int(key[0]), int(key[1])
    for _ in range(10):
        p0 = c0 * _M0
        p1 = c2 * _M1
        hi0, lo0 = p0 >> 32, p0 & 0xFFFFFFFF
        hi1, lo1 = p1 >> 32, p1 & 0xFFFFFFFF
        n0 = (hi1 ^ c1 ^ k0) & 0xFFFFFFFF
        n1 = lo1
        n2 = (hi0 ^ c3 ^ k1) & 0xFFFFFFFF
        n3 = lo0
        c0, c1, c2, c3 = n0, n1, n2, n3
        k0 = (k0 + _W0) & 0xFFFFFFFF
        k1 = (k1 + _W1) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def normals_from_u32(r):
    """4 uint32 -> 4 standard normals by two Box-Muller pairs, in fp64.
    u = (r + 0.5) * 2^-32 in (0,1];  (z0,z1) = sqrt(-2 ln u0) * (cos, sin)(2 pi (u1 - 0.5))."""
    # the uniforms are formed in fp32 exactly as on the device: (float(r) + 0.5f) * 2^-32
    u = ((np.asarray(r, dtype=np.uint32).astype(np.float32) + np.float32(0.5))
         * np.float32(2.3283064365386963e-10)).astype(np.float64)
    rad0 = np.sqrt(-2.0 * np.log(u[..., 0]))
    rad1 = np.sqrt(-2.0 * np.log(u[..., 2]))
    a0 = 2.0 * np.pi * (u[..., 1] - 0.5)
    a1 = 2.0 * np.pi * (u[..., 3] - 0.5)
    return np.stack([rad0 * np.cos(a0), rad0 * np.sin(a0), rad1 * np.cos(a1), rad1 * np.sin(a1)], axis=-1)


def mc_normals(seed, step, trial_ids, n_points, n_extra_blocks=3):
    """Replay of the product's draw layout: for each trial, blocks b=0..(n_extra_blocks+N-1),
    counter = (trial_lo, trial_hi, b, step), key = (seed_lo, seed_hi). Returns
    array (len(trial_ids), n_extra_blocks + N, 4) of standard normals."""
    trial_ids = np.asarray(trial_ids, dtype=np.uint64)
    nb = n_extra_blocks + n_points
    ctr = np.zeros((len(trial_ids), nb, 4), dtype=np.uint64)
    ctr[..., 0] = (trial_ids & 0xFFFFFFFF)[:, None]
    ctr[..., 1] = (trial_ids >> 32)[:, None]
    ctr[..., 2] = np.arange(nb, dtype=np.uint64)[None, :]
    ctr[..., 3] = step
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint64)
    return normals_from_u32(philox4x32_10(ctr, key))
