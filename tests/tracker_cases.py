"""Seeded scenarios for the feature-lifecycle (tracker) tests: shared by tools/make_golden_tracker.py (cv2 + the
reference's own functions -> tests/golden/tracker_golden.npz), tests/test_oracle_tracker.py (oracle vs golden)
and tests/test_gpu_tracker.py (CUDA path vs oracle). Each scenario follows one of the reference's loops:

  exp    flight_experiments/evaluate_exp.py:35-48, 97-113   unmasked top-up, lever arm solve
  node   velocity_measurment_node:93-107, 157-172, 238-250  masked top-up (radius 30), r_tilde gate (r <= T)
  module optical_flow_experiments/of_module.py:12-23, 83-86, 125-131  replace top-up, r >= T gate; two BGR streams,
         plus of_library.static_immobile (of_library.py:88-92)
"""
import numpy as np

import synth

W, H = 320, 240
F = 0.8 * W


def _sequence(seed, n_frames, step, rot_step, occlude=None):
    """Frames cut from one large texture along a drifting, slowly rotating window: features leave through the
    borders, and `occlude` = (frame, x, y, w, h) paints noise over a block from that frame on (lost features)."""
    pad = 96
    big = synth.texture(H + 2 * pad, W + 2 * pad, seed).astype(np.float64)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    rng = np.random.default_rng(500 + seed)
    frames = []
    for k in range(n_frames):
        a = rot_step * k
        c, s = np.cos(a), np.sin(a)
        sx = c * (xx - W / 2) + s * (yy - H / 2) + W / 2 + pad + step[0] * k
        sy = -s * (xx - W / 2) + c * (yy - H / 2) + H / 2 + pad + step[1] * k
        f = np.clip(np.round(synth.bilinear_sample(big, sx, sy)), 0, 255).astype(np.uint8)
        if occlude is not None and k >= occlude[0]:
            _, ox, oy, ow, oh = occlude
            f[oy:oy + oh, ox:ox + ow] = rng.integers(0, 256, (oh, ow), dtype=np.uint8)
        frames.append(f)
    return np.stack(frames)


def _imu(seed, n_frames, step, d_range, prior):
    """Per-frame sonar/IMU samples. prior = None or (sign, noise): a prior velocity for the r_tilde gate =
    sign * (the translation that explains the drift of the window at height d) + noise * |v| * N(0,1)^3 (the node
    passes its last published velocity, node:238; of_module.py:122,149 a Kalman prediction fed with -v_obs)."""
    rng = np.random.default_rng(900 + seed)
    out = []
    for _ in range(n_frames):
        n = np.array([rng.normal(0, 0.05), rng.normal(0, 0.05), 1.0])
        d = float(rng.uniform(*d_range))
        im = dict(d=d, n=n / np.linalg.norm(n), w=rng.normal(0, 0.05, 3), t=np.array([0.02, 0.0, 0.205]), v_prior=None)
        if prior is not None:
            v = np.array([-step[0] / F * d, -step[1] / F * d, 0.0])
            im["v_prior"] = prior[0] * v + prior[1] * np.linalg.norm(v) * rng.normal(0, 1, 3)
        out.append(im)
    return out


def _bgr(gray, seed):
    """A colour frame whose cv2 grey conversion is NOT the input (three different channel maps)."""
    g = gray.astype(np.int32)
    b = np.clip(g + 17 * np.sin(np.arange(g.shape[1]) / 9.0 + seed)[None, :], 0, 255)
    r = np.clip(255 - g // 2 + (np.arange(g.shape[0]) % 13)[:, None], 0, 255)
    return np.stack([b, g, r], axis=-1).astype(np.uint8)


SCENARIOS = {
    "exp": dict(
        streams=[dict(seed=11, step=(7.5, -3.25), rot=0.004, occlude=(4, 60, 50, 120, 90))],
        n_frames=8, bgr=False, d_range=(0.8, 3.0), prior=None,
        tracker=dict(max_features=40, min_features=36, topup="exp", variant="exp", scaling=1.0 / F,
                     feature_params=dict(qualityLevel=0.05, minDistance=10, blockSize=7),
                     lk_params=dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03)))),
    "node": dict(
        streams=[dict(seed=12, step=(-6.0, 4.5), rot=-0.003, occlude=(3, 150, 20, 100, 100))],
        n_frames=8, bgr=False, d_range=(0.8, 3.0), prior=(1.0, 0.25),
        tracker=dict(max_features=60, min_features=45, topup="node", mask_radius=30, variant="node", scaling=1.0 / F,
                     gate=("le", -0.97),
                     feature_params=dict(qualityLevel=0.1, minDistance=10, blockSize=12),
                     lk_params=dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03)))),
    "module": dict(
        streams=[dict(seed=13, step=(5.0, 6.0), rot=0.006, occlude=(2, 30, 120, 140, 80)),
                 dict(seed=14, step=(-8.0, -2.0), rot=0.0, occlude=None)],
        n_frames=7, bgr=True, d_range=(1.6, 3.0), prior=(-1.0, 0.25),
        tracker=dict(max_features=50, min_features=35, topup="module", variant="sim", scaling=1.0 / F,
                     gate=("ge", 0.97), max_speed=14.0, dummy_value=100.0,
                     feature_params=dict(qualityLevel=0.3, minDistance=20, blockSize=3),
                     lk_params=dict(winSize=(15, 15), maxLevel=3, criteria=(3, 10, 0.5)))),
}


def build(name):
    """-> (frames [stream][frame] (H,W) or (H,W,3) uint8, imu [stream][frame] dicts, tracker kwargs)"""
    sc = SCENARIOS[name]
    frames, imus = [], []
    for st in sc["streams"]:
        fr = _sequence(st["seed"], sc["n_frames"], st["step"], st["rot"], st["occlude"])
        if sc["bgr"]:
            fr = np.stack([_bgr(f, st["seed"]) for f in fr])
        frames.append(fr)
        imus.append(_imu(st["seed"], sc["n_frames"], st["step"], sc["d_range"], sc["prior"]))
    kw = dict(sc["tracker"], bgr=sc["bgr"])
    return frames, imus, kw


def run_oracle_tracker(make_tracker, frames, imus, teacher=None):
    """Runs one tracker per stream over the sequence. teacher (optional): per stream, per step, the point set to
    force BEFORE that step (None entries = leave alone). Returns per stream a list of per-step dicts."""
    out = []
    for s, (fr, im) in enumerate(zip(frames, imus)):
        trk = make_tracker()
        steps = []
        for k in range(len(fr)):
            if teacher is not None and teacher[s][k] is not None:
                trk.set_points(teacher[s][k])
            r = trk.step(fr[k], im[k]["d"], im[k]["n"], im[k]["w"], im[k]["t"], im[k]["v_prior"])
            r["pts"] = trk.pts.copy()
            steps.append(r)
        out.append(steps)
    return out


def pack(results, cap):
    """per-stream per-step dicts -> arrays for an .npz"""
    S, T = len(results), len(results[0])
    g = dict(pts=np.zeros((S, T, cap, 2), np.float32), kept_prev=np.zeros((S, T, cap, 2), np.float32),
             kept_next=np.zeros((S, T, cap, 2), np.float32), v=np.zeros((S, T, 3)), s=np.zeros((S, T, 3)),
             res=np.zeros((S, T)), rank=np.zeros((S, T), np.int32), solved=np.zeros((S, T), np.int32))
    for key in ("n_prev", "n_tracked", "n_kept", "n_added", "n_points"):
        g[key] = np.zeros((S, T), np.int32)
    for s in range(S):
        for k in range(T):
            r = results[s][k]
            g["pts"][s, k, :len(r["pts"])] = r["pts"]
            g["kept_prev"][s, k, :r["n_kept"]] = r["kept_prev"]
            g["kept_next"][s, k, :r["n_kept"]] = r["kept_next"]
            g["v"][s, k], g["s"][s, k], g["res"][s, k] = r["v"], r["s"], r["res"]
            g["rank"][s, k], g["solved"][s, k] = r["rank"], int(r["solved"])
            for key in ("n_prev", "n_tracked", "n_kept", "n_added", "n_points"):
                g[key][s, k] = r[key]
    return g


RANDOM_SEEDS = (21, 22, 23)


def random_case(seed):
    """A random drift / rotation / occlusion / parameter draw for one stream: -> (frames, imus, tracker kwargs)"""
    rng = np.random.default_rng(seed)
    T = 6
    step = tuple(rng.uniform(-8, 8, 2))
    occl = (int(rng.integers(2, 5)), int(rng.integers(0, 150)), int(rng.integers(0, 100)), 120, 100)
    frames = [_sequence(seed, T, step, float(rng.uniform(-0.005, 0.005)), occl)]
    mode = ["exp", "node", "module"][seed % 3]
    kw = dict(max_features=int(rng.integers(30, 80)), topup=mode, mask_radius=int(rng.integers(5, 40)),
              variant=["exp", "node", "sim"][seed % 3], scaling=1.0 / F,
              gate=None if seed % 2 else ("le", -0.9), max_speed=0.0 if seed % 3 else 12.0, dummy_value=-1.0,
              feature_params=dict(qualityLevel=float(rng.uniform(0.02, 0.2)), minDistance=int(rng.integers(5, 15)),
                                  blockSize=int(rng.choice([3, 5, 7, 12]))))
    kw["min_features"] = kw["max_features"] - int(rng.integers(3, 10))
    imus = [_imu(seed, T, step, (0.8, 3.0), (1.0, 0.2))]
    return frames, imus, kw


def cv2_engine(reference=True):
    """The same step operators backed by the REAL cv2 and the reference's own functions (AST-extracted by
    oracle/ref_loader.py; needs OFB_REFERENCE_DIR). reference=False keeps the oracle's restatements of the three
    arithmetic functions instead: solve_lgs and r_tilde (pinned to the reference's stored outputs by
    tests/test_oracle_velocity.py) and static_immobile (pinned by tests/test_oracle_tracker.py)."""
    import cv2
    from oracle import ref_loader, tracker_oracle

    class Cv2Operators(tracker_oracle.Engine):
        def good_features(self, img, max_corners, quality, min_distance, block_size, mask=None):
            return cv2.goodFeaturesToTrack(img, mask=mask, maxCorners=max_corners, qualityLevel=quality,
                                           minDistance=min_distance, blockSize=block_size)

        def pyrlk(self, prev, nxt, pts, win, max_level, criteria):
            return cv2.calcOpticalFlowPyrLK(prev, nxt, np.asarray(pts, np.float32).reshape(-1, 1, 2), None, winSize=win,
                                            maxLevel=max_level, criteria=criteria)

        def mask(self, points, radius, width, height):
            m = np.ones((height, width), np.uint8)                       # node:159
            for x, y in np.asarray(points).reshape(-1, 2):
                cv2.circle(m, (int(x), int(y)), radius, 0, cv2.FILLED)   # node:161
            return m

        def bgr2gray(self, bgr):
            return cv2.cvtColor(bgr, cv2.COLOR_BGR2GRAY)

    if not reference:
        return Cv2Operators()
    lib = ref_loader.of_library("root")
    solvers = {"node": ref_loader.node()["solve_lgs"], "exp": ref_loader.evaluate_exp()["solve_lgs"],
               "sim": ref_loader.simulation()["solve_lgs"]}

    class Cv2Engine(Cv2Operators):
        def solve(self, x, u, d, n, w, t, variant):
            if variant == "node":
                v, res, rank, s = solvers["node"](x, u, d, n, w)
            elif variant == "exp":
                v, res = solvers["exp"](x, u, d, n, w, t)
                rank, s = -1, np.zeros(3)
            else:
                v, res, s = solvers["sim"](x, u, d, n, w, t)
                rank = -1
            return v, res, rank, s

        def r_tilde(self, x, u, n, v, d):
            return lib["r_tilde"](x, u, n, v, d)[0]

        def static_immobile(self, new, old, maxspeed, distance, dummy):
            return lib["static_immobile"](np.asarray(new, np.float32).reshape(-1, 1, 2),
                                          np.asarray(old, np.float32).reshape(-1, 1, 2), maxspeed, distance, dummy)

    return Cv2Engine()
