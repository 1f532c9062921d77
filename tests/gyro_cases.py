"""Seeded scenes for the gyro prediction of the LK tracks (oracle/gyro_oracle.py, include/ofb200.h `ofb_gyro_predict`):
shared by tools/make_golden_gyro.py (cv2 -> tests/golden/gyro_golden.npz), tests/test_host_gyro.py and
tests/test_gpu_gyro.py.

rotation_scene: a textured plane seen by a camera that only rotates, frame 2 rendered exactly by the backward warp
p = K R^T K^-1 p' (synth.bilinear_sample). A point p of frame 1 lands at K R K^-1 p, which is what the predictor computes
for R = exp([w dt]x): the truth is known without a flow model. ROTATIONS are chosen so that plain LK with the default
frame_pairs parameters (15x15, 3 levels) loses most of the features at 1280x720.

rotation_pair: synth.warp_pair with a rotation-dominated motion (a large w and a small v), for the velocity solve."""
import numpy as np

import synth

W, H = 1280, 720
F = 0.8 * W
CX, CY = W / 2, H / 2
DT = 1.0 / 30.0
LK = ((15, 15), 3, (3, 20, 0.03))          # frame_pairs' defaults (make_pair_cfg)
N_FEATURES = 400
# gyro rates (rad/s, dt = 1/30 s): yaw / pitch of 4.5 / 3.6 rad/s move the image by 100-160 px per frame
ROTATIONS = {"yaw": np.array([0.6, 4.5, 0.9]), "pitch": np.array([-3.6, 0.9, -0.6])}


def rotation_matrix(r):
    """exp([r]x) (Rodrigues)"""
    t = np.linalg.norm(r)
    if t == 0:
        return np.eye(3)
    k = np.asarray(r, np.float64) / t
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(t) * Kx + (1 - np.cos(t)) * Kx @ Kx


def camera_matrix():
    return np.array([[F, 0, CX], [0, F, CY], [0, 0, 1.0]])


def rotation_scene(name, seed=0):
    """-> (prev, next, w): frame 2 of a pure rotation by exp([w DT]x) of frame 1 (texture seed `seed`)"""
    w = ROTATIONS[name]
    img = synth.texture(H, W, 300 + seed).astype(np.float64)
    K = camera_matrix()
    M = K @ rotation_matrix(w * DT).T @ np.linalg.inv(K)      # frame-2 pixel -> frame-1 pixel
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    X = M[0, 0] * xx + M[0, 1] * yy + M[0, 2]
    Y = M[1, 0] * xx + M[1, 1] * yy + M[1, 2]
    Z = M[2, 0] * xx + M[2, 1] * yy + M[2, 2]
    out = synth.bilinear_sample(img, X / Z, Y / Z)
    return img.astype(np.uint8), np.clip(np.round(out), 0, 255).astype(np.uint8), w


def true_positions(p0, w):
    """where the points p0 (N,2) of frame 1 are in frame 2 of rotation_scene (fp64), and whether they are inside it"""
    p = np.asarray(p0, np.float64).reshape(-1, 2)
    M = camera_matrix() @ rotation_matrix(np.asarray(w) * DT) @ np.linalg.inv(camera_matrix())
    q = np.c_[p, np.ones(len(p))] @ M.T
    t = q[:, :2] / q[:, 2:]
    inside = (t[:, 0] >= 0) & (t[:, 0] <= W - 1) & (t[:, 1] >= 0) & (t[:, 1] <= H - 1)
    return t, inside


def pinhole_kw():
    """make_pair_cfg keywords of the scenes' pinhole: x = (p - c) / F, u = dp / (F DT)"""
    return dict(principal=(CX, CY), pos_scale=1.0 / F, flow_scale=1.0 / (F * DT))


def rotation_pair(k, h=H, w=W):
    """-> (prev, next, motion dict): synth.warp_pair with synth.motion(k)'s v and n scaled to 8 px of translational
    flow and a gyro rate of about 3 rad/s"""
    img = synth.texture(h, w, 400 + k)
    mo = synth.motion(k, w, h, max_disp=8.0)
    rng = np.random.default_rng(500 + k)
    mo["w"] = rng.normal(0, 1, 3) * np.array([1.0, 1.0, 0.3])
    mo["w"] *= 3.0 / np.linalg.norm(mo["w"])
    return img, synth.warp_pair(img, mo), mo
