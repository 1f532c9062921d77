"""Cost of the robust velocity solve (ofb_frame_pairs_robust, ofb_tracker_set_robust; c = 4, 10 iterations): off and on,
alternated in one process so both see the same card state, median of the rounds.

  C2 shape    128 device-resident 1920x1080 pairs, 1000 features, ofb_frame_pairs_robust with rob NULL / set: ms per call
              (CUDA events)
  C5 shape    256 streams x 1280x720, 500 features, device-resident frames (borrowed), ms per fleet step (CUDA events;
              split solve, robust records in device memory)
  1080p       one stream, 500 features, device frames: per-frame latency (step + synchronise, p50)

Prints the card's name and power limit with the numbers.

    python tools/robust_overhead.py [rounds]
"""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ofb200  # noqa: E402
import synth  # noqa: E402

P = ofb200._lib.ptr


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                          # the timing itself does not need it
        q = "nvidia-smi unavailable (%s)" % e
    return q or torch.cuda.get_device_name(0)


def setup(w, h, n_streams, feat):
    pairs = [synth.make_pair(h, w, s, s) for s in range(min(n_streams, 8))]
    mo = pairs[0][2]
    a = torch.from_numpy(np.stack([pairs[s % len(pairs)][0] for s in range(n_streams)])).cuda()
    b = torch.from_numpy(np.stack([pairs[s % len(pairs)][1] for s in range(n_streams)])).cuda()
    imu = np.zeros(n_streams, ofb200._lib.IMU_DTYPE)
    for s in range(n_streams):
        m = pairs[s % len(pairs)][2]
        imu["d"][s], imu["n"][s], imu["w"][s] = m["d"], m["n"], m["w"]
    d_imu = torch.from_numpy(imu.view(np.uint8).reshape(-1).copy()).cuda()
    d_res = torch.zeros(n_streams * ofb200._lib.TRACK_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    d_rob = torch.zeros(n_streams * ofb200._lib.ROBUST_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    kw = dict(max_features=feat, min_features=feat // 2, topup="node", mask_radius=30, variant="node",
              principal=(mo["cx"], mo["cy"]), scaling=1.0 / mo["f"], flow_scaling=1.0 / (mo["f"] * mo["dt"]),
              feature_params=dict(qualityLevel=0.01, minDistance=10, blockSize=7))
    torch.cuda.synchronize()
    return a, b, d_imu, d_res, d_rob, kw


def tracker_steps(ctx, data, w, h, S, rob, borrow):
    a, b, d_imu, d_res, d_rob, kw = data
    trk = ofb200.StreamTracker(w, h, n_streams=S, borrow_frames=borrow, ctx=ctx, robust=rob, **kw)

    def step(k):
        ofb200._lib.check(ctx.lib.ofb_tracker_step_robust(trk.h, P(b if k & 1 else a), w, w * h, P(d_imu), None, P(d_res), None,
                                                          None, None, None, None, P(d_rob) if rob else None))
    return trk, step


def fleet(ctx, data, rob, steps=20):
    w, h, S = 1280, 720, 256
    trk, step = tracker_steps(ctx, data, w, h, S, rob, True)
    for k in range(6):
        step(k)
    ctx.sync()
    ctx.timer_start()
    for k in range(steps):
        step(k)
    ms = ctx.timer_stop() / steps
    rec = data[3].cpu().numpy().view(ofb200._lib.TRACK_RESULT_DTYPE)
    trk.close()
    return ms, float(rec["n_kept"].mean())


def single(ctx, data, rob):
    trk, step = tracker_steps(ctx, data, 1920, 1080, 1, rob, False)
    for k in range(20):
        step(k)
    ctx.sync()
    lat = []
    for k in range(300):
        t0 = time.perf_counter()
        step(k)
        ctx.sync()
        lat.append((time.perf_counter() - t0) * 1e6)
    trk.close()
    return float(np.percentile(lat, 50))


def pairs_setup(n=128, w=1920, h=1080, K=1000):
    pairs = [synth.make_pair(h, w, s, s) for s in range(8)]
    a = torch.from_numpy(np.stack([pairs[s % 8][0] for s in range(n)])).cuda()
    b = torch.from_numpy(np.stack([pairs[s % 8][1] for s in range(n)])).cuda()
    imu = np.zeros(n, ofb200._lib.IMU_DTYPE)
    for s in range(n):
        m = pairs[s % 8][2]
        imu["d"][s], imu["n"][s], imu["w"][s] = m["d"], m["n"], m["w"]
    mo = pairs[0][2]
    cfg = ofb200.make_pair_cfg(w, h, K, 0.01, 10, 7, (15, 15), 3, (3, 20, 0.03), variant="node", principal=(mo["cx"], mo["cy"]),
                               pos_scale=1.0 / mo["f"], flow_scale=1.0 / (mo["f"] * mo["dt"]))
    d_imu = torch.from_numpy(imu.view(np.uint8).reshape(-1).copy()).cuda()
    d_res = torch.zeros(n * ofb200._lib.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    d_rob = torch.zeros(n * ofb200._lib.ROBUST_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    return a, b, d_imu, d_res, d_rob, cfg, n, [p[2] for p in pairs]


ROBUST = ofb200._lib.RobustCfg(4.0, 10)


def c2(ctx, data, rob, calls=10):
    a, b, d_imu, d_res, d_rob, cfg, n, _ = data
    w, h = cfg.width, cfg.height

    def call():
        ofb200._lib.check(ctx.lib.ofb_frame_pairs_robust(ctx.h, C.byref(cfg), None, 0.0, 0, n, P(a), P(b), w, w * h, P(d_imu), None,
                                                         None, P(d_res), None, C.byref(ROBUST) if rob else None,
                                                         P(d_rob) if rob else None, None, None, None))
    for _ in range(3):
        call()
    ctx.sync()
    ctx.timer_start()
    for _ in range(calls):
        call()
    return ctx.timer_stop() / calls


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    ctx = ofb200.Context(0)
    print("card:", card())
    d2 = pairs_setup()
    d5 = setup(1280, 720, 256, 500)
    d1 = setup(1920, 1080, 1, 500)
    rows = {False: [], True: []}
    for r in range(rounds):
        for rob in ((False, True) if r % 2 == 0 else (True, False)):
            c5, kept = fleet(ctx, d5, rob)
            row = (c2(ctx, d2, rob), c5, single(ctx, d1, rob))
            rows[rob].append(row)
            print("round %d robust=%-5s  C2 call %.3f ms   C5 step %.3f ms   1080p latency p50 %.1f us   (C5: %.0f kept "
                  "points per stream)" % ((r, rob) + row + (kept,)), flush=True)
    for rob in (False, True):
        m = np.median(np.array(rows[rob]), axis=0)
        print("median robust=%-5s  C2 call %.3f ms   C5 step %.3f ms   1080p latency p50 %.1f us" % ((rob,) + tuple(m)))
    # what the C2 records say: iterations done and the share of points kept, per distinct scene
    e = d2[4].cpu().numpy().view(ofb200._lib.ROBUST_RESULT_DTYPE)
    res = d2[3].cpu().numpy().view(ofb200._lib.RESULT_DTYPE)
    print("C2 robust records, scenes 0-7: iterations", " ".join("%d" % e["iterations"][s] for s in range(8)),
          "  inlier share", " ".join("%.2f" % (e["n_inliers"][s] / max(res["n_tracked"][s], 1)) for s in range(8)))
    ctx.close()


if __name__ == "__main__":
    main()
