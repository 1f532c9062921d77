"""Cost of the calibrated camera on the tracker step (ofb_tracker_set_camera): with and without a camera, alternated in
one process so both see the same card state.

  C5 shape    256 streams x 1280x720, 500 features, device-resident frames (borrowed), ms per fleet step (CUDA events)
  1080p       one stream, 500 features, device frames: per-frame latency (step + synchronise, p50) and the
              asynchronous rate (us per step over 400 enqueued steps), as tools/tracker_latency.py measures it

The camera is a k1 = -0.3 plumb_bob lens iterated 20 times (the velocity paths' default). Prints the card's name and
power limit with the numbers.

    python tools/camera_overhead.py [rounds]
"""
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
D = [-0.3, 0.12, 0.001, -0.0005, -0.02]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                          # the timing itself does not need it
        q = "nvidia-smi unavailable (%s)" % e
    return q or torch.cuda.get_device_name(0)


def setup(ctx, w, h, n_streams, feat):
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
    kw = dict(max_features=feat, min_features=feat // 2, topup="node", mask_radius=30, variant="node",
              principal=(mo["cx"], mo["cy"]), scaling=1.0 / mo["f"], flow_scaling=1.0 / (mo["f"] * mo["dt"]),
              feature_params=dict(qualityLevel=0.01, minDistance=10, blockSize=7))
    K = np.array([[mo["f"], 0.0, mo["cx"]], [0.0, mo["f"], mo["cy"]], [0.0, 0.0, 1.0]])
    cam = ofb200.make_camera(K, D, 1.0 / mo["dt"], 20)
    torch.cuda.synchronize()
    return a, b, d_imu, d_res, kw, cam


def tracker(ctx, w, h, n_streams, kw, cam, borrow):
    trk = ofb200.StreamTracker(w, h, n_streams=n_streams, borrow_frames=borrow, ctx=ctx, **kw)
    if cam is not None:
        trk.set_camera(cam)
    return trk


def fleet(ctx, data, with_cam, steps=20):
    w, h, S = 1280, 720, 256
    a, b, d_imu, d_res, kw, cam = data
    trk = tracker(ctx, w, h, S, kw, cam if with_cam else None, True)

    def step(k):
        ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, P(b if k & 1 else a), w, w * h, P(d_imu), None, P(d_res), None, None,
                                                   None, None))
    for k in range(6):
        step(k)
    ctx.sync()
    ctx.timer_start()
    for k in range(steps):
        step(k)
    ms = ctx.timer_stop() / steps
    trk.close()
    return ms


def single(ctx, data, with_cam):
    w, h = 1920, 1080
    a, b, d_imu, d_res, kw, cam = data
    trk = tracker(ctx, w, h, 1, kw, cam if with_cam else None, False)

    def step(k):
        ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, P(b if k & 1 else a), w, w * h, P(d_imu), None, P(d_res), None, None,
                                                   None, None))
    for k in range(20):
        step(k)
    ctx.sync()
    t0 = time.perf_counter()
    for k in range(400):
        step(k)
    ctx.sync()
    rate = (time.perf_counter() - t0) / 400 * 1e6
    lat = []
    for k in range(300):
        t0 = time.perf_counter()
        step(k)
        ctx.sync()
        lat.append((time.perf_counter() - t0) * 1e6)
    trk.close()
    return float(np.percentile(lat, 50)), rate


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    ctx = ofb200.Context(0)
    print("card:", card())
    d5 = setup(ctx, 1280, 720, 256, 500)
    d1 = setup(ctx, 1920, 1080, 1, 500)
    rows = {False: [], True: []}
    for r in range(rounds):
        for with_cam in ((False, True) if r % 2 == 0 else (True, False)):
            c5 = fleet(ctx, d5, with_cam)
            p50, rate = single(ctx, d1, with_cam)
            rows[with_cam].append((c5, p50, rate))
            print("round %d camera=%-5s  C5 step %.3f ms   1080p latency p50 %.1f us   1080p async %.1f us/step"
                  % (r, with_cam, c5, p50, rate), flush=True)
    for with_cam in (False, True):
        m = np.median(np.array(rows[with_cam]), axis=0)
        print("median camera=%-5s  C5 step %.3f ms   1080p latency p50 %.1f us   1080p async %.1f us/step"
              % (with_cam, m[0], m[1], m[2]))
    ctx.close()


if __name__ == "__main__":
    main()
