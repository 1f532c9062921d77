"""Cost of the forward-backward check of the LK tracks (ofb_frame_pairs_fb, ofb_tracker_set_fb_check, ofb_pyrlk_fb): with
and without the check, alternated in one process so both see the same card state.

  C2 shape    128 device-resident 1920x1080 pairs, 1000 features, ofb_frame_pairs(_fb): ms per call (CUDA events)
  C5 shape    256 streams x 1280x720, 500 features, device-resident frames (borrowed), ms per fleet step (CUDA events)
  1080p       one stream, 500 features, device frames: per-frame latency (step + synchronise, p50)
  kernel      the fused kernel (ofb_pyrlk_fb) against two plain LK launches (ofb_pyrlk forward, then backward from its
              result) on the same 1080p pyramids and 1000 points x 128 calls, ms per call (CUDA events)

Threshold 1 px. Prints the card's name and power limit with the numbers.

    python tools/fb_overhead.py [rounds]
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
T = 1.0


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
    torch.cuda.synchronize()
    return a, b, d_imu, d_res, kw


def fleet(ctx, data, fb, steps=20):
    w, h, S = 1280, 720, 256
    a, b, d_imu, d_res, kw = data
    trk = ofb200.StreamTracker(w, h, n_streams=S, borrow_frames=True, ctx=ctx, fb_threshold=T if fb else None, **kw)

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
    rec = d_res.cpu().numpy().view(ofb200._lib.TRACK_RESULT_DTYPE)
    trk.close()
    return ms, float(rec["n_tracked"].mean()), float((rec["n_added"] > 0).mean())


def single(ctx, data, fb):
    w, h = 1920, 1080
    a, b, d_imu, d_res, kw = data
    trk = ofb200.StreamTracker(w, h, n_streams=1, ctx=ctx, fb_threshold=T if fb else None, **kw)

    def step(k):
        ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, P(b if k & 1 else a), w, w * h, P(d_imu), None, P(d_res), None, None,
                                                   None, None))
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
    torch.cuda.synchronize()
    return a, b, d_imu, d_res, cfg, n


def c2(ctx, data, fb, calls=10):
    a, b, d_imu, d_res, cfg, n = data
    w, h = cfg.width, cfg.height

    def call():
        ofb200._lib.check(ctx.lib.ofb_frame_pairs_fb(ctx.h, C.byref(cfg), None, T if fb else 0.0, n, P(a), P(b), w, w * h,
                                                     P(d_imu), None, None, P(d_res), None, None, None))
    for _ in range(3):
        call()
    ctx.sync()
    ctx.timer_start()
    for _ in range(calls):
        call()
    return ctx.timer_stop() / calls


def kernel_setup(ctx):
    a, b, _ = synth.make_pair(1080, 1920, 0, 0)
    pa, pb = ofb200.Pyramid(a, 3, ctx), ofb200.Pyramid(b, 3, ctx)
    p0 = ofb200.goodFeaturesToTrack(a, 1000, 0.01, 10, blockSize=7, ctx=ctx).reshape(-1, 2)
    n = len(p0)
    d = {k: torch.zeros(s, dtype=t, device="cuda") for k, s, t in
         (("p1", 2 * n, torch.float32), ("p0r", 2 * n, torch.float32), ("st", n, torch.uint8), ("st0", n, torch.uint8),
          ("err", n, torch.float32), ("err0", n, torch.float32), ("fb", n, torch.float32))}
    d["p0"] = torch.from_numpy(p0.copy()).cuda()
    torch.cuda.synchronize()
    return pa, pb, n, d


def kernels(ctx, data, fused, calls=128):
    pa, pb, n, d = data

    def call():
        if fused:
            ofb200._lib.check(ctx.lib.ofb_pyrlk_fb(ctx.h, pa.h, 0, pb.h, 0, P(d["p0"]), n, 15, 15, 3, 20, 0.03, 1e-4, T, P(d["p1"]),
                                                   P(d["st"]), P(d["err"]), P(d["fb"])))
        else:
            ofb200._lib.check(ctx.lib.ofb_pyrlk(ctx.h, pa.h, 0, pb.h, 0, P(d["p0"]), n, 15, 15, 3, 20, 0.03, 0, 1e-4, P(d["p1"]),
                                                P(d["st"]), P(d["err"])))
            ofb200._lib.check(ctx.lib.ofb_pyrlk(ctx.h, pb.h, 0, pa.h, 0, P(d["p1"]), n, 15, 15, 3, 20, 0.03, 0, 1e-4, P(d["p0r"]),
                                                P(d["st0"]), P(d["err0"])))
    for _ in range(5):
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
    d5 = setup(ctx, 1280, 720, 256, 500)
    d1 = setup(ctx, 1920, 1080, 1, 500)
    dk = kernel_setup(ctx)
    print("kernel comparison: %d points" % dk[2])
    rows = {False: [], True: []}
    for r in range(rounds):
        for fb in ((False, True) if r % 2 == 0 else (True, False)):
            c5, tracked, topups = fleet(ctx, d5, fb)
            row = (c2(ctx, d2, fb), c5, single(ctx, d1, fb), kernels(ctx, dk, fb))
            rows[fb].append(row)
            print("round %d fb=%-5s  C2 call %.3f ms   C5 step %.3f ms   1080p latency p50 %.1f us   LK %s %.4f ms   "
                  "(C5 last step: %.0f points tracked per stream, %.0f %% of the streams topped up)"
                  % ((r, fb) + row[:3] + ("fused" if fb else "two plain", row[3], tracked, 100 * topups)), flush=True)
    for fb in (False, True):
        m = np.median(np.array(rows[fb]), axis=0)
        print("median fb=%-5s  C2 call %.3f ms   C5 step %.3f ms   1080p latency p50 %.1f us   LK %s %.4f ms"
              % ((fb,) + tuple(m[:3]) + ("fused" if fb else "two plain", m[3])))
    ctx.close()


if __name__ == "__main__":
    main()
