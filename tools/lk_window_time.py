"""Time of one LK launch (ofb_pyrlk) at a given window, on device-resident 1080p pyramids (maxLevel 3) and 1000
corners with criteria (3, 30, 0.01): ms per call over 128 calls (CUDA events), the median of `rounds` rounds. Windows
up to 16x15 run the register-resident kernel, larger ones the shared-memory kernel. Prints the card's name and power
limit with the numbers. OFB200_LIB selects the library build, so two builds can be compared by alternating runs.

    python tools/lk_window_time.py [rounds] [WxH ...]        (default: 3 rounds of 15x15, 21x21 and 64x64)
"""
import os
import subprocess
import sys

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


def main():
    args = sys.argv[1:]
    rounds = int(args.pop(0)) if args and args[0].isdigit() else 3
    wins = [tuple(int(v) for v in a.split("x")) for a in args] or [(15, 15), (21, 21), (64, 64)]
    ctx = ofb200.Context(0)
    a, b, _ = synth.make_pair(1080, 1920, 0, 0)
    pa, pb = ofb200.Pyramid(a, 3, ctx), ofb200.Pyramid(b, 3, ctx)
    p0 = ofb200.goodFeaturesToTrack(a, 1000, 0.01, 10, blockSize=7, ctx=ctx).reshape(-1, 2)
    n = len(p0)
    d0 = torch.from_numpy(p0.copy()).cuda()
    d1 = torch.zeros(2 * n, dtype=torch.float32, device="cuda")
    st = torch.zeros(n, dtype=torch.uint8, device="cuda")
    err = torch.zeros(n, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()

    def call(w, h):
        ofb200._lib.check(ctx.lib.ofb_pyrlk(ctx.h, pa.h, 0, pb.h, 0, P(d0), n, w, h, 3, 30, 0.01, 0, 1e-4, P(d1), P(st), P(err)))

    print("card:", card(), " library:", ofb200._lib.LIB_PATH, " points:", n)
    times = {w: [] for w in wins}
    for _ in range(rounds):
        for w in wins:
            for _ in range(5):
                call(*w)
            ctx.sync()
            ctx.timer_start()
            for _ in range(128):
                call(*w)
            times[w].append(ctx.timer_stop() / 128)
    for w in wins:
        print("LK %dx%d: %.4f ms per call (median of %d rounds: %s)"
              % (w[0], w[1], np.median(times[w]), rounds, " ".join("%.4f" % t for t in times[w])))
    ctx.close()


if __name__ == "__main__":
    main()
