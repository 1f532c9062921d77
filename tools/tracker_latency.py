import os, sys, time, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import ofb200, synth
ctx = ofb200.Context(0)
w, h = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (640, 480)
NF = int(sys.argv[3]) if len(sys.argv) > 3 else 200
a, b, mo = synth.make_pair(h, w, 0, 0)
imu = np.zeros(1, ofb200._lib.IMU_DTYPE); imu["d"], imu["n"], imu["w"] = mo["d"], mo["n"], mo["w"]
kw = dict(max_features=NF, min_features=NF // 2, topup="node", mask_radius=30, variant="node", principal=(mo["cx"], mo["cy"]),
          scaling=1.0 / mo["f"], flow_scaling=1.0 / (mo["f"] * mo["dt"]), ctx=ctx)
P = ofb200._lib.ptr
da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
dimu = torch.from_numpy(imu.view(np.uint8).reshape(-1).copy()).cuda()
dres = torch.zeros(ofb200._lib.TRACK_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
for borrow in (False, True):
    trk = ofb200.StreamTracker(w, h, borrow_frames=borrow, **kw)
    def dstep(k):
        ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, P(db if k & 1 else da), w, w * h, P(dimu), None, P(dres), None, None, None, None))
    for k in range(10): dstep(k)
    ctx.sync()
    t0 = time.perf_counter()
    for k in range(400): dstep(k)
    t1 = time.perf_counter(); ctx.sync(); t2 = time.perf_counter()
    print("device frames borrow=%d: enqueue %.1f us/step, total %.1f us/step" % (borrow, (t1 - t0) / 400 * 1e6, (t2 - t0) / 400 * 1e6))
    lat = []
    for k in range(200):
        t0 = time.perf_counter(); dstep(k); ctx.sync(); lat.append((time.perf_counter() - t0) * 1e6)
    print("   sync each step: p50 %.1f us" % np.percentile(lat, 50))
    trk.close()
trk = ofb200.StreamTracker(w, h, **kw)
lat = []
for k in range(210):
    t0 = time.perf_counter(); r = trk.step(b if k & 1 else a, imu); lat.append((time.perf_counter() - t0) * 1e6)
print("host numpy frames via StreamTracker.step: p50 %.1f us" % np.percentile(lat[10:], 50), "graph info", trk.graph_info())
pa = torch.from_numpy(a).pin_memory(); pb = torch.from_numpy(b).pin_memory()
res = np.zeros(1, ofb200._lib.TRACK_RESULT_DTYPE)
lat = []
for k in range(210):
    t0 = time.perf_counter()
    ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, P(pb if k & 1 else pa), w, w * h, P(imu), None, P(res), None, None, None, None))
    lat.append((time.perf_counter() - t0) * 1e6)
print("pinned host frames, C call: p50 %.1f us" % np.percentile(lat[10:], 50))
trk.close()
