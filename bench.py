#!/usr/bin/env python
"""bench.py -- headline measurement (BASELINE.json): 1080p frame-pairs/s (detect + LK flow + velocity solve) and
Monte-Carlo trials/s, plus the other three BASELINE configurations, all in the ONE JSON line of the default run.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (pyramids -> Shi-Tomasi -> pyramidal LK -> velocity solve) over one batch of
`--batch` consecutive synthetic 1080p frame pairs of one stream (BASELINE config 2: 1000 features, maxLevel 4).
  value      pairs/s with the frames already resident in HBM, CUDA events on the library's stream
  e2e        the same through the public Python API with pinned HOST frames: H2D of the frames and D2H of the results
             inside the timed region
  roofline   the dominant kernel: algorithmic bytes per launch / its CUDA-event duration vs the measured HBM copy
             bandwidth (MEASURED_PEAKS.json); `issue` = the same kernel against the warp-issue peak that actually bounds it
  cpu_baseline  cv2 4.13 goodFeaturesToTrack + calcOpticalFlowPyrLK (the reference's own un-vendored dependency) + the
             oracle port of the reference's Python solve_lgs, on the host cores
  mc         config 3: Monte-Carlo error sweep, 1e8 trials x 50 points, trial ranges sharded over the ranks, the merge
             all-reduce inside the timed region; fp32 and fp64 figures; CPU baseline = the oracle port of of_simulation
  c1 / c4    configs 1 and 4: 640x480 / 3840x2160 single-pair latency (p50), each with its CPU baseline
  c5         config 5: 256-stream 1280x720 fleet, stream-sharded over the ranks: pair path, device-resident lifecycle,
             lifecycle end to end from host frames; CPU baseline = one process per core over the streams
With N>1 every rank processes its own C2 batch (streams shard with no data-path collective): weak scaling; the C5
fleet and the Monte-Carlo job have a fixed total size: strong scaling.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, K_FEAT, MAX_LEVEL = 1920, 1080, 1000, 4
QUALITY, MIN_DIST, BLOCK = 0.01, 10.0, 7
WIN, CRIT = (15, 15), (3, 20, 0.03)
METRIC = "1080p frame-pairs/s (LK flow+velocity solve)"
MC_TOTAL, MC_POINTS = 100_000_000, 50
MC_AXES = ("flow_errors", "distance_error", "ang_vel_error", "normal_error", "translation_error", "orientation",
           "height", "point_position")
GEOM = {"c1": (640, 480, 200, 3), "c2": (W, H, K_FEAT, MAX_LEVEL), "c4": (3840, 2160, 5000, 5), "c5": (1280, 720, 500, 3)}
FLEET = 256
SOLVE_NOTE = ("solve_lgs = oracle port of the reference's Python loop with pre-allocated A, B (the reference grows them "
              "with np.append, ~4x slower at 1000 points: this baseline is faster than the verbatim reference)")


_T0 = time.time()


def log(msg):
    """progress on stderr (stdout carries only the JSON line)"""
    sys.stderr.write("[bench %6.1fs] %s\n" % (time.time() - _T0, msg))
    sys.stderr.flush()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of every leg (default: 10, and 50 samples / 400 resident steps in the C1 / C4 "
                         "latency legs, whose percentiles and per-frame means want more)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=128, help="frame pairs per step per GPU")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic pairs generated (tiled to the batch)")
    ap.add_argument("--mc-trials", type=int, default=MC_TOTAL)
    ap.add_argument("--no-mc", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C1 / C4 / C5 legs (kernel A-B runs)")
    ap.add_argument("--ref-pairs", type=int, default=16, help="pairs per step of the reference arm")
    ap.add_argument("--cpu-job", default=None, choices=["fleet", "mc"],
                    help="internal: run one multi-process CPU baseline in this (CUDA-free) process and print its JSON")
    ap.add_argument("--workload", default="all", choices=["all", "c1", "c2", "c4", "c5"],
                    help="all (default: every BASELINE configuration in one line) or a single configuration")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result records of the last timed C2 step (rank 0) as DIR/<field>.npy, float64")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    args.latency_samples, args.latency_reps = (50, 400) if args.steps is None else (args.steps, args.steps)
    if args.steps is None:
        args.steps = 10
    if args.dump_outputs and (args.impl == "reference" or args.workload not in ("all", "c2")):
        ap.error("--dump-outputs writes what the C2 headline path computed: use it with --workload all or c2")
    return args


def dump_outputs(out_dir, rec):
    """One float64 array per field of the result records (the integer fields are exact in float64). The inputs are
    seeded synthetic frames, so two builds run with the same arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    for name in rec.dtype.names:
        np.save(os.path.join(out_dir, name + ".npy"), rec[name].astype(np.float64))


def bind_near_gpu(index):
    """Multi-GPU hosts: run this rank (and first-touch its pinned frame buffers) on the CPUs NVML reports as closest to
    its GPU, so that the end-to-end copies do not cross the socket interconnect. Returns what happened (it goes into
    the JSON line: whether the affinity was applied decides how the 8-GPU end-to-end number is read)."""
    info = {"applied": False}
    try:
        before = sorted(os.sched_getaffinity(0))
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
        after = sorted(os.sched_getaffinity(0))
        info.update(applied=True, cpus_before=len(before), cpus_after=len(after), first_cpu=after[0], last_cpu=after[-1])
    except Exception as e:
        info["error"] = repr(e)[:120]
    return info


def numa_node_of(arr):
    """NUMA node of the first page of a (pinned) host array via move_pages(2) with a NULL node list; None when the call
    is not available in this container."""
    try:
        import ctypes
        libc = ctypes.CDLL("libc.so.6", use_errno=True)
        page = ctypes.c_void_p(arr.ctypes.data & ~4095)
        status = ctypes.c_int(-1)
        rc = libc.syscall(279, 0, ctypes.c_ulong(1), ctypes.byref(page), None, ctypes.byref(status), 0)   # __NR_move_pages
        return int(status.value) if rc == 0 and status.value >= 0 else None
    except Exception:
        return None


def make_data(distinct, rank, w=W, h=H, base=100):
    import synth
    return [synth.make_pair(h, w, stream_id=rank, pair_id=base * rank + i) for i in range(distinct)]


def imu_array(ofb200, pairs, batch):
    imu = np.zeros(batch, ofb200._lib.IMU_DTYPE)
    for i in range(batch):
        mo = pairs[i % len(pairs)][2]
        imu["d"][i], imu["n"][i], imu["w"][i] = mo["d"], mo["n"], mo["w"]
    return imu


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled every 2 ms from a
    thread (nvidia-smi, the recipe's tool, takes ~50 ms per query -- longer than a 10-step timed region; it is the
    fallback when NVML cannot be loaded)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index):
        self.index, self.rows, self.stop, self.t = index, [], threading.Event(), None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _run(self):
        while not self.stop.is_set():
            try:
                if self.nvml is not None:
                    sm = float(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
                    try:
                        mask = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    except Exception:
                        mask = int(self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    self.rows.append((sm, self.max, mask))
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    c = [x.strip() for x in out.strip().split(",")]
                    mask = 0
                    for (bit, _), val in zip(self.REASONS, c[2:6]):
                        if val.lower().startswith("active"):
                            mask |= bit
                    self.rows.append((float(c[0]), float(c[1]), mask))
            except Exception:
                pass
            self.stop.wait(0.002 if self.nvml is not None else 0.2)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(6)

    def summary(self):
        sm = [r[0] for r in self.rows]
        reasons = set()
        for r in self.rows:
            for bit, name in self.REASONS:
                if r[2] & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": max(r[1] for r in self.rows) if self.rows else None, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


WORKLOAD = ("C2: single 1920x1080 stream, consecutive frame pairs, 1000 features, maxLevel 4, "
            "detect+track+solve")


def stream_pair(pairs, k):
    """Pair k of the synthetic single stream (frame k, frame k+1): the stream alternates the base view with moved
    views, so even pairs are motion k/2 forward and odd pairs the way back (gyro rate negated)."""
    a, b, mo = pairs[(k // 2) % len(pairs)]
    if k % 2 == 0:
        return a, b, mo
    back = dict(mo); back["w"] = -np.asarray(mo["w"])
    return b, a, back


# ---- the reference's CPU path ---------------------------------------------------------------------------------
def cpu_one_pair(a, b, mo, feat, ml):
    """cv2 goodFeaturesToTrack + calcOpticalFlowPyrLK + the Python solve_lgs on one pair -> (velocity, split seconds, pts)"""
    import cv2
    from oracle import velocity_oracle as vo
    t1 = time.perf_counter()
    p = cv2.goodFeaturesToTrack(a, feat, QUALITY, MIN_DIST, blockSize=BLOCK)
    t2 = time.perf_counter()
    nxt, st, err = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=WIN, maxLevel=ml, criteria=CRIT)
    t3 = time.perf_counter()
    ok = st.ravel() == 1
    newp = nxt.reshape(-1, 2)[ok]
    x = (newp.astype(np.float64) - np.array([mo["cx"], mo["cy"]])) / mo["f"]
    u = (newp - p.reshape(-1, 2)[ok]).astype(np.float64) / (mo["f"] * mo["dt"])
    v = vo.solve_lgs(x, u, mo["d"], mo["n"], mo["w"], variant="node")[0]
    t4 = time.perf_counter()
    return v, (t2 - t1, t3 - t2, t4 - t3), p


def cpu_pair_path(get_pair, feat, ml, seconds, threads, max_pairs=None):
    """The reference's CPU path, pairs one after the other (as its loops run them), cv2 with `threads` threads."""
    import cv2
    cv2.setNumThreads(threads)
    done, t0, split = 0, time.perf_counter(), np.zeros(3)
    while True:
        a, b, mo = get_pair(done)
        _, sp, _ = cpu_one_pair(a, b, mo, feat, ml)
        split += sp
        done += 1
        el = time.perf_counter() - t0
        if (max_pairs and done >= max_pairs) or (not max_pairs and el >= seconds and done >= 3):
            break
    return done / el, done, (split / done * 1e3).tolist()


_FLEET_PAIRS = None


def _fleet_worker(idx):
    import cv2
    cv2.setNumThreads(1)
    a, b, mo = _FLEET_PAIRS[idx % len(_FLEET_PAIRS)]
    w, h, feat, ml = GEOM["c5"]
    cpu_one_pair(a, b, mo, feat, ml)
    return 1


def cpu_fleet(pairs, ncores, streams=FLEET):
    """BASELINE.md 3: the C5 CPU baseline is one process per core over the 256 streams (cv2 single-threaded in each)."""
    global _FLEET_PAIRS
    import multiprocessing as mp
    _FLEET_PAIRS = pairs
    with mp.get_context("fork").Pool(ncores) as pool:
        pool.map(_fleet_worker, range(ncores))                 # start the workers, import cv2, touch the frames
        t0 = time.perf_counter()
        n = sum(pool.map(_fleet_worker, range(streams), chunksize=max(1, streams // (4 * ncores))))
        el = time.perf_counter() - t0
    return n / el, n


_MC_ARGS = None


def _mc_worker(job):
    from oracle import velocity_oracle as vo
    seed, iters = job
    pos, tf = _MC_ARGS
    rng = np.random.RandomState(seed)
    t0 = time.perf_counter()
    vo.of_simulation(iters, rng, np.ones(3), np.ones(3), 1.0, np.array([0.0, 0, 1]), np.array([0.02, 0, 0.205]), pos, tf,
                     0.00071, 0.005, 0.01, 0.056 * np.sqrt(2) * 1.23, 0.056 * 1.23, 0.00065)
    return iters, time.perf_counter() - t0


def cpu_mc(ncores, total):
    """BASELINE.md 3: of_simulation (oracle port of simulation.py:36-66, same arithmetic per trial) on 1 core for >= 200
    trials and on all cores via multiprocessing (independent seeds), extrapolated linearly to the job size."""
    global _MC_ARGS
    import multiprocessing as mp
    from oracle import velocity_oracle as vo
    pts = np.load(os.path.join(ROOT, "tests", "golden", "points.npy"))
    d = np.array(pts, dtype=np.float64)
    d[:, 0] = (d[:, 0] - d[:, 0].mean()) * 1.27; d[:, 1] = (d[:, 1] - d[:, 1].mean()) * 0.93
    pos = d[:MC_POINTS]
    tf = vo.generate_test_data(pos, np.ones(3), np.ones(3), 1.0, [0, 0, 1], [0.02, 0, 0.205])
    _MC_ARGS = (pos, tf)
    n1, t1 = _mc_worker((1, 200))
    with mp.get_context("fork").Pool(ncores) as pool:
        pool.map(_mc_worker, [(100 + i, 2) for i in range(ncores)])
        t0 = time.perf_counter()
        res = pool.map(_mc_worker, [(200 + i, 100) for i in range(ncores)])
        el = time.perf_counter() - t0
    nall = sum(r[0] for r in res)
    one, allc = n1 / t1, nall / el
    return {"value": allc, "unit": "trials/s", "cores": ncores, "kind": "port", "value_1core": one,
            "sample": "oracle port of of_simulation (simulation.py:36-66, NumPy, %d points): %d trials on 1 core, %d trials on %d "
                      "cores (multiprocessing, independent seeds)" % (MC_POINTS, n1, nall, ncores),
            "extrapolated_seconds_for_job": {"trials": total, "one_core": total / one, "all_cores": total / allc,
                                             "note": "linear extrapolation, not run"}}


def cpu_job_subprocess(name, total=0, timeout=240):
    """The multi-process CPU baselines fork worker pools; forking THIS process (CUDA context, NCCL and NVML threads) is
    not safe, so they run in a fresh interpreter that never touches the GPU and report back through stdout."""
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-job", name, "--mc-trials", str(int(total))]
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    if out.returncode != 0:
        raise RuntimeError("cpu job %s failed: %s" % (name, out.stderr[-300:]))
    return json.loads(out.stdout.strip().split("\n")[-1])


def cpu_job_main(args):
    ncores = len(os.sched_getaffinity(0))
    if args.cpu_job == "fleet":
        w, h, feat, ml = GEOM["c5"]
        pairs = make_data(8, 0, w, h, base=1000)
        v, n = cpu_fleet(pairs, ncores)
        print(json.dumps({"value": v, "unit": "pairs/s", "cores": ncores, "kind": "port",
                          "sample": "%d streams, one pair each, one process per core (cv2 single-threaded per process); %s" % (n, SOLVE_NOTE)}))
    else:
        print(json.dumps(cpu_mc(ncores, args.mc_trials)))


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncores = len(os.sched_getaffinity(0))
    pairs = make_data(min(args.distinct, 4), 0)
    get = lambda k: stream_pair(pairs, k)
    for _ in range(args.warmup):
        cpu_pair_path(get, K_FEAT, MAX_LEVEL, 0, ncores, max_pairs=1)
    t0 = time.perf_counter()
    tot = 0
    for _ in range(args.steps):
        _, n, split = cpu_pair_path(get, K_FEAT, MAX_LEVEL, 0, ncores, max_pairs=args.ref_pairs)
        tot += n
    el = time.perf_counter() - t0
    val = tot / el
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/f32/f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "pairs_per_step": args.ref_pairs,
                       "note": "the CPU arm runs its pairs one after the other, so its rate does not depend on the pairs per step"},
            "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": ncores, "kind": "port",
                             "sample": "%d pairs: cv2 4.13 goodFeaturesToTrack+calcOpticalFlowPyrLK, all host threads; ms "
                                       "gftt/LK/solve = %s; %s" % (tot, [round(s, 1) for s in split], SOLVE_NOTE)},
            "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---- Monte-Carlo (config 3) -----------------------------------------------------------------------------------
def mc_workload(ofb200, trials_total):
    sim = ofb200.simulation
    pts = np.load(os.path.join(ROOT, "tests", "golden", "points.npy"))[:MC_POINTS]
    steps, pos, flow = [], [], []
    for name in MC_AXES:
        s, p, f = sim.build_sweep(name, pts)
        off = sum(len(q) for q in pos)
        for st in s:
            st.pos_offset += off
        steps += s; pos.append(p); flow.append(f)
    per_step = -(-trials_total // len(steps))
    return steps, np.vstack(pos), np.vstack(flow), per_step


def leg_mc(args, ofb200, torch, dist, rank, world, local):
    """1e8 trials x 50 points over 800 sweep steps; this rank's trial range; per-step sums stay on the device and are
    merged by ONE all-reduce (8 doubles per step) on the same stream, inside the timed region (CUDA events)."""
    sim = ofb200.simulation
    steps, pos, flow, per_step = mc_workload(ofb200, args.mc_trials)
    begin, count = sim.shard_range(per_step, rank, world)
    arr = sim._steps_array(steps)
    s = torch.cuda.current_stream()
    mctx = ofb200.Context(local, stream=s.cuda_stream)          # the library works on torch's stream: one timeline
    d_pos, d_flow = torch.from_numpy(pos).cuda(), torch.from_numpy(flow).cuda()
    d_sums = torch.zeros((len(steps), 8), dtype=torch.float64, device="cuda")

    def job(precision, want_R=True):
        if count > 0:
            sim.run_steps(arr, d_pos, d_flow, count, seed=1, trial_begin=begin, precision=precision, ctx=mctx, want_R=want_R,
                          sums_out=d_sums)
        else:
            d_sums.zero_()
        if dist is not None:
            dist.all_reduce(d_sums, op=dist.ReduceOp.SUM)

    def timed(precision, want_R=True, reps=3):
        out = []
        for _ in range(reps):
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s); job(precision, want_R); e1.record(s)
            e1.synchronize()
            out.append(e0.elapsed_time(e1))
        ms = float(np.median(out))
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
        return ms, out

    for _ in range(2):                       # warm-up at full size (clocks drop while the step descriptors are built)
        job("fp32")
    ms32, reps32 = timed("fp32")
    sums = d_sums.cpu().numpy().reshape(-1).view(ofb200._lib.MCSUMS_DTYPE).copy()
    ms32_nr, _ = timed("fp32", want_R=False)
    ms64, _ = timed("fp64", reps=2)
    mean, std, mR, n = sim.stats_from_sums(sums, steps)
    total = float(n.sum())
    flop = 140 * MC_POINTS + 300
    mctx.close()
    return {"metric": "MC trials/s", "value": total / (ms32 * 1e-3), "unit": "trials/s", "trials": total, "points": MC_POINTS,
            "steps": len(steps), "axes": list(MC_AXES), "ms": ms32, "ms_reps": [round(r, 3) for r in reps32],
            "value_fp64": total / (ms64 * 1e-3), "ms_fp64": ms64, "value_without_R": total / (ms32_nr * 1e-3),
            "scaling": "strong", "dtype": "f32 per-point arithmetic with f64 solve/statistics (`value`); f64 throughout (`value_fp64`, "
                                          "what the reference computes in)",
            "timed_region": "per-step sums left on the device + one all-reduce(sum) of %d x 8 doubles on the same stream, CUDA "
                            "events, max over ranks" % len(steps),
            "fp32_tflops_alg": total * flop / (ms32 * 1e-3) / 1e12, "fp32_peak_tflops": 74.4,
            "check_mean_v_step0": [round(float(x), 4) for x in mean[0]]}


# ---- single-pair latency (configs 1 and 4) --------------------------------------------------------------------
def leg_latency(args, ofb200, torch, ctx, name, rank):
    import ctypes as C
    w, h, feat, ml = GEOM[name]
    pairs = make_data(2, rank, w, h, base=1000)
    mo0 = pairs[0][2]
    cfg = ofb200.make_pair_cfg(w, h, feat, QUALITY, MIN_DIST, BLOCK, WIN, ml, CRIT, variant="node",
                               principal=(mo0["cx"], mo0["cy"]), pos_scale=1.0 / mo0["f"], flow_scale=1.0 / (mo0["f"] * mo0["dt"]))
    imu = imu_array(ofb200, pairs, 1)
    a = torch.from_numpy(pairs[0][0][None]).cuda(); b = torch.from_numpy(pairs[0][1][None]).cuda()
    d_imu = torch.from_numpy(imu.view(np.uint8).reshape(-1).copy()).cuda()
    d_res = torch.zeros(ofb200._lib.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    P = ofb200._lib.ptr

    def step():
        ofb200._lib.check(ctx.lib.ofb_frame_pairs(ctx.h, C.byref(cfg), 1, P(a), P(b), w, w * h, P(d_imu), None, None, P(d_res),
                                                  None, None, None))
    for _ in range(max(args.warmup, 5)):
        step()
    ctx.sync()
    lat = []
    for _ in range(args.latency_samples):
        ctx.timer_start(); step(); lat.append(ctx.timer_stop())
    res = np.zeros(1, ofb200._lib.RESULT_DTYPE); ctx.memcpy(res, d_res, res.nbytes)
    ctx.set_profile(True)
    for _ in range(3):
        step()
    ctx.set_profile(True)
    for _ in range(10):
        step()
    sms, calls = ctx.stage_times()
    ctx.set_profile(False)
    # the same pair from (pageable) host arrays through the public call, result read back: what a ROS callback sees
    ha, hb = pairs[0][0], pairs[0][1]
    for _ in range(5):
        ofb200.frame_pairs(ha[None], hb[None], imu[:1], cfg, ctx=ctx)
    e2e_lat = []
    for _ in range(args.latency_samples):
        t0 = time.perf_counter(); ofb200.frame_pairs(ha[None], hb[None], imu[:1], cfg, ctx=ctx); e2e_lat.append((time.perf_counter() - t0) * 1e3)
    # the same camera through the device-resident feature lifecycle: (i) what velocity_measurment_node's image callback
    # would run, one pageable host frame in, one result record out per call; (ii) resident frames, asynchronous calls
    kw = dict(max_features=feat, min_features=feat // 2, feature_params=dict(qualityLevel=QUALITY, minDistance=MIN_DIST, blockSize=BLOCK),
              lk_params=dict(winSize=WIN, maxLevel=ml, criteria=CRIT), topup="node", mask_radius=30, variant="node",
              principal=(mo0["cx"], mo0["cy"]), scaling=1.0 / mo0["f"], flow_scaling=1.0 / (mo0["f"] * mo0["dt"]), ctx=ctx)
    trk = ofb200.StreamTracker(w, h, **kw)
    for k in range(6):
        tres = trk.step(hb if k & 1 else ha, imu[:1])
    trk_lat = []
    for k in range(args.latency_samples):
        t0 = time.perf_counter(); tres = trk.step(hb if k & 1 else ha, imu[:1]); trk_lat.append((time.perf_counter() - t0) * 1e3)
    trk.close()
    trk = ofb200.StreamTracker(w, h, borrow_frames=True, **kw)
    d_tres = torch.zeros(ofb200._lib.TRACK_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    nrep = args.latency_reps             # (a short run is dominated by its first steps: 46 us per 640x480 frame over 50, 41 over 400)

    # (the argument objects are built once: at ~40 us per step the per-call conversion of three tensors to pointers shows)
    step_fn, chk = ctx.lib.ofb_tracker_step, ofb200._lib.check
    argsets = [(trk.h, P(f), w, w * h, P(d_imu), None, P(d_tres), None, None, None, None) for f in (a, b)]

    def rstep(k):
        chk(step_fn(*argsets[k & 1]))
    for k in range(8):
        rstep(k)
    ctx.sync()
    ctx.timer_start()
    for k in range(nrep):
        rstep(k)
    res_ms = ctx.timer_stop() / nrep
    trk.close()
    label = {"c1": "C1: 640x480, 200 features, maxLevel 3", "c4": "C4: 3840x2160, 5000 features, maxLevel 5"}[name]
    return {"metric": "%dx%d frame-pair latency p50 (detect+track+solve), ms" % (w, h), "value": float(np.percentile(lat, 50)),
            "unit": "ms", "p95": float(np.percentile(lat, 95)), "higher_is_better": False, "samples": len(lat),
            "config": {"workload": label + ", one resident pair per call (ofb_frame_pairs), CUDA events around each call"},
            "e2e": {"value": float(np.percentile(e2e_lat, 50)), "unit": "ms", "p95": float(np.percentile(e2e_lat, 95)),
                    "what": "ofb200.frame_pairs on pageable NumPy frames, result read back (host wall clock per call)",
                    "h2d_bytes_per_step": 2 * w * h, "d2h_bytes_per_step": int(res.nbytes)},
            "lifecycle_step": {"host_call_ms_p50": float(np.percentile(trk_lat, 50)), "host_call_ms_p95": float(np.percentile(trk_lat, 95)),
                               "resident_ms_per_frame": res_ms, "n_tracked": int(tres["n_tracked"][0]),
                               "solved": int(tres["flags"][0] & 1),
                               "what": "StreamTracker.step: one frame in, pyramid + LK from the kept frame + filter + solve; "
                                       "host_call = pageable NumPy frame in / record out, resident = device frames, asynchronous calls"},
            "stage_ms_serial": dict(zip(["pyramid", "eig_nms", "select", "lk", "solve"], [round(s / max(calls, 1), 4) for s in sms])),
            "check": {"n_tracked": int(res["n_tracked"][0]), "v": [round(float(x), 5) for x in res["v"][0]],
                      "truth": [round(float(x), 5) for x in pairs[0][2]["v"]]}}, pairs


# ---- the 256-stream fleet (config 5) --------------------------------------------------------------------------
def leg_fleet(args, ofb200, torch, dist, ctx, rank, world, local):
    import ctypes as C
    w, h, feat, ml = GEOM["c5"]
    distinct = 8
    B = FLEET // world + (1 if rank < FLEET % world else 0)
    pairs = make_data(distinct, rank, w, h, base=1000)
    mo0 = pairs[0][2]
    cfg = ofb200.make_pair_cfg(w, h, feat, QUALITY, MIN_DIST, BLOCK, WIN, ml, CRIT, variant="node",
                               principal=(mo0["cx"], mo0["cy"]), pos_scale=1.0 / mo0["f"], flow_scale=1.0 / (mo0["f"] * mo0["dt"]))
    imu = imu_array(ofb200, pairs, B)
    a = torch.from_numpy(np.stack([pairs[i % distinct][0] for i in range(B)])).cuda()
    b = torch.from_numpy(np.stack([pairs[i % distinct][1] for i in range(B)])).cuda()
    d_imu = torch.from_numpy(imu.view(np.uint8).reshape(-1).copy()).cuda()
    d_res = torch.zeros(B * ofb200._lib.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    P = ofb200._lib.ptr

    def maxr(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        ctx.sync(); torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def step():
        ofb200._lib.check(ctx.lib.ofb_frame_pairs(ctx.h, C.byref(cfg), B, P(a), P(b), w, w * h, P(d_imu), None, None, P(d_res),
                                                  None, None, None))
    for _ in range(args.warmup):
        step()
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        step()
    ms = maxr(ctx.timer_stop())
    res = np.zeros(B, ofb200._lib.RESULT_DTYPE); ctx.memcpy(res, d_res, res.nbytes)
    # the same fleet through the device-resident feature lifecycle (ofb_tracker_step, SURVEY 8f-2): one frame per stream
    # and step, point sets kept on the device, masked top-up when fewer than half the features survive
    kw = dict(max_features=feat, min_features=feat // 2, feature_params=dict(qualityLevel=QUALITY, minDistance=MIN_DIST, blockSize=BLOCK),
              lk_params=dict(winSize=WIN, maxLevel=ml, criteria=CRIT), topup="node", mask_radius=30, variant="node",
              principal=(mo0["cx"], mo0["cy"]), scaling=1.0 / mo0["f"], flow_scaling=1.0 / (mo0["f"] * mo0["dt"]))
    trk = ofb200.StreamTracker(w, h, n_streams=B, borrow_frames=True, ctx=ctx, **kw)
    d_tres = torch.zeros(B * ofb200._lib.TRACK_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")

    def tstep(k):
        ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, P(b if k & 1 else a), w, w * h, P(d_imu), None, P(d_tres), None, None,
                                                   None, None))
    for k in range(2 * max(args.warmup, 1)):
        tstep(k)
    barrier()
    l0 = ctx.launch_count()
    ctx.timer_start()
    for k in range(2 * args.steps):
        tstep(k)
    tms = maxr(ctx.timer_stop())
    tl = ctx.launch_count() - l0
    tres = np.zeros(B, ofb200._lib.TRACK_RESULT_DTYPE); ctx.memcpy(tres, d_tres, tres.nbytes)
    trk.close()
    lifecycle = {"value": FLEET * 2 * args.steps / (tms * 1e-3), "unit": "pairs/s", "ms_per_step": tms / (2 * args.steps),
                 "gpu_launches_per_step": tl / (2 * args.steps),
                 "what": "ofb_tracker_step: new frame -> pyramid -> LK from the kept frame -> status filter -> solve -> "
                         "(masked top-up when <= %d points survive); resident frames used in place (borrow_frames)" % (feat // 2),
                 "check": {"min_tracked": int(tres["n_tracked"].min()), "min_points": int(tres["n_points"].min()),
                           "solved": int((tres["flags"] & 1).sum()), "topups_last_step": int((tres["n_added"] > 0).sum())}}
    # BGR fleets (velocity_measurment_node:113 converts every frame): the conversion is fused into the first pyramid step
    # (grey level 0 written once, level 1 from the same read); OFB_BGR_FUSED=0 = the separate conversion kernel of round 1
    bgr_a = torch.stack([a, a, a], dim=-1).contiguous(); bgr_b = torch.stack([b, b, b], dim=-1).contiguous()
    trk = ofb200.StreamTracker(w, h, n_streams=B, bgr=True, ctx=ctx, **kw)

    def bstep(k):
        ofb200._lib.check(ctx.lib.ofb_tracker_step(trk.h, P(bgr_b if k & 1 else bgr_a), 3 * w, 3 * w * h, P(d_imu), None, P(d_tres),
                                                   None, None, None, None))
    bms = {}
    for mode in ("1", "0"):
        os.environ["OFB_BGR_FUSED"] = mode
        for k in range(2 * max(args.warmup, 1)):
            bstep(k)
        barrier()
        ctx.timer_start()
        for k in range(2 * args.steps):
            bstep(k)
        bms[mode] = maxr(ctx.timer_stop()) / (2 * args.steps)
    os.environ.pop("OFB_BGR_FUSED", None)
    tres_b = np.zeros(B, ofb200._lib.TRACK_RESULT_DTYPE); ctx.memcpy(tres_b, d_tres, tres_b.nbytes)
    trk.close()
    del bgr_a, bgr_b
    lifecycle["bgr_frames"] = {"value": FLEET / (bms["1"] * 1e-3), "unit": "pairs/s", "ms_per_step": bms["1"],
                               "ms_per_step_separate_conversion": bms["0"],
                               "dram_bytes_not_moved_per_frame": w * h,
                               "what": "the same lifecycle fed BGR8 frames: BGR->grey fused into the level-0 -> level-1 kernel (the grey "
                                       "level 0 is written once and not read back for level 1)",
                               "check": {"min_tracked": int(tres_b["n_tracked"].min()), "solved": int((tres_b["flags"] & 1).sum())}}
    # end to end: the fleet's frames arrive in (pinned) HOST memory every step. Four sub-fleets on four contexts (own
    # streams): the H2D copy of one sub-fleet overlaps the kernels of the others; every step's result records are read
    # back to the host. Bytes per step: B frames in, B result records out.
    NSUB = 4 if B >= 8 else 1
    bounds = [B * i // NSUB for i in range(NSUB + 1)]
    subs = []
    for i in range(NSUB):
        n_i = bounds[i + 1] - bounds[i]
        c_i = ofb200.Context(local)
        t_i = ofb200.StreamTracker(w, h, n_streams=n_i, ctx=c_i, **kw)
        ha_i = torch.from_numpy(np.stack([pairs[j % distinct][0] for j in range(bounds[i], bounds[i + 1])])).pin_memory()
        hb_i = torch.from_numpy(np.stack([pairs[j % distinct][1] for j in range(bounds[i], bounds[i + 1])])).pin_memory()
        dimu_i = torch.from_numpy(imu[bounds[i]:bounds[i + 1]].view(np.uint8).reshape(-1).copy()).cuda()
        dres_i = torch.zeros(n_i * ofb200._lib.TRACK_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        hres_i = torch.zeros(n_i * ofb200._lib.TRACK_RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
        subs.append((c_i, t_i, ha_i, hb_i, dimu_i, dres_i, hres_i))
    torch.cuda.synchronize()

    def estep(k):
        for c_i, t_i, ha_i, hb_i, dimu_i, dres_i, hres_i in subs:
            ofb200._lib.check(c_i.lib.ofb_tracker_step(t_i.h, P(hb_i if k & 1 else ha_i), w, w * h, P(dimu_i), None, P(dres_i),
                                                       None, None, None, None))
            ofb200._lib.check(c_i.lib.ofb_memcpy_async(c_i.h, P(hres_i), P(dres_i), hres_i.numel()))
        for sub in subs:
            sub[0].sync()
    for k in range(2 * max(args.warmup, 1)):
        estep(k)
    barrier()
    t0 = time.perf_counter()
    for k in range(2 * args.steps):
        estep(k)
    torch.cuda.synchronize()
    ems = maxr((time.perf_counter() - t0) * 1e3)
    eres = np.concatenate([sub[6].numpy().view(ofb200._lib.TRACK_RESULT_DTYPE) for sub in subs])
    for sub in subs:
        sub[1].close(); sub[0].close()
    lifecycle["e2e"] = {"value": FLEET * 2 * args.steps / (ems * 1e-3), "unit": "pairs/s", "ms_per_step": ems / (2 * args.steps),
                        "h2d_bytes_per_step": FLEET * w * h, "d2h_bytes_per_step": FLEET * ofb200._lib.TRACK_RESULT_DTYPE.itemsize,
                        "sub_fleets": NSUB, "check": {"min_tracked": int(eres["n_tracked"].min()), "solved": int((eres["flags"] & 1).sum())}}
    out = {"metric": "fleet 1280x720 frame-pairs/s (%d streams, detect+track+solve per pair)" % FLEET,
           "value": FLEET * args.steps / (ms * 1e-3), "unit": "pairs/s", "ms_per_step": ms / args.steps, "higher_is_better": True,
           "scaling": "strong", "lifecycle": lifecycle,
           "config": {"workload": "C5: %d streams x 1280x720, 500 features, maxLevel 3, stream-sharded over the ranks" % FLEET,
                      "streams_per_gpu": B},
           "check": {"min_tracked": int(res["n_tracked"].min())}}
    return out, pairs


def feature_tie_audit(ofb200, ctx, pairs, cfg):
    """Parity spot check of what was timed: the detector's feature lists of the distinct frames against
    cv2.goodFeaturesToTrack -- identical, or differing only by the documented float ties (tests/tie_rule.py)."""
    try:
        import cv2
        from tie_rule import explain_by_ties
    except Exception as e:
        return {"unavailable": repr(e)[:100]}
    frames = np.stack([p[0] for p in pairs]); nxt = np.stack([p[1] for p in pairs])
    imu = imu_array(ofb200, pairs, len(pairs))
    res, pp, pn, st = ofb200.frame_pairs(frames, nxt, imu, cfg, want_tracks=True, ctx=ctx)
    out = {"frames": len(pairs), "identical": 0, "tie_groups": 0, "unexplained": 0}
    for i, p in enumerate(pairs):
        ref = cv2.goodFeaturesToTrack(p[0], cfg.max_corners, cfg.quality, cfg.min_distance, blockSize=cfg.block_size)
        try:
            g = explain_by_ties(pp[i, :int(res["n_features"][i])], ref, cv2.cornerMinEigenVal(p[0], cfg.block_size))
            out["identical" if g == 0 else "tie_groups"] += 1 if g == 0 else g
        except AssertionError:
            out["unexplained"] += 1
    return out


def main():
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
    args = parse()
    if args.cpu_job:
        return cpu_job_main(args)
    if args.impl == "reference":
        return reference_arm(args)
    import torch
    import ofb200
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    affinity = bind_near_gpu(local)              # BEFORE any pinned allocation: first touch decides the NUMA node
    ctx = ofb200.Context(local)
    ncores = len(os.sched_getaffinity(0))

    def finish(line, cpu_jobs):
        """collectives are over: tear the group down, then rank 0 alone times the CPU baselines and prints the line"""
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        if rank != 0:
            return
        for job in cpu_jobs:
            log("cpu baseline: " + getattr(job, "__name__", "job"))
            try:
                job()
            except Exception as e:       # cv2 missing on the box, fork refused, ...
                line.setdefault("cpu_baseline_errors", []).append(repr(e)[:160])
        print(json.dumps(line))

    # ---- single-configuration runs (kept for quick looks; the default line holds all of them) ----
    if args.workload in ("c1", "c4"):
        out, pairs = leg_latency(args, ofb200, torch, ctx, args.workload, rank)
        w, h, feat, ml = GEOM[args.workload]

        def cpu():
            if not args.no_cpu:
                v, n, split = cpu_pair_path(lambda k: pairs[k % len(pairs)], feat, ml, 3.0, ncores)
                out["cpu_baseline"] = {"value": 1e3 / v, "unit": "ms per pair", "cores": ncores, "kind": "port",
                                       "sample": "%d pairs, cv2 4.13 gftt+pyrLK with %d threads; ms gftt/LK/solve = %s; %s" %
                                                 (n, ncores, [round(x, 2) for x in split], SOLVE_NOTE)}
        out["n_gpus"] = 1
        return finish(out, [cpu])
    if args.workload == "c5":
        out, pairs = leg_fleet(args, ofb200, torch, dist, ctx, rank, world, local)
        out["n_gpus"] = world

        def cpu():
            if not args.no_cpu:
                out["cpu_baseline"] = cpu_job_subprocess("fleet")
        return finish(out, [cpu])

    # ---- config 2: the headline ----
    B = args.batch
    pairs = make_data(args.distinct, rank)
    mo0 = pairs[0][2]
    cfg = ofb200.make_pair_cfg(W, H, K_FEAT, QUALITY, MIN_DIST, BLOCK, WIN, MAX_LEVEL, CRIT, variant="node",
                               principal=(mo0["cx"], mo0["cy"]), pos_scale=1.0 / mo0["f"],
                               flow_scale=1.0 / (mo0["f"] * mo0["dt"]))
    imu = imu_array(ofb200, pairs, B)
    # host frames in pinned memory (e2e path) and a resident copy in HBM (kernel path)
    h_prev = ctx.pinned_array((B, H, W), np.uint8)
    h_next = ctx.pinned_array((B, H, W), np.uint8)
    for i in range(B):
        h_prev[i], h_next[i] = pairs[i % len(pairs)][0], pairs[i % len(pairs)][1]
    d_prev = torch.empty((B, H, W), dtype=torch.uint8, device="cuda")
    d_next = torch.empty((B, H, W), dtype=torch.uint8, device="cuda")
    ctx.memcpy(d_prev, h_prev, h_prev.nbytes)
    ctx.memcpy(d_next, h_next, h_next.nbytes)
    d_imu = torch.from_numpy(imu.view(np.uint8).reshape(-1).copy()).cuda()
    d_res = torch.zeros(B * ofb200._lib.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    # "single stream" (BASELINE config 2): B+1 consecutive frames, pair k = (frame k, frame k+1). The synthetic stream
    # alternates the base view with a moved view (even pairs: motion k/2 forward, odd pairs: the way back), so every
    # consecutive pair is a small, known camera motion.
    h_seq = ctx.pinned_array((B + 1, H, W), np.uint8)
    imu_seq = np.zeros(B, ofb200._lib.IMU_DTYPE)
    for k in range(B):
        fa, fb, mo = stream_pair(pairs, k)
        h_seq[k] = fa
        if k == B - 1:
            h_seq[B] = fb
        imu_seq["d"][k], imu_seq["n"][k], imu_seq["w"][k] = mo["d"], mo["n"], mo["w"]
    d_seq = torch.empty((B + 1, H, W), dtype=torch.uint8, device="cuda")
    ctx.memcpy(d_seq, h_seq, h_seq.nbytes)
    d_imu_seq = torch.from_numpy(imu_seq.view(np.uint8).reshape(-1).copy()).cuda()
    torch.cuda.synchronize()
    lib, C = ctx.lib, __import__("ctypes")
    P = W * H

    def step_independent():
        ofb200._lib.check(lib.ofb_frame_pairs(ctx.h, C.byref(cfg), B, ofb200._lib.ptr(d_prev), ofb200._lib.ptr(d_next), W,
                                              W * H, ofb200._lib.ptr(d_imu), None, None, ofb200._lib.ptr(d_res), None, None,
                                              None))

    def step_resident():
        ofb200._lib.check(lib.ofb_frame_pairs(ctx.h, C.byref(cfg), B, d_seq.data_ptr(), d_seq.data_ptr() + P, W,
                                              W * H, ofb200._lib.ptr(d_imu_seq), None, None, ofb200._lib.ptr(d_res), None, None,
                                              None))

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def maxr(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # the GPU idled (clocks down) while the synthetic frames were generated on the host: spin it up first,
    # then the W warm-up steps of the contract
    for _ in range(30):
        step_resident()
    ctx.sync()
    for _ in range(args.warmup):
        step_resident()
    barrier()
    l0 = ctx.launch_count()
    clk = ClockSampler(local)          # samples until the end-to-end loop ends: every sample is taken under load
    clk.__enter__()
    ctx.timer_start()
    for _ in range(args.steps):
        step_resident()
    ms = ctx.timer_stop()
    launches = ctx.launch_count() - l0
    barrier()
    ms = maxr(ms)
    log("c2 resident timed")
    value = world * B * args.steps / (ms * 1e-3)
    # correctness of what was timed: results must be plausible velocities (forward pairs have an exact truth)
    res = np.zeros(B, ofb200._lib.RESULT_DTYPE)
    ctx.memcpy(res, d_res, res.nbytes)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)
    verr = max(np.abs(res["v"][k] - pairs[(k // 2) % len(pairs)][2]["v"]).max() for k in range(0, B, 2))
    tracked = int(res["n_tracked"].min())
    # the same number of pairs as independent (prev, next) buffers: both frames of every pair uploaded / pyramided
    for _ in range(args.warmup):
        step_independent()
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        step_independent()
    ms_ind = ctx.timer_stop()
    barrier()
    ms_ind = maxr(ms_ind)
    res_i = np.zeros(B, ofb200._lib.RESULT_DTYPE)
    ctx.memcpy(res_i, d_res, res_i.nbytes)
    verr_i = max(np.abs(res_i["v"][i] - pairs[i % len(pairs)][2]["v"]).max() for i in range(B))

    # steady state of the callers (they re-detect only when features run low: evaluate_exp.py:105-107, node:157-163):
    # track+solve of given points -- pyramid, LK and solve, no detection. The points are the detector's output for
    # the same stream, left on the device by one detect pass.
    d_pts = torch.zeros((B, K_FEAT, 2), dtype=torch.float32, device="cuda")
    ofb200._lib.check(lib.ofb_frame_pairs(ctx.h, C.byref(cfg), B, d_seq.data_ptr(), d_seq.data_ptr() + P, W, W * H,
                                          ofb200._lib.ptr(d_imu_seq), None, None, ofb200._lib.ptr(d_res), d_pts.data_ptr(), None, None))
    ctx.sync()
    res_t = np.zeros(B, ofb200._lib.RESULT_DTYPE)
    ctx.memcpy(res_t, d_res, res_t.nbytes)
    d_nin = torch.from_numpy(res_t["n_features"].astype(np.int32)).cuda()
    cfg_t = ofb200.make_pair_cfg(W, H, K_FEAT, QUALITY, MIN_DIST, BLOCK, WIN, MAX_LEVEL, CRIT, variant="node",
                                 principal=(mo0["cx"], mo0["cy"]), pos_scale=1.0 / mo0["f"],
                                 flow_scale=1.0 / (mo0["f"] * mo0["dt"]), detect=False)
    torch.cuda.synchronize()

    def step_track():
        ofb200._lib.check(lib.ofb_frame_pairs(ctx.h, C.byref(cfg_t), B, d_seq.data_ptr(), d_seq.data_ptr() + P, W, W * H,
                                              ofb200._lib.ptr(d_imu_seq), d_pts.data_ptr(), d_nin.data_ptr(),
                                              ofb200._lib.ptr(d_res), None, None, None))

    for _ in range(args.warmup):
        step_track()
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        step_track()
    ms_trk = ctx.timer_stop()
    barrier()
    ms_trk = maxr(ms_trk)
    res_k = np.zeros(B, ofb200._lib.RESULT_DTYPE)
    ctx.memcpy(res_k, d_res, res_k.nbytes)
    track_solve = {"value": world * B * args.steps / (ms_trk * 1e-3), "unit": "pairs/s", "ms_per_step": ms_trk / args.steps,
                   "max_abs_v_diff_vs_detect_mode": float(np.abs(res_k["v"] - res_t["v"]).max()),
                   "note": "track+solve of given points (pyramid, LK, solve; no detection), resident frames"}

    # the same single stream the way the reference's loops consume it: one frame after the other through the
    # device-resident feature lifecycle (ofb_tracker_step: pyramid of the new frame, LK from the kept frame, status
    # filter, solve, masked top-up when fewer than half the features survive). Sequential by construction (frame k+1
    # starts from the points frame k produced), so this is a latency chain, not a batch.
    trk = ofb200.StreamTracker(W, H, max_features=K_FEAT, min_features=K_FEAT // 2,
                               feature_params=dict(qualityLevel=QUALITY, minDistance=MIN_DIST, blockSize=BLOCK),
                               lk_params=dict(winSize=WIN, maxLevel=MAX_LEVEL, criteria=CRIT), topup="node", mask_radius=30,
                               variant="node", principal=(mo0["cx"], mo0["cy"]), scaling=1.0 / mo0["f"],
                               flow_scaling=1.0 / (mo0["f"] * mo0["dt"]), borrow_frames=True, ctx=ctx)
    d_tres = torch.zeros((B + 1) * ofb200._lib.TRACK_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    isz, rsz = ofb200._lib.IMU_DTYPE.itemsize, ofb200._lib.TRACK_RESULT_DTYPE.itemsize

    import ctypes as _C
    life_args = [(trk.h, _C.c_void_p(d_seq.data_ptr() + k * P), W, P, _C.c_void_p(d_imu_seq.data_ptr() + max(k - 1, 0) * isz), None,
                  _C.c_void_p(d_tres.data_ptr() + k * rsz), None, None, None, None) for k in range(B + 1)]
    life_fn, life_chk = lib.ofb_tracker_step, ofb200._lib.check

    def step_lifecycle():
        for a_ in life_args:                # frame k of the stream; pair k-1 = (frame k-1, frame k)
            life_chk(life_fn(*a_))
    for _ in range(max(args.warmup // 2, 1)):
        step_lifecycle()
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        step_lifecycle()
    ms_life = ctx.timer_stop()
    barrier()
    ms_life = maxr(ms_life)
    res_l = np.zeros(B + 1, ofb200._lib.TRACK_RESULT_DTYPE)
    ctx.memcpy(res_l, d_tres, res_l.nbytes)
    trk.close()
    lifecycle = {"value": world * (B + 1) * args.steps / (ms_life * 1e-3), "unit": "frames/s",
                 "ms_per_frame": ms_life / (args.steps * (B + 1)), "min_tracked": int(res_l["n_tracked"][1:].min()),
                 "topups_per_pass": int((res_l["n_added"][1:] > 0).sum()),
                 "max_abs_v_error_vs_truth": float(max(np.abs(res_l["v"][k + 1] - pairs[(k // 2) % len(pairs)][2]["v"]).max()
                                                       for k in range(0, B, 2) if res_l["flags"][k + 1] & 1)),
                 "note": "one stream, frame after frame through ofb_tracker_step (sequential dependency: a latency chain)"}

    # per-stage durations (CUDA events between the kernels of the same call path)
    ctx.set_profile(True)
    for _ in range(3):                     # the profiled call path sizes its own scratch on first use
        step_resident()
    ctx.set_profile(True)                  # resets the accumulated stage times
    for _ in range(args.steps):
        step_resident()
    stage_ms, calls = ctx.stage_times()
    ctx.set_profile(False)
    stage_ms = [s / max(calls, 1) for s in stage_ms]
    skeys = ["pyramid", "eig_nms", "select", "lk", "solve"]
    names = ["pyramid(pyr_down_kernel x%d levels)" % MAX_LEVEL, "eig_march_kernel<false,7>", "select_kernel",
             "lk_track_fast2_kernel", "pair_solve_kernel"]
    g = sum(((W + (1 << l) - 1) >> l) * ((H + (1 << l) - 1) >> l) for l in range(1, MAX_LEVEL + 1))
    nfeat = float(res["n_features"].mean())
    nlev = MAX_LEVEL + 1
    alg = [(P + g) * (B + 1),
           (P + 8 * 4 * nfeat) * B,
           (8 * 4 * nfeat + 8 * nfeat) * B,
           (21 * nfeat + nfeat * nlev * ((WIN[0] + 3) * (WIN[1] + 3) + (WIN[0] + 1) * (WIN[1] + 1))) * B,
           (17 * nfeat + 80) * B]
    dom = int(np.argmax(stage_ms))
    # DRAM bytes and warp instructions per image of each stage's kernel(s) from the committed ncu --set full capture
    tj = {}
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    traffic = float(tj[skeys[dom]]["dram_bytes_per_pair"]) * B if tj.get(skeys[dom]) else None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    ach = alg[dom] / (stage_ms[dom] * 1e-3) / 1e9
    roofline = {"kernel": names[dom], "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "peak_source": "measured" if peaks else "fallback",
                "stage_ms": dict(zip(skeys, [round(s, 4) for s in stage_ms])),
                "stage_gbs": dict(zip(skeys, [round(a / (s * 1e-3) / 1e9, 2) if s > 0 else None for a, s in zip(alg, stage_ms)])),
                "issue_active_pct_ncu": tj.get(skeys[dom], {}).get("issue_active_pct"), "issue": None,
                "note": "the two dominant kernels (lambda_min+NMS, LK) are warp-issue bound (ncu issue-active 73 % / 80 %), "
                        "not HBM bound: their DRAM traffic is the image read once; see DESIGN.md section 6"}

    # end to end through the public API: pinned host frames in, host results out, every step
    def e2e_run(fn):
        for _ in range(max(1, args.warmup // 2)):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r_ = fn()
        dt = time.perf_counter() - t0
        if dist is not None:
            t_ = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            dt = float(t_.item())
        return dt, r_

    log("c2 stage profile done")
    e2e_s, r = e2e_run(lambda: ofb200.frame_sequence(h_seq, imu_seq, cfg, ctx=ctx))
    log("c2 e2e sequence done")
    e2e_i, _ = e2e_run(lambda: ofb200.frame_pairs(h_prev, h_next, imu, cfg, ctx=ctx))
    # copy-only ceiling measured the same way, all ranks copying at the same time: the same pinned buffer through one
    # cudaMemcpyAsync per step and nothing else. e2e / this = how close the pipeline is to the host's H2D limit.
    d_stage = torch.empty((B + 1) * P, dtype=torch.uint8, device="cuda")

    def copy_only():
        ctx.lib.ofb_memcpy_async(ctx.h, ofb200._lib.ptr(d_stage), ofb200._lib.ptr(h_seq), (B + 1) * P)
        ctx.sync()
        return None
    log("c2 e2e independent done")
    cpy_s, _ = e2e_run(copy_only)
    del d_stage
    clk.__exit__()
    h2d_gbs = (B + 1) * P * args.steps / e2e_s / 1e9
    ceil_gbs = (B + 1) * P * args.steps / cpy_s / 1e9
    e2e = {"value": world * B * args.steps / e2e_s, "unit": "pairs/s",
           "h2d_bytes_per_step": int(world * ((B + 1) * P + imu_seq.nbytes)), "d2h_bytes_per_step": int(world * r.nbytes),
           "h2d_gbs_per_gpu": round(h2d_gbs, 1), "h2d_ceiling_gbs_concurrent": round(ceil_gbs, 1),
           "frac_of_copy_ceiling": round(h2d_gbs / ceil_gbs, 3),
           "host": {"cpu_affinity": affinity, "pinned_numa_node": numa_node_of(h_seq), "ranks_copying_concurrently": world,
                    "note": "h2d_ceiling = the same pinned frames through one plain cudaMemcpyAsync per step on every rank at "
                            "once (slowest rank): what this host delivers to %d GPU(s) in parallel" % world}}
    independent = {"value": world * B * args.steps / (ms_ind * 1e-3), "ms_per_step": ms_ind / args.steps,
                   "e2e": world * B * args.steps / e2e_i, "h2d_bytes_per_step": int(world * (2 * B * P + imu.nbytes)),
                   "max_abs_v_error_vs_truth": float(verr_i),
                   "note": "same pairs as separate prev/next buffers (no frame shared between pairs)"}
    clocks = clk.summary()
    # the two dominant kernels against the bound that actually limits them: warp-instruction issue (instruction count per
    # pair from the committed ncu capture, live stage time, live SM clock, 4 schedulers per SM)
    if clocks.get("sm_mhz"):
        sms = torch.cuda.get_device_properties(local).multi_processor_count
        peak_i = sms * 4 * float(clocks["sm_mhz"]) * 1e6
        iss = {}
        for key in ("eig_nms", "lk"):
            wi = tj.get(key, {}).get("warp_inst_per_pair")
            if wi:
                ach_i = float(wi) * B / (stage_ms[skeys.index(key)] * 1e-3)
                iss[key] = {"achieved": ach_i, "peak": peak_i, "unit": "warp-instructions/s", "frac": ach_i / peak_i,
                            "warp_inst_per_pair": wi}
        if iss:
            roofline["issue"] = dict(iss.get(skeys[dom], {}), per_kernel=iss)

    check = {"max_abs_v_error_vs_truth": float(verr), "min_tracked": tracked}

    # ---- the other BASELINE configurations, same process, same box ----
    c1 = c4 = c5 = mc = None
    c1_pairs = c4_pairs = c5_pairs = None
    log("c2 legs done")
    if args.workload == "all" and not args.no_extra:
        # free the C2 buffers first (the 4K / fleet legs allocate their own)
        del d_prev, d_next, d_seq, d_pts
        torch.cuda.empty_cache()
        c1, c1_pairs = leg_latency(args, ofb200, torch, ctx, "c1", rank)
        log("c1 done")
        c4, c4_pairs = leg_latency(args, ofb200, torch, ctx, "c4", rank)
        log("c4 done")
        c5, c5_pairs = leg_fleet(args, ofb200, torch, dist, ctx, rank, world, local)
        log("c5 done")
    if not args.no_mc:
        mc = leg_mc(args, ofb200, torch, dist, rank, world, local)
        log("mc done")

    line = {"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/f32/f64", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "pairs_per_step_per_gpu": B, "frames_per_step_per_gpu": B + 1, "distinct_motions": len(pairs),
                       "l2": "inputs larger than L2 (%d MB of frames per step)" % ((B + 1) * P // 2 ** 20),
                       "parallelism": "streams sharded, one batch per GPU, no data-path collective"},
            "roofline": roofline, "cpu_baseline": None, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clocks, "independent_pairs": independent, "track_solve": track_solve, "lifecycle": lifecycle, "mc": mc,
            "c1": c1, "c4": c4, "c5": c5, "check": check}

    # ---- CPU baselines: rank 0, after the last collective ----
    def cpu_c2():
        v, n, split = cpu_pair_path(lambda k: stream_pair(pairs, k), K_FEAT, MAX_LEVEL, 10.0, ncores)
        line["cpu_baseline"] = {"value": v, "unit": "pairs/s", "cores": ncores, "kind": "port",
                                "sample": "%d pairs of the same workload: cv2 4.13 gftt+pyrLK, %d threads; ms gftt/LK/solve = %s; %s" %
                                          (n, ncores, [round(s, 1) for s in split], SOLVE_NOTE)}
        check["feature_lists_vs_cv2"] = feature_tie_audit(ofb200, ctx, pairs, cfg)

    def cpu_lat(out, prs, name):
        def run():
            w, h, feat, ml = GEOM[name]
            v, n, split = cpu_pair_path(lambda k: prs[k % len(prs)], feat, ml, 3.0, ncores)
            out["cpu_baseline"] = {"value": 1e3 / v, "unit": "ms per pair", "cores": ncores, "kind": "port",
                                   "sample": "%d pairs, cv2 4.13 gftt+pyrLK with %d threads; ms gftt/LK/solve = %s; %s" %
                                             (n, ncores, [round(x, 2) for x in split], SOLVE_NOTE)}
        return run

    def cpu_c5():
        c5["cpu_baseline"] = cpu_job_subprocess("fleet")

    def cpu_mc_job():
        mc["cpu_baseline"] = cpu_job_subprocess("mc", int(mc["trials"]))

    jobs = []
    if not args.no_cpu:
        jobs.append(cpu_c2)
        if c1 is not None:
            jobs += [cpu_lat(c1, c1_pairs, "c1"), cpu_lat(c4, c4_pairs, "c4"), cpu_c5]
        if mc is not None:
            jobs.append(cpu_mc_job)
    finish(line, jobs)


if __name__ == "__main__":
    main()
