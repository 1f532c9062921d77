"""Stage 5 host mirror of numerical_simulation/simulation.py: the Monte-Carlo error propagation.

Same positional signatures as the reference:
    of_simulation(linear_velocity, angular_velocity, height_above_gr, normal_vector, translation, pos,
                  ang_vel_sig, translation_sig, height_sig, flow_sig, position_sig, normal_sig)
        simulation.py:36-66  -> (v_obs (iterations,3), feasible (2,N), R (iterations,))
    feas_simulation(..., normal_sigi, true_vel)      simulation.py:70-104 -> six (N,) per-point means
    overlap(data1, data2)                             simulation.py:124-136
The reference reads `iterations` and `true_flow` (and, in feas_simulation, `normal_sig`,
`velocity_sig`) from module globals; the same names exist here as module attributes and can also be
passed as keywords. The sweep drivers (simulation.py:183-578) are `SWEEPS[name]` /
`run_named_sweep`, which return the flat arrays the reference np.save()s (SURVEY App. C).

All trials run on the GPU (libofb200.so, Philox4x32-10 counter RNG); only per-step sums come back.
Sharded runs (`run_sweep(..., group=...)`) give each rank a contiguous trial range and merge the
sums with one tiny all-reduce, so the statistics equal a single-GPU run up to fp64 summation order.
"""
import ctypes as C

import numpy as np

from . import _lib
from . import velocity as _vel

# ---- reference constants (simulation.py:154-178) ------------------------------------------------
linear_velocity = np.array([1.0, 1.0, 1.0])
angular_velocity = np.array([1.0, 1.0, 1.0])
height_above_gr = 1.0
normal_vector = np.array([0.0, 0.0, 1.0])
translation = np.array([0.02, 0.0, 0.205])
ang_vel_sig = 0.00071
translation_sig = 0.005
height_sig = 0.01
flow_sig = 0.056 * np.sqrt(2) * 1.23
position_sig = 0.056 * 1.23
normal_sig = 0.00065
velocity_sig = 0.01
iterations = 100
true_flow = None          # set by the caller like the reference's global, or passed as keyword
seed = 0                  # RNG key for of_simulation / feas_simulation calls without an explicit seed
_call_counter = [0]       # successive calls draw from disjoint Philox streams (step ids)

PRECISIONS = {"fp32": 0, "fp64": 1}


def _v3(a):
    return np.asarray(a, dtype=np.float64).reshape(3)


def make_step(linear_velocity, angular_velocity, height_above_gr, normal_vector, translation, n_points, pos_offset,
              ang_vel_sig, translation_sig, height_sig, flow_sig, position_sig, normal_sig, velocity_sig=0.0,
              true_vel=(0.0, 0.0, 0.0)):
    s = _lib.McStep()
    s.v[:] = _v3(linear_velocity); s.w[:] = _v3(angular_velocity); s.n[:] = _v3(normal_vector); s.t[:] = _v3(translation)
    s.height = float(np.asarray(height_above_gr, dtype=np.float64).reshape(-1)[0])
    if s.height == 0.0:
        raise ValueError("height_above_gr must be non-zero")
    for name, val in (("ang_vel_sig", ang_vel_sig), ("translation_sig", translation_sig), ("height_sig", height_sig),
                      ("flow_sig", flow_sig), ("position_sig", position_sig), ("normal_sig", normal_sig),
                      ("velocity_sig", velocity_sig)):
        val = float(val)
        if val < 0:
            raise ValueError("%s must be >= 0 (numpy.random.normal rejects negative scales)" % name)
        setattr(s, name, val)
    s.true_vel[:] = _v3(true_vel)
    if int(n_points) < 2:
        raise ValueError("a step needs at least 2 points: with one, the velocity solve is singular (got %d)" % n_points)
    s.n_points = int(n_points)
    s.pos_offset = int(pos_offset)
    return s


def _steps_array(steps):
    arr = (_lib.McStep * len(steps))()
    for i, s in enumerate(steps):
        C.memmove(C.byref(arr, i * C.sizeof(_lib.McStep)), C.byref(s), C.sizeof(_lib.McStep))
    return arr


def run_steps(steps, pos, flow, trials, seed=0, step_id_base=0, trial_begin=0, precision="fp32", dump=False, ctx=None,
              want_R=True, sums_out=None):
    """Run `trials` trials of every step on this GPU. Returns the per-step sums (structured array
    _lib.MCSUMS_DTYPE) and, when dump, v_obs (S,trials,3) and R (S,trials).
    sums_out: a DEVICE buffer (CUDA tensor of len(steps) x 8 float64, or an address) that receives the sums instead; the
    call then only enqueues (no host synchronisation), so a collective on the same stream can follow it directly."""
    ctx = ctx or _lib.default_context()
    trials = int(trials)
    if trials <= 0:
        raise ValueError(' iterations must be a positive number')
    if hasattr(pos, "data_ptr"):              # device-resident point arrays (CUDA tensors, (N,2) float64): used in place
        if tuple(pos.shape) != tuple(flow.shape) or len(pos.shape) != 2 or pos.shape[1] != 2:
            raise ValueError("pos and true_flow must both be (N,2)")
    else:
        pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 2)
        flow = np.ascontiguousarray(flow, dtype=np.float64).reshape(-1, 2)
        if pos.shape != flow.shape:
            raise ValueError("pos and true_flow must have the same shape")
    arr = steps if isinstance(steps, C.Array) else _steps_array(steps)
    if sums_out is not None:
        if dump:
            raise ValueError("sums_out (device-resident sums) and dump are exclusive")
        _lib.check(ctx.lib.ofb_mc_sweep(ctx.h, C.cast(arr, C.c_void_p), len(steps), int(step_id_base), _lib.ptr(pos),
                                        _lib.ptr(flow), len(pos), int(trial_begin), trials, int(seed) & (2 ** 64 - 1),
                                        PRECISIONS[precision] + (0 if want_R else 2), _lib.ptr(sums_out), None, None))
        return sums_out
    sums = np.zeros(len(steps), _lib.MCSUMS_DTYPE)
    vd = Rd = None
    if dump:
        vd = np.zeros((len(steps), trials, 3))
        Rd = np.zeros((len(steps), trials))
    _lib.check(ctx.lib.ofb_mc_sweep(ctx.h, C.cast(arr, C.c_void_p), len(steps), int(step_id_base), _lib.ptr(pos),
                                    _lib.ptr(flow), len(pos), int(trial_begin), trials, int(seed) & (2 ** 64 - 1),
                                    PRECISIONS[precision] + (0 if want_R else 2), _lib.ptr(sums), _lib.ptr(vd), _lib.ptr(Rd)))
    if dump:
        return sums, vd, Rd
    return sums


def run_steps_multi(steps, pos, flow, trials, ctxs, seed=0, step_id_base=0, trial_begin=0, precision="fp32", want_R=True):
    """One process, several GPUs: `ctxs` is a list of Contexts (one per device, or several per device); the trial range is
    sharded over them inside the library (ofb_mc_sweep_multi) and the sums come back merged. No torch.distributed."""
    trials = int(trials)
    if trials <= 0:
        raise ValueError(' iterations must be a positive number')
    if not ctxs:
        raise ValueError("at least one context is required")
    pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 2)
    flow = np.ascontiguousarray(flow, dtype=np.float64).reshape(-1, 2)
    if pos.shape != flow.shape:
        raise ValueError("pos and true_flow must have the same shape")
    arr = steps if isinstance(steps, C.Array) else _steps_array(steps)
    handles = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
    sums = np.zeros(len(steps), _lib.MCSUMS_DTYPE)
    _lib.check(ctxs[0].lib.ofb_mc_sweep_multi(handles, len(ctxs), C.cast(arr, C.c_void_p), len(steps), int(step_id_base),
                                              _lib.ptr(pos), _lib.ptr(flow), len(pos), int(trial_begin), trials,
                                              int(seed) & (2 ** 64 - 1), PRECISIONS[precision] + (0 if want_R else 2),
                                              _lib.ptr(sums)))
    return sums


def shard_range(total, rank, world):
    """Contiguous trial range of `rank`: [begin, begin+count)."""
    base, rem = divmod(int(total), int(world))
    begin = rank * base + min(rank, rem)
    return begin, base + (1 if rank < rem else 0)


def merge_sums(sums, group=None, device=None):
    """All-reduce(sum) of the per-step sums over a torch.distributed group (NCCL on CUDA tensors,
    gloo on CPU tensors). The message is 8 doubles per step."""
    import torch
    import torch.distributed as dist
    flat = np.ascontiguousarray(sums).view(np.float64).reshape(len(sums), 8)
    t = torch.from_numpy(flat.copy())
    if device is not None:
        t = t.to(device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    out = t.cpu().numpy().reshape(-1).view(_lib.MCSUMS_DTYPE)
    return out.copy()


def stats_from_sums(sums, steps):
    """mean (S,3), population std (S,3) (np.std, ddof=0, as simulation.py:197-200), mean R (S,), n (S,)."""
    n = sums["n"]
    vt = np.array([[s.v[0], s.v[1], s.v[2]] for s in steps])
    md = sums["sum_dv"] / n[:, None]
    mean = vt + md
    var = sums["sum_dv2"] / n[:, None] - md ** 2
    std = np.sqrt(np.maximum(var, 0.0))
    return mean, std, sums["sum_R"] / n, n


def run_sweep(steps, pos, flow, trials, seed=0, precision="fp32", distributed=False, group=None, ctx=None):
    """Run a sweep; with distributed=True the trials are sharded over the torch.distributed ranks and
    the sums merged. Returns (mean, std, meanR, n)."""
    if distributed:
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        begin, count = shard_range(trials, rank, world)
        if count > 0:
            sums = run_steps(steps, pos, flow, count, seed=seed, trial_begin=begin, precision=precision, ctx=ctx)
        else:
            sums = np.zeros(len(steps), _lib.MCSUMS_DTYPE)
        dev = torch.device("cuda", (ctx or _lib.default_context()).device) if dist.get_backend(group) == "nccl" else None
        sums = merge_sums(sums, group, dev)
    else:
        sums = run_steps(steps, pos, flow, trials, seed=seed, precision=precision, ctx=ctx)
    return stats_from_sums(sums, steps)


# ---- reference-signature functions ----------------------------------------------------------------
def _philox_normals(seed, step, trial, n_blocks):
    """Host replay of the device's draws for ONE trial (used only to rebuild the `feasible` by-product
    that of_simulation returns for its last trial, simulation.py:65)."""
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
    out = np.zeros((n_blocks, 4))
    for b in range(n_blocks):
        c = [trial & 0xFFFFFFFF, (trial >> 32) & 0xFFFFFFFF, b, step & 0xFFFFFFFF]
        k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
        for _ in range(10):
            p0, p1 = M0 * c[0], M1 * c[2]
            c = [((p1 >> 32) ^ c[1] ^ k0) & 0xFFFFFFFF, p1 & 0xFFFFFFFF, ((p0 >> 32) ^ c[3] ^ k1) & 0xFFFFFFFF,
                 p0 & 0xFFFFFFFF]
            k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
        u = [float((np.float32(x) + np.float32(0.5)) * np.float32(2.3283064365386963e-10)) for x in c]
        for h in (0, 1):
            rad = np.sqrt(-2.0 * np.log(u[2 * h]))
            ang = 2.0 * np.pi * (u[2 * h + 1] - 0.5)
            out[b, 2 * h], out[b, 2 * h + 1] = rad * np.cos(ang), rad * np.sin(ang)
    return out


def of_simulation(linear_velocity, angular_velocity, height_above_gr, normal_vector, translation, pos, ang_vel_sig,
                  translation_sig, height_sig, flow_sig, position_sig, normal_sig, *, iterations=None, true_flow=None,
                  seed=None, step_id=None, precision="fp32", ctx=None):
    g = globals()
    iters = int(g["iterations"] if iterations is None else iterations)
    if iters <= 0:
        raise ValueError(' iterations must be a positive number')
    pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 2)
    tf = g["true_flow"] if true_flow is None else true_flow
    if tf is None:
        tf = _vel.generate_test_data(pos, linear_velocity, angular_velocity, height_above_gr, normal_vector, translation,
                                     ctx=ctx)
    tf = np.ascontiguousarray(tf, dtype=np.float64).reshape(-1, 2)
    sd = int(g["seed"] if seed is None else seed)
    if step_id is None:
        step_id = _call_counter[0]
        _call_counter[0] += 1
    step = make_step(linear_velocity, angular_velocity, height_above_gr, normal_vector, translation, len(pos), 0,
                     ang_vel_sig, translation_sig, height_sig, flow_sig, position_sig, normal_sig)
    _, v_obs, R = run_steps([step], pos, tf, iters, seed=sd, step_id_base=step_id, precision=precision, dump=True, ctx=ctx)
    # `feasible` is the LAST trial's (simulation.py:65): rebuild that trial's noisy inputs on the host
    z = _philox_normals(sd, step_id, iters - 1, 3 + len(pos))
    w_err = _v3(angular_velocity) + ang_vel_sig * z[0, :3]
    t_err = _v3(translation) + translation_sig * z[1, :3]
    flow_err = tf + flow_sig * z[3:, 0:2]
    pos_err = pos + position_sig * z[3:, 2:4]
    n_err = _v3(normal_vector) / np.linalg.norm(_v3(normal_vector))
    feasible = _vel.feasibility(pos_err, linear_velocity, flow_err, w_err, t_err, n_err, ctx=ctx)
    return v_obs[0], feasible, R[0]


def feas_simulation(linear_velocity, angular_velocity, height_above_gr, normal_vector, translation, pos, ang_vel_sig,
                    translation_sig, height_sig, flow_sig, position_sig, normal_sigi, true_vel, *, iterations=None,
                    true_flow=None, seed=None, step_id=None, normal_sig=None, velocity_sig=None, trial_begin=0, ctx=None,
                    return_sums=False):
    """simulation.py:70-104. `normal_sigi` is ignored exactly as in the reference (the global normal_sig
    is what perturbs the normal, lines 87-88); pass normal_sig= to override the module attribute."""
    ctx = ctx or _lib.default_context()
    g = globals()
    iters = int(g["iterations"] if iterations is None else iterations)
    if iters <= 0:
        raise ValueError(' iterations must be a positive number')
    pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 2)
    tf = g["true_flow"] if true_flow is None else true_flow
    if tf is None:
        raise ValueError("feas_simulation needs true_flow (module attribute or keyword), as the reference's global")
    tf = np.ascontiguousarray(tf, dtype=np.float64).reshape(-1, 2)
    if len(tf) != len(pos):
        raise ValueError("true_flow and pos must have the same number of points")   # reference hard-codes 200 (sim:83-84)
    sd = int(g["seed"] if seed is None else seed)
    if step_id is None:
        step_id = _call_counter[0]
        _call_counter[0] += 1
    step = make_step(linear_velocity, angular_velocity, height_above_gr, normal_vector, translation, len(pos), 0,
                     ang_vel_sig, translation_sig, height_sig, flow_sig, position_sig,
                     g["normal_sig"] if normal_sig is None else normal_sig,
                     g["velocity_sig"] if velocity_sig is None else velocity_sig, true_vel)
    sums = np.zeros((6, len(pos)))
    _lib.check(ctx.lib.ofb_mc_feas(ctx.h, C.cast(C.byref(step), C.c_void_p), int(step_id), _lib.ptr(pos), _lib.ptr(tf),
                                   int(trial_begin), iters, sd & (2 ** 64 - 1), _lib.ptr(sums)))
    if return_sums:
        return sums
    m = sums / iters
    return m[0], m[1], m[2], m[3], m[4], m[5]


def merge_range(lo, hi, group=None, device=None):
    """All-reduce(min) / (max) of a shard's value range (SURVEY 8e: the common histogram edges of `overlap` come from
    the pooled sample). Empty shards pass lo=+inf, hi=-inf."""
    import torch
    import torch.distributed as dist
    a = torch.tensor([lo], dtype=torch.float64, device=device)
    b = torch.tensor([hi], dtype=torch.float64, device=device)
    dist.all_reduce(a, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(b, op=dist.ReduceOp.MAX, group=group)
    return float(a.item()), float(b.item())


def merge_counts(counts, group=None, device=None):
    """All-reduce(sum) of histogram bin counts (int64 on the wire)."""
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(np.ascontiguousarray(counts).astype(np.int64))
    if device is not None:
        t = t.to(device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy().astype(np.uint64)


def overlap(data1, data2, ctx=None, distributed=False, group=None):
    """simulation.py:124-136: common 100-bin histogram over the pooled range, sum of bin-wise minima.
    distributed=True: data1/data2 are this rank's SHARDS of the two samples (e.g. the v_obs dumps of its trial range);
    the range is merged with all-reduce(min/max), the bin counts with all-reduce(sum), and every rank returns the
    overlap of the full samples.
    Like numpy.histogram's autodetected range, a NaN or infinite sample raises ValueError (on every rank when
    distributed: a shard with one reports the range (-inf, inf), which the merge hands to all)."""
    d1 = np.ascontiguousarray(data1, dtype=np.float64).reshape(-1)
    d2 = np.ascontiguousarray(data2, dtype=np.float64).reshape(-1)
    finite = bool(np.isfinite(d1).all() and np.isfinite(d2).all())
    if not finite and not distributed:
        raise ValueError("overlap: the data are not finite (NaN or inf), so neither is their range")
    ctx = ctx or _lib.default_context()
    los, his = ([], []) if finite else ([-np.inf], [np.inf])
    for d in (d1, d2) if finite else ():
        if len(d):
            lo, hi = C.c_double(), C.c_double()
            _lib.check(ctx.lib.ofb_minmax(ctx.h, _lib.ptr(d), len(d), C.byref(lo), C.byref(hi)))
            los.append(lo.value); his.append(hi.value)
    dev = None
    if distributed:
        import torch
        import torch.distributed as dist
        dev = torch.device("cuda", ctx.device) if dist.get_backend(group) == "nccl" else None
        lo, hi = merge_range(min(los) if los else np.inf, max(his) if his else -np.inf, group, dev)
        if lo == np.inf:
            return 0                                    # every shard empty
        if not (np.isfinite(lo) and np.isfinite(hi)):
            raise ValueError("overlap: the data are not finite (NaN or inf), so neither is their range")
    else:
        if not los:
            return 0
        lo, hi = min(los), max(his)
    hists = []
    for d in (d1, d2):
        cnt = np.zeros(100, np.uint64)
        if len(d):
            _lib.check(ctx.lib.ofb_histogram(ctx.h, _lib.ptr(d), len(d), lo, hi, 100, _lib.ptr(cnt)))
        hists.append(cnt)
    if distributed:
        both = merge_counts(np.concatenate(hists), group, dev)
        hists = [both[:100], both[100:]]
    return int(np.sum(np.minimum(hists[0], hists[1])))


def stream_shard(n_streams, rank, world):
    """Camera streams of `rank` (SURVEY 8e: gpu = stream_id mod n_gpu, no data-path collective)."""
    return list(range(int(rank), int(n_streams), int(world)))


def gather_stream_velocities(v_local, stream_ids, n_streams, group=None, device=None):
    """Final gather of the per-stream velocities of a sharded fleet (3 doubles per stream): every rank contributes
    its streams' rows to an (n_streams, 3) table, merged with one all-reduce(sum) (rows are disjoint)."""
    return gather_stream_rows(np.asarray(v_local, dtype=np.float64).reshape(-1, 3), stream_ids, n_streams, group, device)


def gather_stream_rows(rows_local, stream_ids, n_streams, group=None, device=None):
    """(n_local, k) per-stream rows -> (n_streams, k) table on every rank, one all-reduce(sum) over disjoint rows."""
    import torch
    import torch.distributed as dist
    rows_local = np.asarray(rows_local, dtype=np.float64)
    rows_local = rows_local.reshape(len(stream_ids), -1) if len(stream_ids) else rows_local.reshape(0, rows_local.shape[-1])
    table = np.zeros((int(n_streams), rows_local.shape[1]))
    table[np.asarray(stream_ids, dtype=np.int64)] = rows_local
    t = torch.from_numpy(table)
    if device is not None:
        t = t.to(device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()


# ---- sweep drivers (simulation.py:183-578; SURVEY App. C) ------------------------------------------
def centred_points(data, fx=1.27, fy=0.93):
    """simulation.py:186-187: x=(x-mean)*1.27, y=(y-mean)*0.93."""
    d = np.array(data, dtype=np.float64)
    d[:, 0] = (d[:, 0] - np.mean(d[:, 0])) * fx
    d[:, 1] = (d[:, 1] - np.mean(d[:, 1])) * fy
    return d


def miscentred_points(data, fx=1.27, fy=0.93):
    """simulation.py:442-443 / 552-553: the precedence slip `x - mean*1.27` of two sweeps, kept."""
    d = np.array(data, dtype=np.float64)
    d[:, 0] = d[:, 0] - np.mean(d[:, 0]) * fx
    d[:, 1] = d[:, 1] - np.mean(d[:, 1]) * fy
    return d


def advect_points(data, linear_velocity, angular_velocity, height_above_gr, normal_vector, translation, k, ctx=None):
    """The dynamic part of the time-evolution sweep (simulation.py:496-499), all k steps in one device launch:
    step s+1 has data += generate_test_data(data, v, [0,0,0], h, n, t) and h += v.n.
    -> (pos (k,N,2), true_flow (k,N,2) = generate_test_data(pos_s, v, w, h_s, n, t), heights (k,))."""
    ctx = ctx or _lib.default_context()
    d = np.ascontiguousarray(data, dtype=np.float64).reshape(-1, 2)
    k = int(k)
    if k < 1:
        raise ValueError("k must be a positive number of steps")
    pos = np.zeros((k, len(d), 2)); flow = np.zeros((k, len(d), 2)); hs = np.zeros(k)
    v3, w3, n3, t3 = _v3(linear_velocity), _v3(angular_velocity), _v3(normal_vector), _v3(translation)
    h0 = float(np.asarray(height_above_gr, dtype=np.float64).reshape(-1)[0])
    if len(d):
        _lib.check(ctx.lib.ofb_advect_points(ctx.h, _lib.ptr(d), len(d), _lib.ptr(v3), _lib.ptr(w3), h0, _lib.ptr(n3),
                                             _lib.ptr(t3), k, _lib.ptr(pos), _lib.ptr(flow), _lib.ptr(hs)))
    else:
        hs[:] = h0 + np.arange(k) * float(v3 @ n3)
    return pos, flow, hs


def _default_sigmas():
    g = globals()
    return dict(ang_vel_sig=g["ang_vel_sig"], translation_sig=g["translation_sig"], height_sig=g["height_sig"],
                flow_sig=g["flow_sig"], position_sig=g["position_sig"], normal_sig=g["normal_sig"])


def build_sweep(name, data, k=None):
    """Steps, point array and true flow of a named sweep. `data` is the (N,2) point set (points.txt)."""
    g = globals()
    v, w, h, n, t = g["linear_velocity"], g["angular_velocity"], g["height_above_gr"], g["normal_vector"], g["translation"]
    steps, pts, flows = [], [], []

    def add(points, height=h, normal=n, **over):
        sig = _default_sigmas()
        sig.update(over)
        off = sum(len(p) for p in pts)
        pts.append(points)
        flows.append(_vel.generate_test_data(points, v, w, height, normal, t))
        steps.append(make_step(v, w, height, normal, t, len(points), off, **sig))

    if name == "flow_errors":                 # simulation.py:183-202
        k = k or 100; d = centred_points(data)
        for i in range(k):
            add(d, flow_sig=0.001 * i, position_sig=np.sqrt(2) / 1000 * i)
    elif name == "distance_error":            # 216-235
        k = k or 100; d = centred_points(data)
        for i in range(k):
            add(d, height_sig=0.001 * i)
    elif name == "ang_vel_error":             # 249-271
        k = k or 100; d = centred_points(data)
        for i in range(k):
            add(d, ang_vel_sig=0.001 * i)
    elif name == "normal_error":              # 285-304 (no effect: SURVEY App. D.1)
        k = k or 100; d = centred_points(data)
        for i in range(k):
            add(d, normal_sig=0.001 * i)
    elif name == "translation_error":         # 319-338
        k = k or 100; d = centred_points(data)
        for i in range(k):
            add(d, translation_sig=0.001 * i)
    elif name == "orientation":               # 357-377
        k = k or 100; d = centred_points(data)
        for i in range(k):
            add(d, normal=np.array([np.sin(np.pi * i / k), 0.0, np.cos(np.pi * i / k)]))
    elif name == "height":                    # 401-423
        k = k or 100; d = centred_points(data)
        for i in range(k):
            add(d, height=0.2 + np.linspace(0.2, 7.65, k)[i])
    elif name == "point_position":            # 442-461
        k = k or 100; d = miscentred_points(data)
        for i in range(k):
            add(d + np.ones_like(d) * i / 100)
    elif name == "number_of_points":          # 552-578
        k = k or 99; d = miscentred_points(data)
        for i in range(k):
            add(d[:2 * i + 2])
    elif name == "time_evolution":            # 472-501: points advected by their own flow, height += v.n per step
        k = k or 100
        d = np.array(data, dtype=np.float64)
        d[:, 0] -= np.mean(d[:, 0]); d[:, 1] -= np.mean(d[:, 1])
        d = d * 10                             # simulation.py:472-474
        if len(d) > _lib.MC_MAX_POINTS:
            raise ValueError("time_evolution: at most %d points" % _lib.MC_MAX_POINTS)
        pos_k, flow_k, h_k = advect_points(d, v, w, h, n, t, k)     # one launch for the k dependent steps
        sig = _default_sigmas()
        for i in range(k):
            pts.append(pos_k[i]); flows.append(flow_k[i])
            steps.append(make_step(v, w, h_k[i], n, t, len(d), i * len(d), **sig))
    else:
        raise ValueError("unknown sweep %r" % name)
    return steps, np.vstack(pts), np.vstack(flows)


SWEEPS = ("flow_errors", "distance_error", "ang_vel_error", "normal_error", "translation_error", "orientation", "height",
          "point_position", "number_of_points", "time_evolution")
SWEEP_FILES = {"flow_errors": "effect_of_flow_errors", "distance_error": "effect_of_distance_error",
               "ang_vel_error": "effect_o_ang_vel_error", "normal_error": "effect_of_normal_error",
               "translation_error": "effect_of_translation_error", "orientation": "effect_of_orientation",
               "height": "effect_of_height", "point_position": "effect_of_point_position",
               "number_of_points": "number_of_point"}


def run_named_sweep(name, data, trials=100, k=None, seed=0, precision="fp32", distributed=False, group=None, ctx=None):
    """-> (flat, meanR): flat = np.append(v_flow, v_flow_err), the array the reference saves
    (layout [means (3k) | stds (3k)], numerical_simulation/visualisation.py:5-14)."""
    steps, pts, flows = build_sweep(name, data, k)
    mean, std, mR, _ = run_sweep(steps, pts, flows, trials, seed=seed, precision=precision, distributed=distributed,
                                 group=group, ctx=ctx)
    return np.append(mean, std), mR


# ---- sorting study (simulation.py:604-894): which per-point metric separates moving points / other planes ----------
def rotate_flows(flow, minang, rng):
    """simulation.py:702-705 / 767-770 / 858-861: every row turned in the image plane by an angle drawn from
    U(minang, 2 pi - minang) -- the flows of independently moving points."""
    out = np.array(flow, dtype=np.float64)
    for i in range(len(out)):
        a = rng.uniform(minang, 2 * np.pi - minang)
        out[i] = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]) @ out[i]
    return out


SORTING_KINDS = ("planes", "moving", "moving_and_plane", "dynamic")


def sorting_scenario(kind, data, minang=None, rng=None, velocity_scale=None):
    """Point set, composite true flow and truth of one sorting scenario of the reference:
      "planes"            simulation.py:615-628  thirds of the points on planes at h = 3, 2, 1 m
      "moving"            simulation.py:693-706  v x 10; second half: flows rotated (moving points)
      "moving_and_plane"  simulation.py:753-772  (the LIVE section) h = 2, v x 2.9 h; [0, N/5) static at 2 m,
                                                 [N/5, 2(N/3)) moving at 1 m, [2(N/3), N) static at 1 m
      "dynamic"           simulation.py:856-864  one step of the velocity sweep: thirds = static, moving, plane at h + 1;
                                                 velocity_scale multiplies the module's linear_velocity
    minang: lower end of the rotation-angle range. The reference writes 10/360*2*np.pi, which Python 2 (the
    interpreter it ran under) evaluates to 0 -- the default; "dynamic" uses 1 rad (simulation.py:859).
    -> dict(data, true_flow, linear_velocity, height, groups={name: slice})."""
    g = globals()
    rng = rng or np.random.RandomState(0)
    v = np.array(g["linear_velocity"], dtype=np.float64)
    w, n, t = g["angular_velocity"], g["normal_vector"], g["translation"]
    d = np.array(data, dtype=np.float64)
    N = len(d)
    gtd = _vel.generate_test_data
    if kind == "planes":
        d = centred_points(d)
        h = 3.0
        a, b = int(N / 3), 2 * int(N / 3)
        tf = np.vstack([gtd(d[:a], v, w, h, n, t), gtd(d[a:b], v, w, h - 1, n, t), gtd(d[b:], v, w, h - 2, n, t)])
        groups = {"3m": slice(0, a), "2m": slice(a, b), "1m": slice(b, N)}
    elif kind == "moving":
        d[:, 0] -= np.mean(d[:, 0]); d[:, 1] -= np.mean(d[:, 1])
        h = float(g["height_above_gr"])
        v = v * 10
        a = int(N / 2)
        tf = np.vstack([gtd(d[:a], v, w, h, n, t), rotate_flows(gtd(d[a:], v, w, h, n, t), 0.0 if minang is None else minang, rng)])
        groups = {"static": slice(0, a), "moving": slice(a, N)}
    elif kind == "moving_and_plane":
        d[:, 0] -= np.mean(d[:, 0]); d[:, 1] -= np.mean(d[:, 1])
        h = 2.0
        v = v * 2.9 * h
        a, b = int(N / 5), 2 * int(N / 3)
        tf = np.vstack([gtd(d[:a], v, w, h, n, t),
                        rotate_flows(gtd(d[a:b], v, w, h - 1, n, t), 0.0 if minang is None else minang, rng),
                        gtd(d[b:], v, w, h - 1, n, t)])
        groups = {"static_2m": slice(0, a), "moving_1m": slice(a, b), "static_1m": slice(b, N)}
    elif kind == "dynamic":
        d[:, 0] -= np.mean(d[:, 0]); d[:, 1] -= np.mean(d[:, 1])
        h = 1.0
        v = v * (1.0 if velocity_scale is None else velocity_scale)
        a, b = int(N / 3), 2 * int(N / 3)
        tf = np.vstack([gtd(d[:a], v, w, h, n, t), rotate_flows(gtd(d[a:b], v, w, h, n, t), 1.0 if minang is None else minang, rng),
                        gtd(d[b:], v, w, h + 1, n, t)])
        groups = {"static": slice(0, a), "moving": slice(a, b), "plane": slice(b, N)}
    else:
        raise ValueError("unknown sorting scenario %r (one of %s)" % (kind, ", ".join(SORTING_KINDS)))
    return dict(data=d, true_flow=tf, linear_velocity=v, height=h, groups=groups)


METRICS = ("backward_para", "backward_dist", "forward_para", "forward_dist", "backward_res", "forward_res")


def sorting_study(kind, data, iterations=None, seed=0, minang=None, k=100, cumulative=False, ctx=None):
    """The sorting simulations of simulation.py:604-894 on the GPU (feas_simulation trials + overlap histograms).

    "planes" / "moving" / "moving_and_plane": one feas_simulation over the scenario's composite flow field ->
        dict with the six per-point means (METRICS), `groups`, and
        "planes":            sorted_distance, distance_diff (simulation.py:630-631)
        "moving_and_plane":  sorted_out_forward / sorted_out_backward = the two fractions the live section prints
                             (parallelity > 0.88 over the middle third, simulation.py:778-779).
    "dynamic": the velocity sweep of simulation.py:850-877: k steps, step i at linear_velocity * i * 0.05, twelve
        overlap curves "mov_overlap_<metric>" (static vs moving) and "plane_overlap_<metric>" (static vs the plane one
        metre further), each (k,). The reference rescales the velocity cumulatively (`linear_velocity=linear_velocity*i*
        0.05`, which makes it zero from step 0 on); cumulative=True reproduces that, the default sweeps the intended 0..5x."""
    g = globals()
    iters = int(g["iterations"] if iterations is None else iterations)
    rng = np.random.RandomState(int(seed) & 0x7fffffff)
    w, n, t = g["angular_velocity"], g["normal_vector"], g["translation"]
    sig = _default_sigmas()

    def run(sc, step_id):
        return feas_simulation(sc["linear_velocity"], w, sc["height"], n, t, sc["data"], sig["ang_vel_sig"],
                               sig["translation_sig"], sig["height_sig"], sig["flow_sig"], sig["position_sig"],
                               sig["normal_sig"], sc["linear_velocity"], iterations=iters, true_flow=sc["true_flow"],
                               seed=seed, step_id=step_id, ctx=ctx)

    if kind != "dynamic":
        sc = sorting_scenario(kind, data, minang=minang, rng=rng)
        out = dict(zip(METRICS, run(sc, 0)))
        out["groups"] = sc["groups"]
        out["scenario"] = sc
        if kind == "planes":
            out["sorted_distance"] = np.sort(out["forward_dist"])
            out["distance_diff"] = np.diff(out["sorted_distance"])
        if kind == "moving_and_plane":
            third = int(len(sc["data"]) / 3)
            mid = slice(third, 2 * third)
            out["sorted_out_forward"] = float(np.sum(out["forward_para"][mid] > 0.88)) / float(third)
            out["sorted_out_backward"] = float(np.sum(out["backward_para"][mid] > 0.88)) / float(third)
        return out
    curves = {("%s_overlap_%s" % (grp, m)): np.zeros(k) for grp in ("mov", "plane") for m in METRICS}
    scale = 1.0
    for i in range(k):
        scale = scale * i * 0.05 if cumulative else i * 0.05
        sc = sorting_scenario("dynamic", data, minang=minang, rng=rng, velocity_scale=scale)
        res = dict(zip(METRICS, run(sc, i)))
        gs = sc["groups"]
        for m in METRICS:
            curves["mov_overlap_" + m][i] = overlap(res[m][gs["static"]], res[m][gs["moving"]], ctx=ctx)
            curves["plane_overlap_" + m][i] = overlap(res[m][gs["static"]], res[m][gs["plane"]], ctx=ctx)
    curves["velocity_scale"] = np.arange(k) * 0.05
    return curves
