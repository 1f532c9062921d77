"""Feature lifecycle around the tracker, device resident (SURVEY 8f-2, include/ofb200.h `ofb_tracker_*`).

`StreamTracker.step(frame, imu)` is one iteration of the reference's per-frame loops
(flight_experiments/evaluate_exp.py:77-120, velocity_measurment_node:110-172 + 224-260,
optical_flow_experiments/of_module.py:78-147): grey conversion, calcOpticalFlowPyrLK from the previous frame,
`new_pos[status==1]`, the optional `of.static_immobile` / `of.r_tilde` gates, `solve_lgs`, and a
goodFeaturesToTrack top-up when the features run low. The point sets never leave the GPU; only the small
per-stream result record (velocity, counts) comes back.

There is no CPU path: everything runs in libofb200.so (csrc/tracker.cu)."""
import ctypes as C

import numpy as np

from . import _lib
from .vision import _ego_flag, _fb_threshold, _gyro_flag, as_camera, make_pair_cfg


class StreamTracker:
    """n_streams camera streams advancing in lockstep, one frame each per `step`.

    feature_params / lk_params take the reference's dictionaries verbatim, e.g.
    dict(qualityLevel=0.7, minDistance=10, blockSize=12) (node:96-102) and
    dict(winSize=(15,15), maxLevel=3, criteria=(3, 20, 0.03)) (node:105-107).
    topup: "exp"  -> evaluate_exp.py:105-107 (unmasked, maxCorners=max_features, appended),
           "node" -> node:157-172 (circles of mask_radius around surviving points, maxCorners=max_features-count),
           "module" -> of_module.py:83-86 (the set is replaced).
    gate: None, ("ge", T) (of_module.py:129) or ("le", T) (node:240-245) on of.r_tilde(x, u, n, v_prior, d); the prior is
          `v_prior` of the step, else the stream's last solved velocity, else `v_init` (node:183 uses [0.1, 0.1, 0.1]);
          while it is exactly zero the gate is skipped (r_tilde is 1 for every point then).
    max_speed > 0 enables of.static_immobile(new, old, max_speed, d, dummy_value).
    borrow_frames: device-resident grey frames (CUDA tensors) are tracked in place instead of being copied into the
    tracker; pass a NEW tensor every step (the tracker keeps the previous one alive; do not overwrite it).
    camera: (K, D, rate[, iterations]) or vision.make_camera(...) -- see set_camera.
    fb_threshold: None / 0 = off, T > 0 = forward-backward check of the LK tracks -- see set_fb_threshold.
    gyro_prediction: LK starts from the rotation the step's gyro sample measured -- see set_gyro_prediction.
    ego_motion: every stream's angular rate is also estimated from its kept points -- see set_ego_motion.
    robust: None / False, True or (c, iterations): the robust velocity solve of every stream -- see set_robust."""

    def __init__(self, width, height, max_features=100, min_features=20, n_streams=1, feature_params=None,
                 lk_params=None, topup="exp", mask_radius=30, bgr=False, variant="exp", principal=None,
                 scaling=1.0, flow_scaling=None, max_speed=0.0, dummy_value=float("nan"), gate=None, min_solve=3,
                 min_eig_thr=1e-4, borrow_frames=False, v_init=None, camera=None, fb_threshold=None,
                 gyro_prediction=False, ego_motion=False, robust=None, ctx=None):
        fb = _fb_threshold(fb_threshold)
        gyro = _gyro_flag(gyro_prediction)
        ego = _ego_flag(ego_motion)
        rcfg = _lib.robust_cfg(robust)
        fp = dict(qualityLevel=0.01, minDistance=10, blockSize=7)
        fp.update(feature_params or {})
        lk = dict(winSize=(15, 15), maxLevel=3, criteria=(3, 20, 0.03))
        lk.update(lk_params or {})
        self.ctx = ctx or _lib.default_context()
        cfg = _lib.TrackerCfg()
        cfg.pair = make_pair_cfg(width, height, max_features, quality=fp["qualityLevel"], min_distance=fp["minDistance"],
                                 block_size=fp["blockSize"], win=lk["winSize"], max_level=lk["maxLevel"],
                                 criteria=lk["criteria"], min_eig_thr=min_eig_thr, variant=variant, principal=principal,
                                 pos_scale=scaling, flow_scale=scaling if flow_scaling is None else flow_scaling)
        cfg.n_streams = int(n_streams)
        cfg.min_features = int(min_features)
        cfg.topup_mode = _lib.TOPUP_MODES[topup]
        cfg.mask_radius = int(mask_radius)
        cfg.bgr_input = 1 if bgr else 0
        cfg.max_speed = float(max_speed)
        cfg.dummy_value = float(dummy_value)
        if gate is None:
            cfg.gate_mode, cfg.gate_T = _lib.GATE_NONE, 0.0
        else:
            cfg.gate_mode = {"ge": _lib.GATE_R_GE, "le": _lib.GATE_R_LE}[gate[0]]
            cfg.gate_T = float(gate[1])
        cfg.min_solve = int(min_solve)
        cfg.borrow_frames = 1 if borrow_frames else 0
        if v_init is not None:       # the node's self.vel = [0.1, 0.1, 0.1] (velocity_measurment_node:183)
            cfg.v_init[:] = [float(x) for x in np.asarray(v_init, dtype=np.float64).reshape(3)]
        self._held = []          # borrow_frames: the last two device frames stay referenced until they are no longer read
        self.cfg = cfg
        self.n_streams, self.width, self.height, self.bgr = int(n_streams), int(width), int(height), bool(bgr)
        h = C.c_void_p()
        _lib.check(self.ctx.lib.ofb_tracker_create(self.ctx.h, C.byref(cfg), C.byref(h)))
        self.h = h
        cap = C.c_int()
        _lib.check(self.ctx.lib.ofb_tracker_capacity(self.h, C.byref(cap)))
        self.capacity = cap.value
        self._has_cam = False
        if camera is not None:
            self.set_camera(camera)
        if fb:
            _lib.check(self.ctx.lib.ofb_tracker_set_fb_check(self.h, fb))
        if gyro:
            self.set_gyro_prediction(True)
        self.ego_motion = False
        if ego:
            self.set_ego_motion(True)
        self.robust = None
        if rcfg is not None:
            self.set_robust((rcfg.c, rcfg.iterations))

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.lib.ofb_tracker_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def graph_steps(self):
        """steps replayed from a captured CUDA graph so far (small fleets fed from host memory; include/ofb200.h)"""
        return self.graph_info()[0]

    def graph_info(self):
        """(steps replayed from a graph, False): the second element is always False, the graphs hold no conditional node"""
        n, c = C.c_uint64(), C.c_int()
        _lib.check(self.ctx.lib.ofb_tracker_graph_info(self.h, C.byref(n), C.byref(c)))
        return n.value, bool(c.value)

    def reset(self):
        _lib.check(self.ctx.lib.ofb_tracker_reset(self.h))

    def set_camera(self, camera):
        """Calibrated camera of every stream from the next step on: the gate and the solve see
        x = undistort(p_new), u = (undistort(p_new) - undistort(p_old)) * rate (OpenCV's lens model, iterations default to
        vision.CAMERA_ITERATIONS) instead of the pinhole principal / scaling / flow_scaling. None detaches it."""
        cam = as_camera(camera)
        _lib.check(self.ctx.lib.ofb_tracker_set_camera(self.h, C.byref(cam) if cam is not None else None))
        self._has_cam = cam is not None

    def set_fb_threshold(self, threshold):
        """Forward-backward check of every stream's LK tracks from the next step on (vision.track_forward_backward): a
        point that does not return within `threshold` px of where it started counts as lost (status 0). None or 0
        turns it off."""
        _lib.check(self.ctx.lib.ofb_tracker_set_fb_check(self.h, _fb_threshold(threshold)))

    def set_gyro_prediction(self, enable):
        """Gyro prediction of every stream's LK tracks from the next step on (vision.gyro_predict): LK starts each point
        from where the step's gyro rate imu["w"] rotates it over one frame, with the camera when one is set and the
        pinhole principal / scaling / flow_scaling otherwise (dt = scaling / flow_scaling). False turns it off."""
        on = _gyro_flag(enable)
        p = self.cfg.pair
        if on and not self._has_cam and (p.flow_scale == 0 or p.pos_scale == 0 or not np.isfinite(p.pos_scale / p.flow_scale)):
            raise ValueError("gyro prediction with the pinhole needs flow_scaling != 0 and a finite, non-zero "
                             "scaling / flow_scaling")
        _lib.check(self.ctx.lib.ofb_tracker_set_gyro_prediction(self.h, on))

    def set_ego_motion(self, enable):
        """Ego-motion solve of every stream from the next step on (velocity.solve_ego_motion on the kept points, right
        after the velocity solve): step(..., want_ego=True) returns its _lib.EGO_RESULT_DTYPE records. The standard
        records do not change. Not available for variant="module" (no gyro term). False turns it off."""
        on = _ego_flag(enable)
        _lib.check(self.ctx.lib.ofb_tracker_set_ego_motion(self.h, 1 if on else 0))
        self.ego_motion = on

    def set_robust(self, robust):
        """Robust velocity solve of every stream from the next step on (velocity.solve_velocity_robust on the kept
        points, after the velocity and ego-motion solves): step(..., want_robust=True) returns its
        _lib.ROBUST_RESULT_DTYPE records. None / False turns it off, True uses c = 4 and 10 iterations, (c, iterations)
        sets them. The standard records, the point sets and the r_tilde gate's prior (the plain velocity) do not
        change. Not available for variant="module"."""
        cfg = _lib.robust_cfg(robust)
        _lib.check(self.ctx.lib.ofb_tracker_set_robust(self.h, C.byref(cfg) if cfg is not None else None))
        self.robust = None if cfg is None else (cfg.c, cfg.iterations)

    def set_points(self, points):
        """points: one (N,2)/(N,1,2) array per stream (or a single array when n_streams == 1)."""
        if self.n_streams == 1 and not isinstance(points, (list, tuple)):
            points = [points]
        if len(points) != self.n_streams:
            raise ValueError("one point array per stream is required")
        buf = np.zeros((self.n_streams, self.capacity, 2), np.float32)
        cnt = np.zeros(self.n_streams, np.int32)
        for s, p in enumerate(points):
            p = np.asarray(p, dtype=np.float32).reshape(-1, 2)
            if len(p) > self.capacity:
                raise ValueError("stream %d: %d points exceed the capacity %d" % (s, len(p), self.capacity))
            buf[s, :len(p)] = p
            cnt[s] = len(p)
        _lib.check(self.ctx.lib.ofb_tracker_set_points(self.h, _lib.ptr(buf), _lib.ptr(cnt)))

    def step(self, frames, imu, v_prior=None, want_points=False, want_kept=False, want_ego=False, want_robust=False):
        """frames: (H,W) / (S,H,W) uint8 (or (...,3) BGR when bgr=True), NumPy or CUDA tensor; imu: _lib.IMU_DTYPE
        (S,). Returns the _lib.TRACK_RESULT_DTYPE records (S,); with want_points additionally the list of (N,1,2)
        float32 point sets after the step; with want_kept the lists of (old, new) positions the solve used; with
        want_ego (needs set_ego_motion) the _lib.EGO_RESULT_DTYPE records (S,); with want_robust (needs set_robust) the
        _lib.ROBUST_RESULT_DTYPE records (S,), last."""
        if want_ego and not self.ego_motion:
            raise ValueError("want_ego needs ego-motion: StreamTracker(..., ego_motion=True) or set_ego_motion(True)")
        if want_robust and self.robust is None:
            raise ValueError("want_robust needs the robust solve: StreamTracker(..., robust=True) or set_robust(True)")
        S, h, w = self.n_streams, self.height, self.width
        shape = tuple(frames.shape)
        tail = (h, w, 3) if self.bgr else (h, w)
        if shape == tail:
            shape = (1,) + shape
        if shape != (S,) + tail:
            raise ValueError("frames must have shape %r, got %r" % ((S,) + tail, tuple(frames.shape)))
        if isinstance(frames, np.ndarray):
            frames = np.ascontiguousarray(frames, dtype=np.uint8)
        else:
            if not frames.is_contiguous():
                frames = frames.contiguous()
            if self.cfg.borrow_frames:
                self._held = (self._held + [frames])[-2:]
        bpp = 3 if self.bgr else 1
        imu = np.ascontiguousarray(imu, dtype=_lib.IMU_DTYPE).reshape(-1)
        if len(imu) != S:
            raise ValueError("one IMU sample per stream is required")
        if v_prior is not None:
            v_prior = np.ascontiguousarray(v_prior, dtype=np.float64).reshape(S, 3)
        res = np.zeros(S, _lib.TRACK_RESULT_DTYPE)
        ego = np.zeros(S, _lib.EGO_RESULT_DTYPE) if want_ego else None
        rob = np.zeros(S, _lib.ROBUST_RESULT_DTYPE) if want_robust else None
        pts = cnt = kp = kn = None
        if want_points:
            pts = np.zeros((S, self.capacity, 2), np.float32)
            cnt = np.zeros(S, np.int32)
        if want_kept:
            kp = np.zeros((S, self.capacity, 2), np.float32)
            kn = np.zeros((S, self.capacity, 2), np.float32)
        _lib.check(self.ctx.lib.ofb_tracker_step_robust(self.h, _lib.ptr(frames), bpp * w, bpp * w * h, _lib.ptr(imu),
                                                        _lib.ptr(v_prior), _lib.ptr(res), _lib.ptr(pts), _lib.ptr(cnt),
                                                        _lib.ptr(kp), _lib.ptr(kn), _lib.ptr(ego), _lib.ptr(rob)))
        out = [res]
        if want_points:
            out.append([pts[s, :cnt[s]].reshape(-1, 1, 2).copy() for s in range(S)])
        if want_kept:
            out.append([kp[s, :res["n_kept"][s]].copy() for s in range(S)])
            out.append([kn[s, :res["n_kept"][s]].copy() for s in range(S)])
        if want_ego:
            out.append(ego)
        if want_robust:
            out.append(rob)
        return out[0] if len(out) == 1 else tuple(out)


def exclusion_mask(points, radius, width, height, ctx=None):
    """The mask of the masked top-up (node:159-161): ones with cv2.circle(mask, (int(x), int(y)), radius, 0, FILLED)
    at every point. Returns (H,W) uint8."""
    ctx = ctx or _lib.default_context()
    p = np.ascontiguousarray(np.asarray(points, dtype=np.float32).reshape(-1, 2))
    m = np.zeros((int(height), int(width)), np.uint8)
    _lib.check(ctx.lib.ofb_tracker_render_mask(ctx.h, _lib.ptr(p) if len(p) else None, len(p), int(radius), int(width),
                                               int(height), _lib.ptr(m)))
    return m


class FleetTracker:
    """A fleet of camera streams sharded over the ranks of a torch.distributed group (SURVEY 8e: stream s lives on
    rank s mod world, no data-path collective). Every rank steps only its own streams through a local StreamTracker;
    `gather_velocities` merges the per-stream velocities of the last step into one (n_streams, 3) table on every rank
    with a single all-reduce (NCCL on the GPU box, gloo in the CPU tests).

    tracker_factory(n_local_streams, **kw) builds the local tracker (default: StreamTracker on this rank's GPU)."""

    def __init__(self, n_streams, width, height, group=None, tracker_factory=None, **tracker_kw):
        import torch.distributed as dist
        from .simulation import stream_shard
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.n_streams = int(n_streams)
        self.streams = stream_shard(self.n_streams, self.rank, self.world)
        if tracker_factory is None:
            def tracker_factory(n_local, **kw):
                return StreamTracker(width, height, n_streams=n_local, **kw)
        self.local = tracker_factory(len(self.streams), **tracker_kw) if self.streams else None
        self.last = None

    def select(self, per_stream):
        """this rank's rows of a per-stream array / list indexed by global stream id"""
        return [per_stream[s] for s in self.streams]

    def step(self, frames_local, imu_local, **kw):
        """frames_local / imu_local: this rank's streams in the order of `self.streams` (see `select`)."""
        if self.local is None:
            self.last = None
            return None
        out = self.local.step(frames_local, imu_local, **kw)
        self.last = out[0] if isinstance(out, tuple) else out
        return out

    def set_camera(self, camera):
        """StreamTracker.set_camera on this rank's streams"""
        if self.local is not None:
            self.local.set_camera(camera)

    def set_fb_threshold(self, threshold):
        """StreamTracker.set_fb_threshold on this rank's streams"""
        t = _fb_threshold(threshold)
        if self.local is not None:
            self.local.set_fb_threshold(t)

    def set_gyro_prediction(self, enable):
        """StreamTracker.set_gyro_prediction on this rank's streams (gyro_prediction=True at construction is passed to
        the local tracker with the other keywords)"""
        on = bool(_gyro_flag(enable))
        if self.local is not None:
            self.local.set_gyro_prediction(on)

    def set_ego_motion(self, enable):
        """StreamTracker.set_ego_motion on this rank's streams (ego_motion=True at construction is passed to the local
        tracker with the other keywords)"""
        on = _ego_flag(enable)
        if self.local is not None:
            self.local.set_ego_motion(on)

    def set_robust(self, robust):
        """StreamTracker.set_robust on this rank's streams (robust=... at construction is passed to the local tracker
        with the other keywords)"""
        cfg = _lib.robust_cfg(robust)
        if self.local is not None:
            self.local.set_robust(None if cfg is None else (cfg.c, cfg.iterations))

    def gather_velocities(self):
        """(n_streams, 3) velocities of the last step on every rank; rows of streams that did not solve (or have not
        stepped yet) are NaN. One all-reduce of an (n_streams, 4) table: velocity + a validity column (NaN cannot ride
        a sum)."""
        from .simulation import gather_stream_rows
        import torch.distributed as dist
        rows = np.zeros((len(self.streams), 4))
        if self.last is not None:
            ok = (self.last["flags"] & _lib.TRACK_SOLVED) != 0
            rows[:, :3] = np.where(ok[:, None], self.last["v"], 0.0)
            rows[:, 3] = ok
        if self.world == 1:
            table = rows
        else:
            dev = None
            if dist.get_backend(self.group) == "nccl":
                # a rank that owns no stream still takes part in the collective, from ITS OWN GPU
                import torch
                dev = torch.device("cuda", self.local.ctx.device if self.local is not None else torch.cuda.current_device())
            table = gather_stream_rows(rows, self.streams, self.n_streams, self.group, dev)
        out = table[:, :3].copy()
        out[table[:, 3] == 0] = np.nan
        return out

    def close(self):
        if self.local is not None:
            self.local.close()
            self.local = None
