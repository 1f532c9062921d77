"""Stages 0-3 host mirror: cv2-shaped entry points so the reference's callers can swap `cv2.` for this
module (SURVEY 8b):

    goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance, mask=None, blockSize=3, ...)
        velocity_measurment_node:120,163; evaluate_exp.py:66,106; of_module.py:44,86; of_library.py:238
    calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, nextPts, winSize=, maxLevel=, criteria=, ...)
        velocity_measurment_node:133; evaluate_exp.py:98; of_module.py:88; of_library.py:249
    cvtColor(img, COLOR_BGR2GRAY)  velocity_measurment_node:113
    frame_pairs(...)               the per-frame dataflow of node:224-267 / evaluate_exp.py:77-120, batched
    undistortPoints(src, cameraMatrix, distCoeffs, R=None, P=None)    cv2.undistortPoints (5 iterations)
    undistortPointsIter(src, cameraMatrix, distCoeffs, R, P, criteria) with the COUNT criterion
    track_forward_backward(prevImg, nextImg, prevPts, threshold, ...)  LK forwards + backwards, lk_track.py's check
"""
import ctypes as C
import numbers

import numpy as np

from . import _lib

COLOR_BGR2GRAY = 6            # cv2.COLOR_BGR2GRAY
TERM_CRITERIA_COUNT, TERM_CRITERIA_EPS = 1, 2
OPTFLOW_USE_INITIAL_FLOW = 4


def _gray(img, name="image"):
    a = np.asarray(img)
    if a.dtype != np.uint8 or a.ndim != 2:
        raise ValueError("%s must be a 2-D uint8 array" % name)
    return np.ascontiguousarray(a)


def cvtColor(src, code=COLOR_BGR2GRAY, ctx=None):
    if code != COLOR_BGR2GRAY:
        raise ValueError("only COLOR_BGR2GRAY is on the hot path")
    ctx = ctx or _lib.default_context()
    a = np.ascontiguousarray(np.asarray(src))
    if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
        raise ValueError("src must be HxWx3 uint8")
    h, w, _ = a.shape
    out = np.empty((h, w), np.uint8)
    _lib.check(ctx.lib.ofb_bgr2gray(ctx.h, _lib.ptr(a), w, h, 3 * w, _lib.ptr(out), w))
    return out


class Pyramid:
    """Device-resident Gaussian pyramid(s) of n_images same-sized frames (ofb_pyr)."""

    def __init__(self, images, max_level, ctx=None, bgr=False):
        """bgr=True: images are BGR8 frames (H,W,3) / (N,H,W,3); the grey conversion (cv2.cvtColor at
        velocity_measurment_node:113) is fused into the first pyramid step (ofb_pyramid_bgr)."""
        self.ctx = ctx or _lib.default_context()
        a = np.asarray(images)
        nd = (3, 4) if bgr else (2, 3)
        if a.dtype != np.uint8 or a.ndim not in nd or (bgr and a.shape[-1] != 3):
            raise ValueError("images must be uint8 (H,W) or (N,H,W)" + (" with 3 channels last" if bgr else ""))
        a = np.ascontiguousarray(a)
        if a.ndim == nd[0]:
            a = a[None]
        n, h, w = a.shape[:3]
        self._keep = a
        hdl = C.c_void_p()
        if bgr:
            _lib.check(self.ctx.lib.ofb_pyramid_bgr(self.ctx.h, _lib.ptr(a), w, h, 3 * w, 3 * w * h, n, int(max_level), C.byref(hdl)))
        else:
            _lib.check(self.ctx.lib.ofb_pyramid(self.ctx.h, _lib.ptr(a), w, h, w, w * h, n, int(max_level), C.byref(hdl)))
        self.h = hdl
        ni, nl = C.c_int(), C.c_int()
        ws = (C.c_int * 16)(); hs = (C.c_int * 16)(); ps = (C.c_int * 16)()
        _lib.check(self.ctx.lib.ofb_pyr_info(self.h, C.byref(ni), C.byref(nl), ws, hs, ps))
        self.n_images, self.n_levels = ni.value, nl.value
        self.sizes = [(ws[i], hs[i]) for i in range(nl.value)]

    def level(self, level, image=0):
        w, h = self.sizes[level]
        out = np.empty((h, w), np.uint8)
        _lib.check(self.ctx.lib.ofb_pyr_download(self.ctx.h, self.h, image, level, _lib.ptr(out), w))
        return out

    def close(self):
        if getattr(self, "h", None) and self.ctx.h:
            self.ctx.lib.ofb_pyr_free(self.ctx.h, self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def buildPyramid(img, maxlevel, ctx=None):
    """cv2.buildPyramid-shaped helper: list of maxlevel+1 images (level 0 = input)."""
    p = Pyramid(_gray(img), maxlevel, ctx)
    try:
        return [p.level(l) for l in range(p.n_levels)]
    finally:
        p.close()


def pyrDown(img, ctx=None):
    return buildPyramid(img, 1, ctx)[1]


def cornerMinEigenVal(image, blockSize, ksize=3, ctx=None):
    if ksize != 3:
        raise ValueError("only the aperture-3 Sobel used by goodFeaturesToTrack is supported")
    ctx = ctx or _lib.default_context()
    a = _gray(image)
    h, w = a.shape
    out = np.empty((h, w), np.float32)
    _lib.check(ctx.lib.ofb_min_eig_map(ctx.h, _lib.ptr(a), w, h, w, int(blockSize), _lib.ptr(out)))
    return out


def goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance, mask=None, blockSize=3,
                        useHarrisDetector=False, k=0.04, ctx=None, **kw):
    """-> (N,1,2) float32, or None when no corner qualifies (as cv2)."""
    if useHarrisDetector:
        raise ValueError("the Harris variant is not on the reference's path (every call site uses min-eigenvalue)")
    if "corners" in kw or "gradientSize" in kw and kw["gradientSize"] != 3:
        raise ValueError("unsupported argument")
    ctx = ctx or _lib.default_context()
    a = _gray(image)
    h, w = a.shape
    m = None
    if mask is not None:
        m = np.ascontiguousarray(np.asarray(mask))
        if m.dtype != np.uint8 or m.shape != a.shape:
            raise ValueError("mask must be uint8 with the image's shape")
    maxCorners = int(maxCorners)
    cap = maxCorners if maxCorners > 0 else w * h
    xy = np.empty((cap, 2), np.float32)
    n = C.c_int(0)
    _lib.check(ctx.lib.ofb_good_features(ctx.h, _lib.ptr(a), w, h, w, _lib.ptr(m), w, maxCorners, float(qualityLevel),
                                         float(minDistance), int(blockSize), _lib.ptr(xy), cap, C.byref(n)))
    if n.value == 0:
        return None
    return xy[:n.value].reshape(-1, 1, 2).copy()


def _criteria(criteria):
    # cv2.calcOpticalFlowPyrLK: a missing COUNT flag means 30 iterations, a missing EPS flag 0.01
    typ, count, eps = criteria
    count = int(count) if (int(typ) & TERM_CRITERIA_COUNT) else 30
    eps = float(eps) if (int(typ) & TERM_CRITERIA_EPS) else 0.01
    return count, eps


def calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, nextPts=None, status=None, err=None, winSize=(21, 21),
                         maxLevel=3, criteria=(TERM_CRITERIA_COUNT | TERM_CRITERIA_EPS, 30, 0.01), flags=0,
                         minEigThreshold=1e-4, ctx=None):
    """-> (nextPts (N,1,2) f32, status (N,1) u8, err (N,1) f32). prevImg/nextImg may be uint8 frames or
    Pyramid objects (so a caller can keep the previous frame's pyramid, which cv2 rebuilds every call)."""
    ctx = ctx or _lib.default_context()
    pts = np.ascontiguousarray(np.asarray(prevPts, dtype=np.float32).reshape(-1, 2))
    n = len(pts)
    own = []
    pp = prevImg if isinstance(prevImg, Pyramid) else Pyramid(_gray(prevImg, "prevImg"), maxLevel, ctx)
    if pp is not prevImg:
        own.append(pp)
    pn = nextImg if isinstance(nextImg, Pyramid) else Pyramid(_gray(nextImg, "nextImg"), maxLevel, ctx)
    if pn is not nextImg:
        own.append(pn)
    try:
        if pp.sizes[0] != pn.sizes[0]:
            raise ValueError("prevImg and nextImg must have the same size")
        out = np.zeros((n, 2), np.float32)
        if flags & OPTFLOW_USE_INITIAL_FLOW:
            if nextPts is None:
                raise ValueError("OPTFLOW_USE_INITIAL_FLOW needs nextPts")
            out[:] = np.asarray(nextPts, dtype=np.float32).reshape(-1, 2)
        st = np.zeros(n, np.uint8)
        er = np.zeros(n, np.float32)
        count, eps = _criteria(criteria)
        if n:
            _lib.check(ctx.lib.ofb_pyrlk(ctx.h, pp.h, 0, pn.h, 0, _lib.ptr(pts), n, int(winSize[0]), int(winSize[1]),
                                         int(maxLevel), count, eps, int(flags) & OPTFLOW_USE_INITIAL_FLOW,
                                         float(minEigThreshold), _lib.ptr(out), _lib.ptr(st), _lib.ptr(er)))
        return out.reshape(-1, 1, 2), st.reshape(-1, 1), er.reshape(-1, 1)
    finally:
        for p in own:
            p.close()


def _fb_threshold(threshold):
    """The forward-backward check's threshold as the C ABI takes it: None or 0 = off (0.0), else a positive number of
    pixels (+inf allowed). Raises ValueError for a negative, NaN or non-numeric value."""
    if threshold is None:
        return 0.0
    if isinstance(threshold, (bool, np.bool_)) or not isinstance(threshold, numbers.Real):
        raise ValueError("fb threshold must be a number of pixels, got %r" % (threshold,))
    t = float(threshold)
    if not t >= 0.0:
        raise ValueError("fb threshold must be >= 0 (0 or None = off), got %r" % (threshold,))
    return t


def track_forward_backward(prevImg, nextImg, prevPts, threshold=1.0, winSize=(21, 21), maxLevel=3,
                           criteria=(TERM_CRITERIA_COUNT | TERM_CRITERIA_EPS, 30, 0.01), minEigThreshold=1e-4, ctx=None):
    """calcOpticalFlowPyrLK forwards, then backwards from the forward result, in one launch (the check of OpenCV's
    samples/python/lk_track.py). -> (nextPts (N,1,2) f32, status (N,1) u8, err (N,1) f32, fbErr (N,) f32).
    nextPts and err are the forward call's; status is 1 where the forward and the backward status are 1 and
    fbErr = max(|x0 - x0r|, |y0 - y0r|) < threshold; fbErr is +inf where either pass lost the point (everywhere
    when threshold is 0 or None: then status is the forward one). Defaults are calcOpticalFlowPyrLK's; prevImg /
    nextImg may be Pyramid objects."""
    thr = _fb_threshold(threshold)
    ctx = ctx or _lib.default_context()
    pts = np.ascontiguousarray(np.asarray(prevPts, dtype=np.float32).reshape(-1, 2))
    n = len(pts)
    own = []
    pp = prevImg if isinstance(prevImg, Pyramid) else Pyramid(_gray(prevImg, "prevImg"), maxLevel, ctx)
    if pp is not prevImg:
        own.append(pp)
    pn = nextImg if isinstance(nextImg, Pyramid) else Pyramid(_gray(nextImg, "nextImg"), maxLevel, ctx)
    if pn is not nextImg:
        own.append(pn)
    try:
        if pp.sizes[0] != pn.sizes[0]:
            raise ValueError("prevImg and nextImg must have the same size")
        out = np.zeros((n, 2), np.float32)
        st = np.zeros(n, np.uint8)
        er = np.zeros(n, np.float32)
        fb = np.full(n, np.inf, np.float32)
        count, eps = _criteria(criteria)
        if n:
            _lib.check(ctx.lib.ofb_pyrlk_fb(ctx.h, pp.h, 0, pn.h, 0, _lib.ptr(pts), n, int(winSize[0]), int(winSize[1]),
                                            int(maxLevel), count, eps, float(minEigThreshold), thr, _lib.ptr(out),
                                            _lib.ptr(st), _lib.ptr(er), _lib.ptr(fb)))
        return out.reshape(-1, 1, 2), st.reshape(-1, 1), er.reshape(-1, 1), fb
    finally:
        for p in own:
            p.close()


# The velocity paths iterate the inverse lens model 20 times by default, cv2.undistortPoints 5 times. For a wide-angle
# k1 = -0.3 lens (1280x720, fx = 900 px) 5 iterations leave up to 0.48 px of error at the image edge against the
# converged inverse, 10 leave 1.3e-3 px and 20 leave 1e-8 px. A bias of 0.48 px enters x and u directly and with them
# the velocity, so the velocity paths pay for the converged inverse (the cost is a few hundred fp64 operations per point).
CAMERA_ITERATIONS = 20


def make_camera(cameraMatrix, distCoeffs, rate=1.0, iterations=CAMERA_ITERATIONS):
    """ofb_camera from OpenCV's K (3x3, no skew) and D (None or 4, 5 or 8 coefficients: plumb_bob /
    rational_polynomial). rate: u = (x_new - x_old) * rate (the frame rate 1/dt for a velocity in m/s)."""
    K = np.asarray(cameraMatrix, dtype=np.float64)
    if K.size != 9:
        raise ValueError("cameraMatrix must be 3x3")
    K = K.reshape(3, 3)
    D = np.zeros(0) if distCoeffs is None else np.asarray(distCoeffs, dtype=np.float64).ravel()
    if len(D) not in (0, 4, 5, 8):
        raise ValueError("distCoeffs must have 0, 4, 5 or 8 entries (got %d)" % len(D))
    if not (np.isfinite(K).all() and np.isfinite(D).all() and np.isfinite(rate)):
        raise ValueError("non-finite camera parameter")
    if K[0, 1] != 0 or K[1, 0] != 0 or K[2, 0] != 0 or K[2, 1] != 0 or K[2, 2] != 1:
        raise ValueError("cameraMatrix must be [[fx, 0, cx], [0, fy, cy], [0, 0, 1]] (no skew)")
    if K[0, 0] <= 0 or K[1, 1] <= 0:
        raise ValueError("fx and fy must be positive")
    if not rate > 0:
        raise ValueError("rate must be positive")
    if int(iterations) != iterations or not 1 <= int(iterations) <= 1000:
        raise ValueError("iterations must be an integer in 1..1000")
    cam = _lib.Camera()
    cam.fx, cam.fy, cam.cx, cam.cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    cam.dist[:len(D)] = [float(d) for d in D]
    cam.n_dist, cam.iterations, cam.rate = len(D), int(iterations), float(rate)
    return cam


def as_camera(camera):
    """The `camera=` argument of the velocity paths: None, an _lib.Camera, or (K, D, rate[, iterations])."""
    if camera is None or isinstance(camera, _lib.Camera):
        return camera
    if not isinstance(camera, (tuple, list)) or len(camera) not in (3, 4):
        raise ValueError("camera must be (K, D, rate) or (K, D, rate, iterations)")
    return make_camera(*camera)


def _rectification(R, P):
    """H = P[:, :3] @ R as cvUndistortPointsInternal forms it (sums in index order), None for the identity."""
    if R is None and P is None:
        return None
    Rm = np.eye(3) if R is None else np.asarray(R, dtype=np.float64)
    if Rm.size != 9:
        raise ValueError("R must be 3x3")
    Rm = Rm.reshape(3, 3)
    if P is None:
        H = Rm.copy()
    else:
        Pm = np.asarray(P, dtype=np.float64)
        if Pm.shape not in ((3, 3), (3, 4)):
            raise ValueError("P must be 3x3 or 3x4")
        H = np.zeros((3, 3))
        for i in range(3):
            for j in range(3):
                H[i, j] = Pm[i, 0] * Rm[0, j] + Pm[i, 1] * Rm[1, j] + Pm[i, 2] * Rm[2, j]
    if not np.isfinite(H).all():
        raise ValueError("non-finite entry in R or P")
    return np.ascontiguousarray(H)


def undistortPointsIter(src, cameraMatrix, distCoeffs, R, P, criteria, ctx=None):
    """cv2.undistortPointsIter with the COUNT criterion: src (N,2) / (N,1,2) float32 or float64 pixels ->
    (N,1,2) of src's dtype (normalised coordinates, or rectified / projected by P @ R)."""
    typ, count, _ = criteria
    if int(typ) & TERM_CRITERIA_EPS or not int(typ) & TERM_CRITERIA_COUNT:
        raise ValueError("only the TERM_CRITERIA_COUNT criterion is supported")
    a = np.asarray(src)
    if a.dtype not in (np.float32, np.float64) or a.ndim not in (2, 3) or a.shape[-1] != 2 or (a.ndim == 3 and a.shape[1] != 1):
        raise ValueError("src must be an (N,2) or (N,1,2) float32 / float64 array")
    cam = make_camera(cameraMatrix, distCoeffs, 1.0, count)
    H = _rectification(R, P)
    pts = np.ascontiguousarray(a.reshape(-1, 2), dtype=np.float64)
    out = np.empty_like(pts)
    if len(pts):
        ctx = ctx or _lib.default_context()
        _lib.check(ctx.lib.ofb_undistort_points(ctx.h, C.byref(cam), _lib.ptr(pts), len(pts), _lib.ptr(H), _lib.ptr(out)))
    return out.astype(a.dtype).reshape(-1, 1, 2)


def undistortPoints(src, cameraMatrix, distCoeffs, R=None, P=None, ctx=None):
    """cv2.undistortPoints: 5 fixed-point iterations of the inverse lens model."""
    return undistortPointsIter(src, cameraMatrix, distCoeffs, R, P, (TERM_CRITERIA_COUNT, 5, 0), ctx=ctx)


def gyro_predict(points, omega, camera=None, cfg=None, ctx=None, **pinhole):
    """Where each pixel point lands when the camera rotates by the gyro rate `omega` (3 floats, rad per unit of time)
    over one frame interval: the initial flow the velocity paths give LK with gyro_prediction=True (include/ofb200.h,
    ofb_gyro_predict). points (N,2) / (N,1,2) -> (N,1,2) float32.
    camera: (K, D, rate[, iterations]) or make_camera(...): the lens model, dt = 1 / rate. Otherwise the pinhole of
    `cfg` (make_pair_cfg) or of make_pair_cfg's keywords in **pinhole (width, height, principal, pos_scale, flow_scale),
    with dt = pos_scale / flow_scale."""
    cam = as_camera(camera)
    w = np.asarray(omega, dtype=np.float64).ravel()
    if w.shape != (3,):
        raise ValueError("omega must have 3 entries")
    if cam is None:
        if cfg is None:
            pin = dict(pinhole)
            width, height = pin.pop("width", 0), pin.pop("height", 0)
            if pin.get("principal") is None and not (width and height):
                raise ValueError("the pinhole needs cfg, or principal=, or width= and height=")
            cfg = make_pair_cfg(width, height, 1, **pin)
        elif pinhole:
            raise ValueError("pass either cfg or pinhole keywords, not both")
        if cfg.flow_scale == 0 or not np.isfinite(cfg.pos_scale / cfg.flow_scale) or cfg.pos_scale == 0:
            raise ValueError("the pinhole needs flow_scale != 0 and a finite, non-zero pos_scale / flow_scale")
    elif cfg is not None or pinhole:
        raise ValueError("pass either camera or a pinhole, not both")
    a = np.asarray(points)
    if a.ndim not in (2, 3) or a.shape[-1] != 2 or (a.ndim == 3 and a.shape[1] != 1):
        raise ValueError("points must be an (N,2) or (N,1,2) array")
    pts = np.ascontiguousarray(a.reshape(-1, 2), dtype=np.float32)
    out = np.empty_like(pts)
    if len(pts):
        ctx = ctx or _lib.default_context()
        _lib.check(ctx.lib.ofb_gyro_predict(ctx.h, C.byref(cfg) if cfg is not None else None,
                                            C.byref(cam) if cam is not None else None, _lib.ptr(pts), len(pts),
                                            _lib.ptr(np.ascontiguousarray(w)), _lib.ptr(out)))
    return out.reshape(-1, 1, 2)


def _gyro_flag(gyro_prediction):
    if not isinstance(gyro_prediction, (bool, np.bool_)):
        raise ValueError("gyro_prediction must be True or False, got %r" % (gyro_prediction,))
    return 1 if gyro_prediction else 0


def make_pair_cfg(width, height, max_corners, quality=0.01, min_distance=10.0, block_size=7, win=(15, 15),
                  max_level=3, criteria=(3, 20, 0.03), min_eig_thr=1e-4, variant="node", principal=None,
                  pos_scale=1.0, flow_scale=1.0, detect=True):
    from .of_library import pix_trans
    cfg = _lib.PairCfg()
    cfg.width, cfg.height, cfg.max_level, cfg.max_corners = int(width), int(height), int(max_level), int(max_corners)
    cfg.quality, cfg.min_distance, cfg.block_size = float(quality), float(min_distance), int(block_size)
    cfg.win_w, cfg.win_h = int(win[0]), int(win[1])
    cfg.max_count, cfg.eps = _criteria(criteria)
    cfg.min_eig_thr = float(min_eig_thr)
    cfg.variant = _lib.TRACKER_VARIANTS[variant]       # 'module' is accepted by the tracker only (the C side checks)
    c = principal if principal is not None else pix_trans((width, height))
    cfg.cx, cfg.cy = float(c[0]), float(c[1])
    cfg.pos_scale, cfg.flow_scale = float(pos_scale), float(flow_scale)
    cfg.detect = 1 if detect else 0
    return cfg


def _ego_flag(ego_motion):
    if not isinstance(ego_motion, (bool, np.bool_)):
        raise ValueError("ego_motion must be True or False, got %r" % (ego_motion,))
    return bool(ego_motion)


def frame_pairs(prev, nxt, imu, cfg, pts_in=None, n_in=None, want_tracks=False, ctx=None, on_overflow="raise", camera=None,
                fb_threshold=None, gyro_prediction=False, ego_motion=False, robust=None):
    """Batched detect(+)track+solve. prev/nxt: (N,H,W) uint8 numpy arrays (host) or CUDA tensors;
    imu: structured array _lib.IMU_DTYPE (N,). Returns a structured array _lib.RESULT_DTYPE (N,)
    (and prev_pts, next_pts, status when want_tracks).
    A pair whose detector ran out of candidate slots (plateau images: more than w*h/4 + 1024 local maxima above the
    quality threshold) carries `flags & PAIR_OVERFLOW`; its feature list is truncated, so by default that raises
    OfbError (on_overflow="ignore" returns the flagged records instead).
    camera: (K, D, rate[, iterations]) or make_camera(...): the solve sees x = undistort(p_new) and
    u = (undistort(p_new) - undistort(p_old)) * rate instead of cfg's pinhole (cx, cy, pos_scale, flow_scale);
    iterations default to CAMERA_ITERATIONS.
    fb_threshold: None / 0 = off; T > 0 = forward-backward check of every track (track_forward_backward): a track that
    does not return within T px counts as lost (status 0, not in n_tracked, not in the solve). It runs on pixel
    positions, before the camera model.
    gyro_prediction: LK starts each track from where the pair's gyro rate imu["w"] rotates it (gyro_predict, with
    `camera` or cfg's pinhole) instead of from the point itself; with fb_threshold the backward pass starts from
    p1 + (p0 - guess).
    ego_motion: also estimate every pair's angular rate from its tracks together with the velocity (velocity.
    solve_ego_motion on the points the pair's solve uses; the gyro sample is not used there): the _lib.EGO_RESULT_DTYPE
    records (N,) are appended as the last element of the return. The standard results do not change.
    robust: None / False = off; True = the robust velocity solve (velocity.solve_velocity_robust, c = 4, 10 iterations)
    of every pair on the points its solve uses; (c, iterations) sets them. The _lib.ROBUST_RESULT_DTYPE records (N,)
    are appended as the last element of the return, after the ego records. The standard results do not change."""
    thr = _fb_threshold(fb_threshold)
    ego_on = _ego_flag(ego_motion)
    rcfg = _lib.robust_cfg(robust)
    gyro = _gyro_flag(gyro_prediction)
    cam = as_camera(camera)
    if gyro and cam is None and (cfg.flow_scale == 0 or cfg.pos_scale == 0 or not np.isfinite(cfg.pos_scale / cfg.flow_scale)):
        raise ValueError("gyro_prediction with the pinhole needs flow_scale != 0 and a finite, non-zero "
                         "pos_scale / flow_scale")
    ctx = ctx or _lib.default_context()
    n = int(prev.shape[0])
    h, w = int(prev.shape[1]), int(prev.shape[2])
    if (h, w) != (cfg.height, cfg.width) or tuple(nxt.shape) != tuple(prev.shape):
        raise ValueError("frame shapes do not match the configuration")
    if isinstance(prev, np.ndarray):
        prev = np.ascontiguousarray(prev, dtype=np.uint8)
        nxt = np.ascontiguousarray(nxt, dtype=np.uint8)
    imu = np.ascontiguousarray(imu, dtype=_lib.IMU_DTYPE)
    if len(imu) != n:
        raise ValueError("one IMU sample per pair is required")
    res = np.zeros(n, _lib.RESULT_DTYPE)
    ego = np.zeros(n, _lib.EGO_RESULT_DTYPE) if ego_on else None
    rob = np.zeros(n, _lib.ROBUST_RESULT_DTYPE) if rcfg is not None else None
    K = cfg.max_corners
    pp = pn = st = None
    if want_tracks:
        pp = np.zeros((n, K, 2), np.float32)
        pn = np.zeros((n, K, 2), np.float32)
        st = np.zeros((n, K), np.uint8)
    if pts_in is not None:
        pts_in = np.ascontiguousarray(pts_in, dtype=np.float32)
        n_in = np.ascontiguousarray(n_in, dtype=np.int32)
    _lib.check(ctx.lib.ofb_frame_pairs_robust(ctx.h, C.byref(cfg), C.byref(cam) if cam is not None else None, thr, gyro, n,
                                              _lib.ptr(prev), _lib.ptr(nxt), w, w * h, _lib.ptr(imu), _lib.ptr(pts_in),
                                              _lib.ptr(n_in), _lib.ptr(res), _lib.ptr(ego),
                                              C.byref(rcfg) if rcfg is not None else None, _lib.ptr(rob), _lib.ptr(pp),
                                              _lib.ptr(pn), _lib.ptr(st)))
    if on_overflow == "raise" and (res["flags"] & _lib.PAIR_OVERFLOW).any():
        bad = np.nonzero(res["flags"] & _lib.PAIR_OVERFLOW)[0]
        raise _lib.OfbError("frame_pairs: detector candidate buffer overflowed for pair(s) %s: the image has more than "
                            "w*h/4 + 1024 local maxima above the quality threshold (plateaus)" % bad[:8].tolist())
    out = (res, pp, pn, st) if want_tracks else (res,)
    if ego_on:
        out = out + (ego,)
    if rob is not None:
        out = out + (rob,)
    return out if len(out) > 1 else out[0]


def frame_sequence(frames, imu, cfg, want_tracks=False, ctx=None, on_overflow="raise", camera=None, fb_threshold=None,
                   gyro_prediction=False, ego_motion=False, robust=None):
    """One camera stream: frames (N+1,H,W) uint8 -> N consecutive pairs (frame i, frame i+1), as
    velocity_measurment_node:224-267 sees them (it keeps the previous callback's image). Passing the two views
    of ONE buffer lets the library upload every frame and build its pyramid once (`next == prev + image_stride`
    is the C ABI's sequence layout, include/ofb200.h)."""
    if isinstance(frames, np.ndarray):
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
    return frame_pairs(frames[:-1], frames[1:], imu, cfg, want_tracks=want_tracks, ctx=ctx, on_overflow=on_overflow,
                       camera=camera, fb_threshold=fb_threshold, gyro_prediction=gyro_prediction, ego_motion=ego_motion,
                       robust=robust)

