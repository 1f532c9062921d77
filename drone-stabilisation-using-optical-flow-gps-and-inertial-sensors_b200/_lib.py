"""ctypes binding of libofb200.so (include/ofb200.h). No CPU fallback: every call needs the
CUDA library and a B200; a missing library or device raises immediately."""
import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# OFB200_LIB selects another build of the same library (the debug build with device-side index assertions,
# `python -m ofb200._build --debug` -> libofb200_dbg.so); there is still no CPU path behind it
LIB_PATH = os.environ.get("OFB200_LIB") or os.path.join(_HERE, "libofb200.so")

OFB_OK, OFB_E_INVALID, OFB_E_CUDA, OFB_E_NOMEM, OFB_E_UNSUPPORTED = 0, -1, -2, -3, -4
VARIANT_NODE, VARIANT_EXP, VARIANT_SIM, VARIANT_MODULE = 0, 1, 2, 3
VARIANTS = {"node": VARIANT_NODE, "exp": VARIANT_EXP, "sim": VARIANT_SIM}
TRACKER_VARIANTS = dict(VARIANTS, module=VARIANT_MODULE)
LK_USE_INITIAL_FLOW = 4
MC_MAX_POINTS = 256


class OfbError(RuntimeError):
    pass


class PairCfg(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("max_level", C.c_int), ("max_corners", C.c_int),
                ("quality", C.c_double), ("min_distance", C.c_double), ("block_size", C.c_int),
                ("win_w", C.c_int), ("win_h", C.c_int), ("max_count", C.c_int),
                ("eps", C.c_double), ("min_eig_thr", C.c_double), ("variant", C.c_int),
                ("cx", C.c_double), ("cy", C.c_double), ("pos_scale", C.c_double), ("flow_scale", C.c_double),
                ("detect", C.c_int)]


class Camera(C.Structure):
    """ofb_camera: K without skew, OpenCV's distortion coefficients (k1 k2 p1 p2 k3 k4 k5 k6), the fixed-point
    iteration count of the inverse lens model and the flow rate (u = (x_new - x_old) * rate)."""
    _fields_ = [("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double), ("dist", C.c_double * 8),
                ("n_dist", C.c_int), ("iterations", C.c_int), ("rate", C.c_double)]


class ImuSample(C.Structure):
    _fields_ = [("d", C.c_double), ("n", C.c_double * 3), ("w", C.c_double * 3), ("t", C.c_double * 3)]


class PairResult(C.Structure):
    _fields_ = [("v", C.c_double * 3), ("s", C.c_double * 3), ("res", C.c_double), ("rank", C.c_int),
                ("n_features", C.c_int), ("n_tracked", C.c_int), ("flags", C.c_int)]


class TrackerCfg(C.Structure):
    _fields_ = [("pair", PairCfg), ("n_streams", C.c_int), ("min_features", C.c_int), ("topup_mode", C.c_int),
                ("mask_radius", C.c_int), ("bgr_input", C.c_int), ("max_speed", C.c_double),
                ("dummy_value", C.c_double), ("gate_mode", C.c_int), ("gate_T", C.c_double), ("min_solve", C.c_int),
                ("borrow_frames", C.c_int), ("v_init", C.c_double * 3)]


class TrackResult(C.Structure):
    _fields_ = [("v", C.c_double * 3), ("s", C.c_double * 3), ("res", C.c_double), ("rank", C.c_int),
                ("flags", C.c_int), ("n_prev", C.c_int), ("n_tracked", C.c_int), ("n_kept", C.c_int),
                ("n_added", C.c_int), ("n_points", C.c_int)]


class McStep(C.Structure):
    _fields_ = [("v", C.c_double * 3), ("w", C.c_double * 3), ("n", C.c_double * 3), ("t", C.c_double * 3),
                ("height", C.c_double),
                ("ang_vel_sig", C.c_double), ("translation_sig", C.c_double), ("height_sig", C.c_double),
                ("flow_sig", C.c_double), ("position_sig", C.c_double), ("normal_sig", C.c_double),
                ("velocity_sig", C.c_double), ("true_vel", C.c_double * 3),
                ("n_points", C.c_int), ("pos_offset", C.c_int)]


class McSums(C.Structure):
    _fields_ = [("n", C.c_double), ("sum_dv", C.c_double * 3), ("sum_dv2", C.c_double * 3), ("sum_R", C.c_double)]


IMU_DTYPE = np.dtype([("d", "<f8"), ("n", "<f8", 3), ("w", "<f8", 3), ("t", "<f8", 3)])
RESULT_DTYPE = np.dtype([("v", "<f8", 3), ("s", "<f8", 3), ("res", "<f8"), ("rank", "<i4"),
                         ("n_features", "<i4"), ("n_tracked", "<i4"), ("flags", "<i4")], align=True)
TRACK_RESULT_DTYPE = np.dtype([("v", "<f8", 3), ("s", "<f8", 3), ("res", "<f8"), ("rank", "<i4"), ("flags", "<i4"),
                               ("n_prev", "<i4"), ("n_tracked", "<i4"), ("n_kept", "<i4"), ("n_added", "<i4"),
                               ("n_points", "<i4")], align=True)
TOPUP_APPEND_MASKED, TOPUP_APPEND, TOPUP_REPLACE = 0, 1, 2
TOPUP_MODES = {"node": TOPUP_APPEND_MASKED, "exp": TOPUP_APPEND, "module": TOPUP_REPLACE}
GATE_NONE, GATE_R_GE, GATE_R_LE = 0, 1, 2
TRACK_SOLVED, TRACK_OVERFLOW = 1, 2
PAIR_OVERFLOW = 2
MCSUMS_DTYPE = np.dtype([("n", "<f8"), ("sum_dv", "<f8", 3), ("sum_dv2", "<f8", 3), ("sum_R", "<f8")])

_lib = None
_lock = threading.Lock()

vp, i32, f64, u64, sz = C.c_void_p, C.c_int, C.c_double, C.c_uint64, C.c_size_t

_SIGNATURES = {
    "ofb_last_error": (C.c_char_p, []),
    "ofb_version": (i32, []),
    "ofb_ctx_create": (i32, [i32, C.POINTER(vp)]),
    "ofb_ctx_create_on_stream": (i32, [i32, vp, C.POINTER(vp)]),
    "ofb_ctx_destroy": (i32, [vp]),
    "ofb_ctx_sync": (i32, [vp]),
    "ofb_ctx_stream": (i32, [vp, C.POINTER(vp)]),
    "ofb_ctx_launch_count": (i32, [vp, C.POINTER(u64)]),
    "ofb_ctx_set_profile": (i32, [vp, i32]),
    "ofb_ctx_stage_times": (i32, [vp, C.POINTER(C.c_float), C.POINTER(u64)]),
    "ofb_timer_start": (i32, [vp]),
    "ofb_timer_stop": (i32, [vp, C.POINTER(C.c_float)]),
    "ofb_dev_alloc": (i32, [vp, sz, C.POINTER(vp)]),
    "ofb_dev_free": (i32, [vp, vp]),
    "ofb_host_alloc_pinned": (i32, [vp, sz, C.POINTER(vp)]),
    "ofb_host_free_pinned": (i32, [vp, vp]),
    "ofb_memcpy": (i32, [vp, vp, vp, sz]),
    "ofb_memcpy_async": (i32, [vp, vp, vp, sz]),
    "ofb_bgr2gray": (i32, [vp, vp, i32, i32, i32, vp, i32]),
    "ofb_pyramid": (i32, [vp, vp, i32, i32, i32, sz, i32, i32, C.POINTER(vp)]),
    "ofb_pyramid_bgr": (i32, [vp, vp, i32, i32, i32, sz, i32, i32, C.POINTER(vp)]),
    "ofb_pyr_free": (i32, [vp, vp]),
    "ofb_pyr_info": (i32, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
    "ofb_pyr_download": (i32, [vp, vp, i32, i32, vp, i32]),
    "ofb_good_features": (i32, [vp, vp, i32, i32, i32, vp, i32, i32, f64, f64, i32, vp, i32, C.POINTER(i32)]),
    "ofb_min_eig_map": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "ofb_pyrlk": (i32, [vp, vp, i32, vp, i32, vp, i32, i32, i32, i32, i32, f64, i32, f64, vp, vp, vp]),
    "ofb_solve_velocity": (i32, [vp, i32, vp, vp, i32, f64, vp, vp, vp, vp, vp, vp, vp]),
    "ofb_solve_velocity_batched": (i32, [vp, i32, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "ofb_solve_velocity_module": (i32, [vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
    "ofb_advect_points": (i32, [vp, vp, i32, vp, vp, f64, vp, vp, i32, vp, vp, vp]),
    "ofb_generate_flow": (i32, [vp, vp, i32, vp, vp, f64, vp, vp, vp]),
    "ofb_r_tilde": (i32, [vp, vp, vp, i32, i32, vp, vp, f64, vp, vp]),
    "ofb_feasibility": (i32, [vp, vp, vp, vp, i32, vp, vp, vp, vp]),
    "ofb_frame_pairs": (i32, [vp, C.POINTER(PairCfg), i32, vp, vp, i32, sz, vp, vp, vp, vp, vp, vp, vp]),
    "ofb_tracker_create": (i32, [vp, C.POINTER(TrackerCfg), C.POINTER(vp)]),
    "ofb_tracker_destroy": (i32, [vp]),
    "ofb_tracker_reset": (i32, [vp]),
    "ofb_tracker_capacity": (i32, [vp, C.POINTER(i32)]),
    "ofb_tracker_set_points": (i32, [vp, vp, vp]),
    "ofb_tracker_step": (i32, [vp, vp, i32, sz, vp, vp, vp, vp, vp, vp, vp]),
    "ofb_tracker_graph_info": (i32, [vp, C.POINTER(u64), C.POINTER(i32)]),
    "ofb_tracker_render_mask": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "ofb_tracker_set_camera": (i32, [vp, C.POINTER(Camera)]),
    "ofb_undistort_points": (i32, [vp, C.POINTER(Camera), vp, i32, vp, vp]),
    "ofb_frame_pairs_cam": (i32, [vp, C.POINTER(PairCfg), C.POINTER(Camera), i32, vp, vp, i32, sz, vp, vp, vp, vp, vp, vp, vp]),
    "ofb_pyrlk_fb": (i32, [vp, vp, i32, vp, i32, vp, i32, i32, i32, i32, i32, f64, f64, f64, vp, vp, vp, vp]),
    "ofb_frame_pairs_fb": (i32, [vp, C.POINTER(PairCfg), C.POINTER(Camera), f64, i32, vp, vp, i32, sz, vp, vp, vp, vp, vp, vp, vp]),
    "ofb_tracker_set_fb_check": (i32, [vp, f64]),
    "ofb_mc_sweep": (i32, [vp, vp, i32, i32, vp, vp, i32, u64, u64, u64, i32, vp, vp, vp]),
    "ofb_mc_sweep_multi": (i32, [vp, i32, vp, i32, i32, vp, vp, i32, u64, u64, u64, i32, vp]),
    "ofb_mc_feas": (i32, [vp, vp, i32, vp, vp, u64, u64, u64, vp]),
    "ofb_minmax": (i32, [vp, vp, sz, C.POINTER(f64), C.POINTER(f64)]),
    "ofb_histogram": (i32, [vp, vp, sz, f64, f64, i32, vp]),
}


def load():
    """Load libofb200.so; raises OfbError when it is missing (there is no CPU path)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise OfbError("libofb200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`; "
                               "there is no CPU fallback." % LIB_PATH)
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc):
    if rc == OFB_OK:
        return
    msg = load().ofb_last_error().decode("utf-8", "replace")
    if rc == OFB_E_INVALID:
        raise ValueError(msg)
    if rc == OFB_E_NOMEM:
        raise MemoryError(msg)
    raise OfbError("libofb200 error %d: %s" % (rc, msg))


def ptr(a):
    """void* of a numpy array, a torch tensor (host or CUDA), an int address or None."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    if isinstance(a, (C.Structure, C.Array)):
        return C.cast(C.byref(a), C.c_void_p)
    raise TypeError("cannot take the address of %r" % type(a))


class Context:
    """One CUDA device + one stream + scratch arenas (ofb_ctx). Not thread-safe; make one per thread."""

    def __init__(self, device=None, stream=None):
        lib = load()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        h = vp()
        if stream is None:
            check(lib.ofb_ctx_create(int(device), C.byref(h)))
        else:
            check(lib.ofb_ctx_create_on_stream(int(device), vp(int(stream)), C.byref(h)))
        self.h = h
        self.device = int(device)
        self.lib = lib

    def close(self):
        if getattr(self, "h", None):
            self.lib.ofb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        check(self.lib.ofb_ctx_sync(self.h))

    def launch_count(self):
        n = u64()
        check(self.lib.ofb_ctx_launch_count(self.h, C.byref(n)))
        return n.value

    def set_profile(self, enable=True):
        check(self.lib.ofb_ctx_set_profile(self.h, 1 if enable else 0))

    def stage_times(self):
        """(ms[5] accumulated over calls: pyramids, lambda_min+NMS, selection, LK, solve; n_calls)"""
        ms = (C.c_float * 5)()
        n = u64()
        check(self.lib.ofb_ctx_stage_times(self.h, ms, C.byref(n)))
        return [float(x) for x in ms], n.value

    def timer_start(self):
        check(self.lib.ofb_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        check(self.lib.ofb_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def dev_alloc(self, nbytes):
        p = vp()
        check(self.lib.ofb_dev_alloc(self.h, nbytes, C.byref(p)))
        return p.value

    def dev_free(self, p):
        check(self.lib.ofb_dev_free(self.h, vp(p)))

    def pinned_array(self, shape, dtype):
        """numpy array backed by pinned host memory (kept alive by the returned object's base)."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = vp()
        check(self.lib.ofb_host_alloc_pinned(self.h, max(n, 1), C.byref(p)))
        buf = (C.c_uint8 * max(n, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        self._pinned = getattr(self, "_pinned", [])
        self._pinned.append(p.value)
        return arr

    def memcpy(self, dst, src, nbytes):
        check(self.lib.ofb_memcpy(self.h, ptr(dst), ptr(src), nbytes))


_default = threading.local()


def default_context():
    ctx = getattr(_default, "ctx", None)
    if ctx is None:
        ctx = Context()
        _default.ctx = ctx
    return ctx
