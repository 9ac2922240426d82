"""ctypes binding of libklt_b200.so (include/klt_b200.h).  No fallback: if the library or a B200 is
missing, every entry point raises."""
import ctypes
import os
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KLT_LIB_PATH") or os.path.join(_PKG, "lib", "libklt_b200.so")   # override: A/B runs of another build

KLT_MAX_LEVELS = 16
KLT_MAX_WIN_AREA = 4096
KLT_MAX_GRID_CELLS = 1024
KLT_MAX_SUBPIX_WIN = 15
KLT_MAX_CLAHE_TILES = 65536
TERM_COUNT, TERM_EPS = 1, 2
OPTFLOW_USE_INITIAL_FLOW, OPTFLOW_LK_GET_MIN_EIGENVALS = 4, 8

KLT_OK = 0
KLT_ERR_INVALID_ARG, KLT_ERR_UNSUPPORTED, KLT_ERR_NO_DEVICE, KLT_ERR_OUT_OF_MEMORY, KLT_ERR_INTERNAL = -1, -2, -3, -4, -5


class klt_level(ctypes.Structure):
    _fields_ = [("w", ctypes.c_int32), ("h", ctypes.c_int32), ("pitch", ctypes.c_int64),
                ("batch_stride", ctypes.c_int64), ("offset", ctypes.c_int64)]


class klt_pyr_layout(ctypes.Structure):
    _fields_ = [("top", ctypes.c_int32), ("batch", ctypes.c_int32), ("level", klt_level * KLT_MAX_LEVELS),
                ("bytes", ctypes.c_int64)]


class klt_lk_params(ctypes.Structure):
    _fields_ = [("win_w", ctypes.c_int32), ("win_h", ctypes.c_int32), ("crit_type", ctypes.c_int32),
                ("crit_max_count", ctypes.c_int32), ("crit_eps", ctypes.c_double), ("flags", ctypes.c_int32),
                ("min_eig_threshold", ctypes.c_double)]


class klt_step_control(ctypes.Structure):
    _fields_ = [("d_drop", ctypes.c_void_p), ("d_restart", ctypes.c_void_p), ("d_restart_pts", ctypes.c_void_p),
                ("d_restart_counts", ctypes.c_void_p), ("d_restart_ids", ctypes.c_void_p), ("d_restart_next_id", ctypes.c_void_p),
                ("d_restarted", ctypes.c_void_p)]


# every symbol include/klt_b200.h declares: name -> (restype, argtypes)
_c = ctypes
_P = ctypes.c_void_p
SYMBOLS = {
    "klt_create": (_c.c_int, [_c.c_int, _c.POINTER(_P)]),
    "klt_destroy": (_c.c_int, [_P]),
    "klt_version": (_c.c_int, []),
    "klt_status_string": (_c.c_char_p, [_c.c_int]),
    "klt_device_info": (_c.c_int, [_P, _c.POINTER(_c.c_int), _c.POINTER(_c.c_int), _c.POINTER(_c.c_int), _c.c_char_p, _c.c_int]),
    "klt_host_alloc": (_c.c_int, [_c.POINTER(_P), _c.c_int64]),
    "klt_host_free": (_c.c_int, [_P]),
    "klt_pyr_plan": (_c.c_int, [_c.c_int] * 6 + [_c.POINTER(klt_pyr_layout)]),
    "klt_pyr_build": (_c.c_int, [_P, _P, _c.POINTER(klt_pyr_layout), _P, _c.c_int, _c.c_int, _P]),
    "klt_pyr_down": (_c.c_int, [_P, _P, _c.c_int, _c.c_int, _c.c_int64, _c.c_int64, _P, _c.c_int64, _c.c_int64, _c.c_int, _P]),
    "klt_lk_track": (_c.c_int, [_P, _P, _P, _P, _P, _c.POINTER(klt_pyr_layout), _c.c_int, _c.c_int, _c.c_int, _c.c_int, _P, _P, _P, _P, _P, _c.c_int,
                                _c.POINTER(klt_lk_params), _P]),
    "klt_calc_optical_flow_pyr_lk_host": (_c.c_int, [_P, _P, _c.c_int64, _P, _c.c_int64, _c.c_int, _c.c_int, _P, _P, _P, _P,
                                                     _c.c_int, _c.c_int, _c.POINTER(klt_lk_params), _c.POINTER(_c.c_int)]),
    "klt_track_filter": (_c.c_int, [_P, _P, _P, _P, _c.c_int64, _c.c_float, _c.c_int, _c.c_int, _P, _P, _P]),
    "klt_track_bidirectional_host": (_c.c_int, [_P, _P, _c.c_int64, _P, _c.c_int64, _c.c_int, _c.c_int, _P, _c.c_int, _c.c_int,
                                                _c.POINTER(klt_lk_params), _c.c_float, _P, _P, _P, _P, _P]),
    "klt_track_fb_host": (_c.c_int, [_P, _P, _c.c_int64, _P, _c.c_int64, _c.c_int, _c.c_int, _P, _c.c_int, _c.c_int,
                                     _c.POINTER(klt_lk_params), _c.c_float, _P, _P, _P, _P, _P]),
    "klt_build_optical_flow_pyramid_host": (_c.c_int, [_P, _P, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                                       _P, _c.POINTER(_c.c_int64), _c.POINTER(_c.c_int)]),
    "klt_corner_ws_bytes": (_c.c_int64, [_c.c_int, _c.c_int, _c.c_int]),
    "klt_corner_min_eigen_val": (_c.c_int, [_P, _P, _c.c_int, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int, _c.c_int, _P, _c.c_int64,
                                            _c.c_int64, _P, _c.c_int64, _c.c_int64, _P, _P, _c.c_int64, _P]),
    "klt_corner_candidates": (_c.c_int, [_P, _P, _c.c_int64, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _P, _c.c_int64, _c.c_int64,
                                         _P, _c.c_double, _P, _c.c_int64, _c.c_int, _P, _P]),
    "klt_select_corners_host": (_c.c_int, [_P, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_double, _P, _c.c_int,
                                           _c.POINTER(_c.c_int)]),
    "klt_corner_min_eigen_val_host": (_c.c_int, [_P, _P, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _P]),
    "klt_good_features_to_track_host": (_c.c_int, [_P, _P, _c.c_int64, _c.c_int, _c.c_int, _P, _c.c_int64, _c.c_int, _c.c_double,
                                                   _c.c_double, _c.c_int, _P, _c.c_int, _c.POINTER(_c.c_int)]),
    "klt_good_features_to_track_points_host": (_c.c_int, [_P, _P, _c.c_int64, _c.c_int, _c.c_int, _P, _c.c_int, _c.c_int, _c.c_int,
                                                          _c.c_double, _c.c_double, _c.c_int, _P, _c.c_int, _c.POINTER(_c.c_int)]),
    "klt_corner_mask_from_points": (_c.c_int, [_P, _P, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _P, _c.c_int64, _P]),
    "klt_frame_step_ws_bytes": (_c.c_int64, [_c.c_int, _c.c_int, _c.c_int, _c.c_int]),
    "klt_frame_step_batch": (_c.c_int, [_P, _P, _P, _P, _P, _c.POINTER(klt_pyr_layout), _c.c_int, _c.c_int, _c.c_int, _c.c_int, _P, _P,
                                        _c.c_int, _c.POINTER(klt_lk_params), _c.c_float, _c.c_int, _c.c_int, _c.c_double, _c.c_double,
                                        _c.c_int, _P, _c.c_int64, _P, _P, _P, _P, _P, _c.c_int64, _P]),
    "klt_frame_step_batch_async": (_c.c_int, [_P, _P, _P, _P, _P, _c.POINTER(klt_pyr_layout), _c.c_int, _c.c_int, _c.c_int, _c.c_int, _P,
                                              _P, _c.c_int, _c.POINTER(klt_lk_params), _c.c_float, _c.c_int, _c.c_int, _c.c_double,
                                              _c.c_double, _c.c_int, _P, _c.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _c.c_int64, _P]),
    "klt_track_records_step": (_c.c_int, [_P, _c.c_int, _c.c_int, _c.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _c.c_int, _P, _P, _P, _P,
                                          _P, _P]),
    "klt_frame_step_batch_control_async": (_c.c_int, [_P, _P, _P, _P, _P, _c.POINTER(klt_pyr_layout), _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                                      _P, _P, _c.c_int, _c.POINTER(klt_lk_params), _c.c_float, _c.c_int, _c.c_int,
                                                      _c.c_double, _c.c_double, _c.c_int, _P, _c.c_int64, _P, _P, _P, _P, _P, _P, _P, _P,
                                                      _c.c_int64, _c.POINTER(klt_step_control), _P]),
    "klt_track_records_step_control": (_c.c_int, [_P, _c.c_int, _c.c_int, _c.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _c.c_int, _P, _P, _P,
                                                  _P, _P, _P, _P, _P, _P, _P]),
    "klt_frame_step_batch_init_async": (_c.c_int, [_P, _P, _P, _P, _P, _c.POINTER(klt_pyr_layout), _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                                   _P, _P, _c.c_int, _c.POINTER(klt_lk_params), _c.c_float, _c.c_int, _c.c_int,
                                                   _c.c_double, _c.c_double, _c.c_int, _P, _c.c_int64, _P, _P, _P, _P, _P, _P, _P, _P,
                                                   _c.c_int64, _P, _c.POINTER(klt_step_control), _P]),
    "klt_frame_step_batch_fb_async": (_c.c_int, [_P, _P, _P, _P, _P, _c.POINTER(klt_pyr_layout), _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                                 _P, _P, _c.c_int, _c.POINTER(klt_lk_params), _c.c_float, _c.c_int, _c.c_int,
                                                 _c.c_double, _c.c_double, _c.c_int, _P, _c.c_int64, _P, _P, _P, _P, _P, _P, _P, _P,
                                                 _c.c_int64, _P, _c.POINTER(klt_step_control), _P, _P]),
    "klt_frame_step_batch_thin_async": (_c.c_int, [_P, _P, _P, _P, _P, _c.POINTER(klt_pyr_layout), _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                                   _P, _P, _c.c_int, _c.POINTER(klt_lk_params), _c.c_float, _c.c_int, _c.c_int,
                                                   _c.c_double, _c.c_double, _c.c_int, _P, _c.c_int64, _P, _P, _P, _P, _P, _P, _P, _P,
                                                   _c.c_int64, _P, _c.POINTER(klt_step_control), _P, _c.c_int, _c.c_double, _P, _P]),
    "klt_frame_step_grid_ws_bytes": (_c.c_int64, [_c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_int]),
    "klt_frame_step_batch_grid_async": (_c.c_int, [_P, _P, _P, _P, _P, _c.POINTER(klt_pyr_layout), _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                                   _P, _P, _c.c_int, _c.POINTER(klt_lk_params), _c.c_float, _c.c_int, _c.c_int,
                                                   _c.c_double, _c.c_double, _c.c_int, _P, _c.c_int64, _P, _P, _P, _P, _P, _P, _P, _P,
                                                   _c.c_int64, _P, _c.POINTER(klt_step_control), _P, _c.c_int, _c.c_double, _P,
                                                   _c.c_int, _c.c_int, _c.c_int, _P]),
    "klt_good_features_to_track_grid_ws_bytes": (_c.c_int64, [_c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_int]),
    "klt_good_features_to_track_grid": (_c.c_int, [_P, _P, _c.c_int, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int, _c.c_int, _c.c_int,
                                                   _c.c_int, _c.c_double, _c.c_double, _c.c_int, _P, _c.c_int64, _c.c_int64, _P, _P, _P,
                                                   _c.c_int64, _P]),
    "klt_track_predict": (_c.c_int, [_P, _c.c_int, _c.c_int, _P, _P, _P, _P, _c.c_int, _P, _P, _P, _P, _P, _P]),
    "klt_track_window": (_c.c_int, [_P, _c.c_int, _c.c_int64, _c.c_int, _P, _P, _P, _P, _c.c_int, _P, _P]),
    "klt_bilateral_filter": (_c.c_int, [_P, _P, _c.c_int, _c.c_int, _c.c_int64, _c.c_int64, _P, _c.c_int64, _c.c_int64, _c.c_int,
                                        _c.c_int, _c.c_double, _c.c_double, _P]),
    "klt_bilateral_filter_host": (_c.c_int, [_P, _P, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_double, _c.c_double, _P,
                                             _c.c_int64]),
    "klt_corner_sub_pix": (_c.c_int, [_P, _P, _c.c_int, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int, _P, _c.c_int64, _P, _P, _c.c_int,
                                      _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_double, _P]),
    "klt_corner_sub_pix_host": (_c.c_int, [_P, _P, _c.c_int64, _c.c_int, _c.c_int, _P, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                           _c.c_int, _c.c_int, _c.c_double]),
    "klt_clahe_ws_bytes": (_c.c_int64, [_c.c_int, _c.c_int, _c.c_int]),
    "klt_clahe": (_c.c_int, [_P, _P, _c.c_int, _c.c_int, _c.c_int64, _c.c_int64, _P, _c.c_int64, _c.c_int64, _c.c_int, _c.c_double,
                             _c.c_int, _c.c_int, _P, _c.c_int64, _P]),
    "klt_clahe_host": (_c.c_int, [_P, _P, _c.c_int64, _c.c_int, _c.c_int, _c.c_double, _c.c_int, _c.c_int, _P, _c.c_int64]),
}

_lib = None
_lock = threading.Lock()


class KLTLibraryError(RuntimeError):
    """The native library is missing / unloadable, or a CUDA call failed.  Never silently ignored."""


def load():
    """Load libklt_b200.so and bind every declared symbol.  Raises if it has not been built."""
    global _lib
    if _lib is not None:      # fast path, no lock: the reference is assigned once
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise KLTLibraryError(
                    "libklt_b200.so not found at %s -- build it with `python __graft_entry__.py build` "
                    "(nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
            L = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SYMBOLS.items():
                fn = getattr(L, name)
                fn.restype = res
                fn.argtypes = args
            _lib = L
    return _lib


def status_string(code):
    return load().klt_status_string(int(code)).decode()


class Context:
    """Owns a klt_ctx (device, stream, workspaces).  One per device per process is plenty."""

    def __init__(self, device=0):
        L = load()
        h = _P()
        rc = L.klt_create(int(device), ctypes.byref(h))
        if rc != KLT_OK:
            raise KLTLibraryError("klt_create(device=%d) failed: %s" % (device, status_string(rc)))
        self._h = h
        self.device = int(device)
        sm, major, minor = _c.c_int(), _c.c_int(), _c.c_int()
        name = ctypes.create_string_buffer(128)
        L.klt_device_info(h, ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor), name, 128)
        self.sm_count, self.cc, self.name = sm.value, (major.value, minor.value), name.value.decode()

    @property
    def handle(self):
        if self._h is None:
            raise KLTLibraryError("context already destroyed")
        return self._h

    def close(self):
        if getattr(self, "_h", None) is not None and _lib is not None:
            _lib.klt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_contexts = {}


def default_context(device=0):
    ctx = _contexts.get(device)      # fast path, no lock: entries are only ever added
    if ctx is not None:
        return ctx
    with _lock:
        ctx = _contexts.get(device)
    if ctx is None:
        ctx = Context(device)
        with _lock:
            _contexts.setdefault(device, ctx)
            ctx = _contexts[device]
    return ctx
