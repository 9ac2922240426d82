"""Drop-in replacements for the OpenCV calls on the reference's tracking hot path.

``calcOpticalFlowPyrLK`` has the signature and return contract of ``cv2.calcOpticalFlowPyrLK`` as
the reference calls it (src/extractor/extractor.py:44,45,65,66; parameters :16-19):

    nextPts, status, err = calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, None,
                                                winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))

numpy in -> numpy out (host buffers, synchronous, fresh output arrays), results bit-identical to
cv2 4.13 (SURVEY.md Appendix A).  All arithmetic runs in hand-written sm_100a kernels behind the
C ABI of include/klt_b200.h; there is no CPU fallback -- without the library or a B200 the call
raises.  torch CUDA tensors are accepted as well and then stay on the device (see tracker.py).
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import (KLT_ERR_INVALID_ARG, KLT_ERR_UNSUPPORTED, KLT_OK, OPTFLOW_LK_GET_MIN_EIGENVALS,
                   OPTFLOW_USE_INITIAL_FLOW, TERM_COUNT, TERM_EPS, klt_lk_params)

try:  # raise the same exception class the reference's callers would see from OpenCV
    import cv2 as _cv2
    _ErrorBase = _cv2.error
except Exception:  # pragma: no cover - cv2 is present in the target image
    _ErrorBase = ValueError


class error(_ErrorBase):
    """Invalid arguments (OpenCV error -215 equivalent).  Subclass of cv2.error when cv2 exists."""


def _fail(msg):
    raise error("klt_b200: (-215:Assertion failed) " + msg)


def _raise_status(rc, what):
    if rc == KLT_ERR_INVALID_ARG:
        _fail("%s: invalid argument" % what)
    if rc == KLT_ERR_UNSUPPORTED:
        raise error("klt_b200: %s: %s" % (what, _lib.status_string(rc)))
    raise _lib.KLTLibraryError("%s failed: %s" % (what, _lib.status_string(rc)))


def _check_win_level(winSize, maxLevel):
    try:
        win_w, win_h = int(winSize[0]), int(winSize[1])
    except Exception:
        _fail("winSize must be a (width, height) pair")
    maxLevel = int(maxLevel)
    if not (maxLevel >= 0 and win_w > 2 and win_h > 2):
        _fail("maxLevel >= 0 && winSize.width > 2 && winSize.height > 2 in function 'calc'")
    return win_w, win_h, maxLevel


SECOND_PASSES = ("reference", "reverse")


def check_second_pass(second_pass):
    """The second LK pass of a tracking step: "reference", the reference's same-direction call started from the forward
    result, or "reverse", the forward-backward check that tracks the result from the new frame back into the old one."""
    if not (isinstance(second_pass, str) and second_pass in SECOND_PASSES):
        raise error("klt_b200: second_pass must be 'reference' or 'reverse', not %r" % (second_pass,))
    return second_pass


def make_params(winSize=(21, 21), criteria=(TERM_COUNT | TERM_EPS, 30, 0.01), flags=0, minEigThreshold=1e-4):
    win_w, win_h = int(winSize[0]), int(winSize[1])
    try:
        ctype, ccount, ceps = int(criteria[0]), int(criteria[1]), float(criteria[2])
    except Exception:
        _fail("criteria must be (type, maxCount, epsilon)")
    return klt_lk_params(win_w, win_h, ctype, ccount, ceps, int(flags), float(minEigThreshold))


_PARAMS_CACHE = {}


def _cached_params(win_w, win_h, criteria, flags, minEigThreshold):
    """make_params with the struct cached per parameter set (the reference calls with the same parameters for every frame;
    building a ctypes structure costs more than a microsecond).  The structs are only ever read."""
    try:
        key = (win_w, win_h, criteria[0], criteria[1], criteria[2], flags, minEigThreshold)
        prm = _PARAMS_CACHE.get(key)
    except Exception:
        key, prm = None, None
    if prm is None:
        prm = make_params((win_w, win_h), criteria, flags, minEigThreshold)
        if key is not None and len(_PARAMS_CACHE) < 256:
            _PARAMS_CACHE[key] = prm
    return prm


_CHAR0 = ctypes.c_char * 0


def _addr(arr):
    """Address of a numpy array's first element.  arr.ctypes.data builds a helper object on every access (2 us; six of them
    were most of the wrapper's cost); going through the buffer protocol takes a third of that.  Read-only or
    non-contiguous arrays do not export a writable simple buffer: they take the slow way."""
    try:
        return ctypes.addressof(_CHAR0.from_buffer(arr))
    except (TypeError, ValueError, BufferError):
        return arr.ctypes.data


def _host_image(img, name):
    if not isinstance(img, np.ndarray):
        _fail("%s is not a numpy array, neither a scalar" % name)
    if img.ndim == 3 and img.shape[2] == 1:
        img = img[:, :, 0]
    if img.dtype != np.uint8:
        _fail("%s.depth() == CV_8U in function 'buildOpticalFlowPyramid'" % name)
    if img.ndim != 2:
        raise error("klt_b200: %s: only single-channel images are supported (the reference tracks on "
                    "grayscale frames, src/loader/loader.py:86)" % name)
    if img.size == 0:
        _fail("%s is empty" % name)
    if img.strides[1] != 1 or img.strides[0] < img.shape[1]:
        img = np.ascontiguousarray(img)
    return img


def _host_points(pts, name):
    if not isinstance(pts, np.ndarray):
        _fail("%s is not a numpy array, neither a scalar" % name)
    ok = pts.dtype == np.float32 and (
        (pts.ndim == 2 and pts.shape[1] == 2) or
        (pts.ndim == 3 and pts.shape[2] == 2 and (pts.shape[1] == 1 or pts.shape[0] == 1)))
    if pts.dtype == np.float32 and pts.size == 0 and pts.ndim in (1, 2, 3):
        return np.empty((0, 2), np.float32), pts.shape
    if not ok:
        _fail("(npoints = %s.checkVector(2, CV_32F, true)) >= 0 in function 'calc'" % name)
    return np.ascontiguousarray(pts.reshape(-1, 2)), pts.shape


def _is_torch_cuda(x):
    return type(x).__module__.startswith("torch") and hasattr(x, "is_cuda") and x.is_cuda


def calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, nextPts=None, status=None, err=None, winSize=(21, 21),
                         maxLevel=3, criteria=(TERM_COUNT | TERM_EPS, 30, 0.01), flags=0, minEigThreshold=1e-4,
                         device=0):
    """cv2.calcOpticalFlowPyrLK on a B200.  -> (nextPts, status, err)

    ``status`` / ``err`` arguments are accepted for signature compatibility and ignored (cv2's Python
    binding allocates fresh outputs as well).  ``nextPts`` is read only with OPTFLOW_USE_INITIAL_FLOW.
    """
    if _is_torch_cuda(prevImg):
        from .tracker import calc_optical_flow_pyr_lk_device
        return calc_optical_flow_pyr_lk_device(prevImg, nextImg, prevPts, nextPts, winSize=winSize, maxLevel=maxLevel,
                                               criteria=criteria, flags=flags, minEigThreshold=minEigThreshold)
    win_w, win_h, maxLevel = _check_win_level(winSize, maxLevel)
    prev = _host_image(prevImg, "prevImg")
    nxt = _host_image(nextImg, "nextImg")
    if prev.shape != nxt.shape:
        _fail("prevPyr[level * lvlStep1].size() == nextPyr[level * lvlStep2].size() in function 'calc'")
    pts, shape = _host_points(prevPts, "prevPts")
    n = pts.shape[0]
    if n == 0:
        return None, None, None
    params = _cached_params(win_w, win_h, criteria, flags, minEigThreshold)
    out = np.empty((n, 2), np.float32)
    if int(flags) & OPTFLOW_USE_INITIAL_FLOW:
        if nextPts is None:
            _fail("OPTFLOW_USE_INITIAL_FLOW requires nextPts")
        init, _ = _host_points(np.asarray(nextPts), "nextPts")
        if init.shape[0] != n:
            _fail("nextPts.checkVector(2, CV_32F, true) == npoints in function 'calc'")
        out[:] = init
    st = np.empty((n, 1), np.uint8)
    er = np.empty((n, 1), np.float32)
    h, w = prev.shape
    ctx = _lib.default_context(device)
    rc = _lib.load().klt_calc_optical_flow_pyr_lk_host(
        ctx.handle, _addr(prev), prev.strides[0], _addr(nxt), nxt.strides[0], w, h,
        _addr(pts), _addr(out), _addr(st), _addr(er), n, maxLevel, ctypes.byref(params), None)
    if rc != KLT_OK:
        _raise_status(rc, "calcOpticalFlowPyrLK")
    return out.reshape(shape), st, er


def trackBidirectional(prevImg, nextImg, prevPts, max_bidir_error=30, winSize=(31, 31), maxLevel=3,
                       criteria=(TERM_COUNT | TERM_EPS, 30, 0.03), minEigThreshold=1e-4, device=0, second_pass="reference"):
    """The KLT part of the reference's ``extend_tracks`` / ``extend_landmarks`` in one call
    (src/extractor/extractor.py:43-53 and :64-75; defaults = its ``_lk_params``, :16-19):

        p1, st, err = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **lk)
        p0r, _, _   = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **lk)     # same direction, as in the reference
        d    = abs(p0 - p0r).reshape(-1, 2).max(-1)
        keep = (d < max_bidir_error) & (0 <= x <= W) & (0 <= y <= H)          # (x, y) = p1

    -> (p1 like prevPts, keep (N,) bool, d (N,) float32, status (N,1) uint8, err (N,1) float32).
    One upload and one pyramid build per image (cv2 builds four pyramids for the two calls), both LK passes and the
    filter on the device; p1 / status / err are bit-identical to cv2's first call.  N == 0 -> (None,) * 5.

    second_pass="reverse" runs the forward-backward check instead of the reference's second call:
    p0r = cv2.calcOpticalFlowPyrLK(im1, im0, p1, None, **lk), from the new image back into the old one.  d is then the
    tracking error of a correct track (not about twice the frame's motion), and a useful max_bidir_error is about 1 px.
    """
    check_second_pass(second_pass)
    win_w, win_h, maxLevel = _check_win_level(winSize, maxLevel)
    prev = _host_image(prevImg, "prevImg")
    nxt = _host_image(nextImg, "nextImg")
    if prev.shape != nxt.shape:
        _fail("prevPyr[level * lvlStep1].size() == nextPyr[level * lvlStep2].size() in function 'calc'")
    pts, shape = _host_points(prevPts, "prevPts")
    n = pts.shape[0]
    if n == 0:
        return None, None, None, None, None
    params = make_params((win_w, win_h), criteria, 0, minEigThreshold)
    out = np.empty((n, 2), np.float32)
    st = np.empty((n, 1), np.uint8)
    er = np.empty((n, 1), np.float32)
    keep = np.empty(n, np.uint8)
    bd = np.empty(n, np.float32)
    h, w = prev.shape
    ctx = _lib.default_context(device)
    entry = _lib.load().klt_track_fb_host if second_pass == "reverse" else _lib.load().klt_track_bidirectional_host
    rc = entry(
        ctx.handle, _addr(prev), prev.strides[0], _addr(nxt), nxt.strides[0], w, h, _addr(pts), n,
        maxLevel, ctypes.byref(params), float(max_bidir_error),
        _addr(out), _addr(st), _addr(er), _addr(keep), _addr(bd))
    if rc != KLT_OK:
        _raise_status(rc, "trackBidirectional")
    return out.reshape(shape), keep.view(np.bool_), bd, st, er


def buildOpticalFlowPyramid(img, winSize, maxLevel, pyramid=None, withDerivatives=False, pyrBorder=None,
                            derivBorder=None, tryReuseInputImage=True, device=0):
    """cv2.buildOpticalFlowPyramid(img, winSize, maxLevel, withDerivatives=False) -> (retval, pyramid).

    Returns the un-bordered u8 levels (what cv2's list elements show as their .shape views).  The
    LK kernel computes Scharr derivatives on the fly, so ``withDerivatives=True`` is not offered.
    """
    if withDerivatives:
        raise error("klt_b200: withDerivatives=True is not supported (derivatives are fused into the LK kernel)")
    win_w, win_h, maxLevel = _check_win_level(winSize, maxLevel)
    im = _host_image(img, "img")
    h, w = im.shape
    ctx = _lib.default_context(device)
    L = _lib.load()
    offs = (ctypes.c_int64 * (_lib.KLT_MAX_LEVELS + 1))()
    top = ctypes.c_int()
    rc = L.klt_build_optical_flow_pyramid_host(ctx.handle, None, 0, w, h, win_w, win_h, maxLevel, None, offs,
                                               ctypes.byref(top))
    if rc != KLT_OK:
        _raise_status(rc, "buildOpticalFlowPyramid")
    buf = np.empty(offs[top.value + 1], np.uint8)
    rc = L.klt_build_optical_flow_pyramid_host(ctx.handle, _addr(im), im.strides[0], w, h, win_w, win_h,
                                               maxLevel, _addr(buf), offs, ctypes.byref(top))
    if rc != KLT_OK:
        _raise_status(rc, "buildOpticalFlowPyramid")
    levels, lw, lh = [], w, h
    for l in range(top.value + 1):
        levels.append(buf[offs[l]:offs[l + 1]].reshape(lh, lw))
        lw, lh = (lw + 1) // 2, (lh + 1) // 2
    return top.value, levels


class _PinnedBuffer:
    """Page-locked host allocation exposed through the array interface (freed with the last view)."""

    def __init__(self, nbytes):
        self._L = _lib.load()
        p = ctypes.c_void_p()
        rc = self._L.klt_host_alloc(ctypes.byref(p), max(int(nbytes), 1))
        if rc != KLT_OK:
            raise _lib.KLTLibraryError("klt_host_alloc failed: " + _lib.status_string(rc))
        self._ptr = p
        self.__array_interface__ = {"data": (p.value, False), "shape": (int(nbytes),), "typestr": "|u1", "version": 3}

    def __del__(self):
        try:
            self._L.klt_host_free(self._ptr)
        except Exception:
            pass


def pinned_empty(shape, dtype=np.uint8):
    """numpy array in page-locked host memory (DMA-able without a staging copy)."""
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    return np.asarray(_PinnedBuffer(nbytes)).view(dtype).reshape(shape)
