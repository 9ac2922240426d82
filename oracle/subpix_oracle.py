"""ctypes front-end of oracle/subpix_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Restates cv2.cornerSubPix and the cv2.getRectSubPix it calls, OpenCV's own code path (S.1-S.6 in subpix_oracle.c),
pinned bit-exactly against the live cv2 module with cv2.ipp.setUseIPP(False) in tests/test_subpix_cpu.py.  Compiled with
gcc on first use, with the flags of oracle/Makefile (one rounding per float operation), into its own library next to
libklt_oracle.so, or into a temporary directory when the tree is read-only.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "subpix_oracle.c")
_CFLAGS = ["-O2", "-fPIC", "-std=c11", "-Wall", "-Wextra", "-ffp-contract=off", "-fno-fast-math", "-fno-unsafe-math-optimizations"]
_lib = None


def _compile(out_dir):
    so = os.path.join(out_dir, "libsubpix_oracle.so")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(_SRC):
        os.makedirs(out_dir, exist_ok=True)
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call([os.environ.get("CC", "gcc")] + _CFLAGS + ["-shared", "-o", tmp, _SRC, "-lm"])
        os.replace(tmp, so)
    return so


def build():
    """Compile subpix_oracle.c (a second) -> path of the shared library."""
    try:
        return _compile(os.path.join(_HERE, "_build"))
    except OSError:
        return _compile(os.path.join(tempfile.gettempdir(), "klt_subpix_oracle_%d" % os.getuid()))


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        c = ctypes
        L.klt_oracle_subpix_mask.argtypes = [c.c_int, c.c_int, c.c_int, c.c_int, c.c_void_p]
        L.klt_oracle_subpix_mask.restype = None
        L.klt_oracle_corner_sub_pix.argtypes = [c.c_void_p, c.c_int, c.c_int, c.c_int64, c.c_void_p, c.c_int, c.c_int, c.c_int,
                                                c.c_int, c.c_int, c.c_int, c.c_int, c.c_double, c.c_void_p]
        L.klt_oracle_corner_sub_pix.restype = c.c_int
        L.klt_oracle_rect_sub_pix.argtypes = [c.c_void_p, c.c_int, c.c_int, c.c_int64, c.c_int, c.c_int, c.c_float, c.c_float, c.c_void_p]
        L.klt_oracle_rect_sub_pix.restype = c.c_int
        _lib = L
    return _lib


def _u8_image(img):
    img = np.asarray(img)
    if img.dtype != np.uint8 or img.ndim != 2:
        raise ValueError("oracle: image must be 2-D uint8")
    if img.strides[1] != 1:
        img = np.ascontiguousarray(img)
    return img


def subpix_mask(win_size, zero_zone=(-1, -1)):
    """The float32 weight mask of cv2.cornerSubPix (S.2) -> (2wy + 1, 2wx + 1)."""
    wx, wy = int(win_size[0]), int(win_size[1])
    out = np.empty((2 * wy + 1, 2 * wx + 1), np.float32)
    lib().klt_oracle_subpix_mask(wx, wy, int(zero_zone[0]), int(zero_zone[1]), out.ctypes.data)
    return out


def rect_sub_pix(img, patch_size, center):
    """cv2.getRectSubPix(img, patchSize, center, patchType=cv2.CV_32F) on a uint8 (h, w) image, OpenCV's own code path
    (S.5 / S.6) -> float32 (ph, pw)."""
    img = _u8_image(img)
    h, w = img.shape
    pw, ph = int(patch_size[0]), int(patch_size[1])
    out = np.empty((ph, pw), np.float32)
    rc = lib().klt_oracle_rect_sub_pix(img.ctypes.data, w, h, img.strides[0], pw, ph, float(center[0]), float(center[1]), out.ctypes.data)
    if rc < 0:
        raise ValueError("oracle: rect_sub_pix failed (%d)" % rc)
    return out


def corner_sub_pix(img, corners, win_size, zero_zone, criteria, return_iters=False):
    """cv2.cornerSubPix(img, corners, winSize, zeroZone, criteria) on a uint8 (h, w) image, OpenCV's own code path
    (S.1-S.6) -> a refined float32 copy of `corners` [, iterations per point (n,) int32].  Raises ValueError where cv2
    asserts."""
    img = _u8_image(img)
    h, w = img.shape
    c = np.asarray(corners)
    if c.dtype != np.float32 or c.size % 2:
        raise ValueError("oracle: corners must be float32 Nx2")
    out = np.ascontiguousarray(c.reshape(-1, 2)).copy()
    iters = np.zeros(len(out), np.int32)
    rc = lib().klt_oracle_corner_sub_pix(img.ctypes.data, w, h, img.strides[0], out.ctypes.data if len(out) else None, len(out),
                                         int(win_size[0]), int(win_size[1]), int(zero_zone[0]), int(zero_zone[1]),
                                         int(criteria[0]), int(criteria[1]), float(criteria[2]), iters.ctypes.data)
    if rc < 0:
        raise ValueError("oracle: corner_sub_pix failed (%d)" % rc)
    out = out.reshape(c.shape)
    return (out, iters) if return_iters else out
