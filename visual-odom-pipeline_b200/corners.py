"""Drop-in replacements for the OpenCV calls of the reference's feature-detection step (SURVEY.md s8f rank 2).

``goodFeaturesToTrack`` has the signature and return contract of ``cv2.goodFeaturesToTrack`` as the reference calls
it (src/extractor/extractor.py:110-111 with the parameters of :21-24; once per frame, src/pipeline/pipeline.py:159-163):

    kp = goodFeaturesToTrack(img, mask=mask, maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)

numpy in -> float32 (N, 1, 2) out (``None`` when nothing is found, like cv2), strongest corner first, results
bit-identical to the cv2 wheel (oracle/gftt_oracle.c G.1-G.8).  The eigenvalue map, threshold, dilation and
local-maximum test run in sm_100a kernels (csrc/klt_corners.cu); the sort of the surviving candidates and the greedy
minimum-distance selection are sequential and run on the host inside the C ABI.  No CPU fallback.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import KLT_OK
from .lk import _addr, _fail, _raise_status, error


def _u8_image(img, name, func):
    if not isinstance(img, np.ndarray):
        _fail("%s is not a numpy array, neither a scalar" % name)
    if img.ndim == 3 and img.shape[2] == 1:
        img = img[:, :, 0]
    if img.ndim != 2 or img.dtype != np.uint8:
        if img.ndim == 2 and img.dtype == np.float32:
            raise error("klt_b200: %s: float32 images are not supported (the reference detects on uint8 grayscale "
                        "frames, src/loader/loader.py:86)" % func)
        _fail("%s: 8-bit single-channel image expected in function '%s'" % (name, func))
    if img.size == 0:
        _fail("%s is empty" % name)
    if img.strides[1] != 1 or img.strides[0] < img.shape[1]:
        img = np.ascontiguousarray(img)
    return img


def cornerMinEigenVal(src, blockSize, dst=None, ksize=3, borderType=4, device=0):
    """cv2.cornerMinEigenVal(src, blockSize[, dst[, ksize[, borderType]]]) -> float32 (h, w), on a B200."""
    if int(ksize) != 3 or int(borderType) != 4:
        raise error("klt_b200: cornerMinEigenVal: only ksize=3 and BORDER_REFLECT_101 (the defaults goodFeaturesToTrack uses)")
    img = _u8_image(src, "src", "cornerMinEigenVal")
    h, w = img.shape
    blockSize = int(blockSize)
    if blockSize < 1:
        _fail("blockSize > 0 in function 'cornerMinEigenVal'")
    out = np.empty((h, w), np.float32)
    ctx = _lib.default_context(device)
    rc = _lib.load().klt_corner_min_eigen_val_host(ctx.handle, _addr(img), img.strides[0], w, h, blockSize, _addr(out))
    if rc != KLT_OK:
        _raise_status(rc, "cornerMinEigenVal")
    return out


def goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance, corners=None, mask=None, blockSize=3,
                        useHarrisDetector=False, k=0.04, gradientSize=3, device=0):
    """cv2.goodFeaturesToTrack on a B200 -> float32 (N, 1, 2) or None.

    ``corners`` is accepted for signature compatibility and ignored (cv2's binding allocates a fresh output too).
    """
    if useHarrisDetector:
        raise error("klt_b200: goodFeaturesToTrack: the Harris response is not implemented (the reference uses the "
                    "default minimum-eigenvalue response, src/extractor/extractor.py:21-24)")
    if int(gradientSize) != 3:
        raise error("klt_b200: goodFeaturesToTrack: only gradientSize=3")
    img = _u8_image(image, "image", "goodFeaturesToTrack")
    h, w = img.shape
    maxCorners, blockSize = int(maxCorners), int(blockSize)
    qualityLevel, minDistance = float(qualityLevel), float(minDistance)
    if not (qualityLevel > 0 and minDistance >= 0 and maxCorners >= 0):
        _fail("qualityLevel > 0 && minDistance >= 0 && maxCorners >= 0 in function 'goodFeaturesToTrack'")
    if blockSize < 1:
        _fail("blockSize > 0 in function 'goodFeaturesToTrack'")
    mptr, mpitch = None, 0
    if mask is not None:
        if not isinstance(mask, np.ndarray):
            _fail("mask is not a numpy array, neither a scalar")
        if mask.ndim == 3 and mask.shape[2] == 1:
            mask = mask[:, :, 0]
        if mask.dtype != np.uint8 or mask.shape != img.shape:
            _fail("_mask.empty() || (_mask.type() == CV_8UC1 && _mask.sameSize(_image)) in function 'goodFeaturesToTrack'")
        if mask.strides[1] != 1 or mask.strides[0] < w:
            mask = np.ascontiguousarray(mask)
        mptr, mpitch = _addr(mask), mask.strides[0]
    cap = maxCorners if maxCorners > 0 else w * h   # candidates are distinct pixels
    out = np.empty((cap, 2), np.float32)
    n = ctypes.c_int(0)
    ctx = _lib.default_context(device)
    rc = _lib.load().klt_good_features_to_track_host(ctx.handle, _addr(img), img.strides[0], w, h, mptr, mpitch,
                                                     maxCorners, qualityLevel, minDistance, blockSize,
                                                     _addr(out), cap, ctypes.byref(n))
    if rc != KLT_OK:
        _raise_status(rc, "goodFeaturesToTrack")
    if n.value == 0:
        return None
    return out[:n.value].reshape(-1, 1, 2).copy() if n.value < cap else out.reshape(-1, 1, 2)


def detectNewFeatures(image, trackedPoints, maskRadius, maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31,
                      device=0):
    """The detection step of the reference's ``Extractor.extract(..., detector='shi-tomasi')`` fused into one call
    (src/extractor/extractor.py:102-111; opt-in, like trackBidirectional for the tracking step):

        mask = 255; for (x, y) in np.int32(tracked): cv2.circle(mask, (x, y), maskRadius, 0, -1)
        return cv2.goodFeaturesToTrack(image, mask=mask, maxCorners=..., qualityLevel=..., minDistance=..., blockSize=...)

    The mask is rasterised on the device from the tracked keypoints (float32 (N, 2) / (N, 1, 2); 8 bytes per point go up
    instead of a w x h mask, and the Python loop over cv2.circle disappears).  Same corners, same order as the two cv2
    calls.  Defaults are the reference's parameters (extractor.py:21-24)."""
    img = _u8_image(image, "image", "goodFeaturesToTrack")
    h, w = img.shape
    maxCorners, blockSize, maskRadius = int(maxCorners), int(blockSize), int(maskRadius)
    qualityLevel, minDistance = float(qualityLevel), float(minDistance)
    if not (qualityLevel > 0 and minDistance >= 0 and maxCorners >= 0):
        _fail("qualityLevel > 0 && minDistance >= 0 && maxCorners >= 0 in function 'goodFeaturesToTrack'")
    if blockSize < 1 or maskRadius < 0:
        _fail("blockSize > 0 && radius >= 0")
    pts = np.zeros((0, 2), np.float32) if trackedPoints is None else np.ascontiguousarray(np.asarray(trackedPoints, np.float32).reshape(-1, 2))
    cap = maxCorners if maxCorners > 0 else w * h
    out = np.empty((cap, 2), np.float32)
    n = ctypes.c_int(0)
    ctx = _lib.default_context(device)
    rc = _lib.load().klt_good_features_to_track_points_host(ctx.handle, _addr(img), img.strides[0], w, h,
                                                            _addr(pts) if len(pts) else None, len(pts), maskRadius,
                                                            maxCorners, qualityLevel, minDistance, blockSize,
                                                            _addr(out), cap, ctypes.byref(n))
    if rc != KLT_OK:
        _raise_status(rc, "detectNewFeatures")
    if n.value == 0:
        return None
    return out[:n.value].reshape(-1, 1, 2).copy() if n.value < cap else out.reshape(-1, 1, 2)


def check_subpix(winSize, zeroZone, criteria, w, h, func="cornerSubPix"):
    """The window, zero zone and criteria of cv2.cornerSubPix checked against a w x h image as cv2 asserts them (plus the
    window cap of include/klt_b200.h) -> (win_w, win_h, zero_w, zero_h, crit_type, max_count, eps)."""
    try:
        win_w, win_h = (int(v) for v in winSize)
        zero_w, zero_h = (int(v) for v in zeroZone)
        crit_type, max_count, eps = int(criteria[0]), int(criteria[1]), float(criteria[2])
    except (TypeError, ValueError, IndexError):
        raise error("klt_b200: %s: winSize and zeroZone must be pairs of ints, criteria (type, maxCount, epsilon)" % func)
    if not (win_w > 0 and win_h > 0):
        _fail("win.width > 0 && win.height > 0 in function '%s'" % func)
    if not (w >= win_w * 2 + 5 and h >= win_h * 2 + 5):
        _fail("src.cols >= win.width*2 + 5 && src.rows >= win.height*2 + 5 in function '%s'" % func)
    if win_w > _lib.KLT_MAX_SUBPIX_WIN or win_h > _lib.KLT_MAX_SUBPIX_WIN:
        raise error("klt_b200: %s: winSize %r is larger than KLT_MAX_SUBPIX_WIN (%d)" % (func, (win_w, win_h), _lib.KLT_MAX_SUBPIX_WIN))
    return win_w, win_h, zero_w, zero_h, crit_type, max_count, eps


def cornerSubPix(image, corners, winSize, zeroZone, criteria, device=0):
    """cv2.cornerSubPix(image, corners, winSize, zeroZone, criteria) on a B200: refines the float32 (N, 1, 2) or (N, 2)
    array `corners` in place and returns it, bit-identical to OpenCV's own code path (oracle/subpix_oracle.c; the cv2 wheel
    with cv2.ipp.setUseIPP(False)).  Every assertion cv2 makes is checked on the host before any device work, so a point
    outside the image or NaN raises with `corners` unchanged (cv2 refines the points before it in place first)."""
    img = _u8_image(image, "image", "cornerSubPix")
    h, w = img.shape
    c = corners
    if not (isinstance(c, np.ndarray) and c.dtype == np.float32 and c.flags.c_contiguous
            and ((c.ndim == 2 and c.shape[1] == 2) or (c.ndim == 3 and c.shape[2] == 2 and 1 in (c.shape[0], c.shape[1])))):
        _fail("count >= 0 in function 'cornerSubPix'")
    n = c.size // 2
    if n == 0:
        return c
    args = check_subpix(winSize, zeroZone, criteria, w, h)
    p = c.reshape(-1, 2)
    if not bool(((p[:, 0] >= 0) & (p[:, 0] < w) & (p[:, 1] >= 0) & (p[:, 1] < h)).all()):
        _fail("Rect(0, 0, src.cols, src.rows).contains(cT) in function 'cornerSubPix'")
    ctx = _lib.default_context(device)
    rc = _lib.load().klt_corner_sub_pix_host(ctx.handle, _addr(img), img.strides[0], w, h, _addr(c), n, *args)
    if rc != KLT_OK:
        _raise_status(rc, "cornerSubPix")
    return c
