"""Device-resident, batched corner detection on torch CUDA tensors (SURVEY.md s8f rank 2).

PyTorch is used for device memory and streams only; every kernel is libklt_b200's (csrc/klt_corners.cu).  This is what
the batched configs use (BASELINE.json configs[3]: many independent sequences): one launch sequence computes the
minimum-eigenvalue maps and candidate lists of B frames, the sequential tail of goodFeaturesToTrack (greedy
minimum-distance selection, reference parameters src/extractor/extractor.py:21-24) then runs per frame on the host
through klt_select_corners_host.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import KLT_OK
from .lk import _fail, _raise_status, error
from .tracker import _as_image_batch, _batch_stride, _stream_ptr, _torch


def corner_min_eigen_val(images, blockSize, mask=None, ctx=None, return_max=False):
    """cv2.cornerMinEigenVal(img, blockSize, ksize=3) for a (B, H, W) / (H, W) uint8 CUDA tensor -> (B, H, W) float32.

    With return_max also returns the (B,) uint32 order-preserving encoding of max(eig over mask != 0) that
    klt_corner_candidates consumes."""
    torch = _torch()
    img = _as_image_batch(images)
    B, H, W = img.shape
    blockSize = int(blockSize)
    if blockSize < 1:
        _fail("blockSize > 0 in function 'cornerMinEigenVal'")
    ctx = ctx or _lib.default_context(img.device.index or 0)
    L = _lib.load()
    m_ptr, m_pitch, m_bs = None, 0, 0
    if mask is not None:
        mask = _as_image_batch(mask)
        if tuple(mask.shape) != (B, H, W):
            _fail("_mask.empty() || (_mask.type() == CV_8UC1 && _mask.sameSize(_image)) in function 'goodFeaturesToTrack'")
        m_ptr = mask.data_ptr()
        m_pitch, m_bs = mask.stride(1), _batch_stride(mask)
    eig = torch.empty((B, H, W), dtype=torch.float32, device=img.device)
    mx = torch.zeros((B,), dtype=torch.int32, device=img.device)
    ws_bytes = int(L.klt_corner_ws_bytes(W, H, B))
    ws = torch.empty((ws_bytes + 256,), dtype=torch.uint8, device=img.device)
    ws_ptr = (ws.data_ptr() + 255) // 256 * 256
    rc = L.klt_corner_min_eigen_val(ctx.handle, img.data_ptr(), W, H, img.stride(1), _batch_stride(img), B, blockSize, eig.data_ptr(), W, H * W,
                                    m_ptr, m_pitch, m_bs, mx.data_ptr(), ws_ptr, ws_bytes, _stream_ptr(img))
    if rc != KLT_OK:
        _raise_status(rc, "klt_corner_min_eigen_val")
    return (eig, mx, mask) if return_max else eig


def good_features_to_track(images, maxCorners, qualityLevel, minDistance, mask=None, blockSize=3, ctx=None):
    """cv2.goodFeaturesToTrack for every frame of a (B, H, W) uint8 CUDA tensor (mask: same shape or None).
    -> list of B float32 (N_b, 1, 2) numpy arrays (None where cv2 would return None), bit-identical to cv2 per frame."""
    torch = _torch()
    maxCorners, qualityLevel, minDistance = int(maxCorners), float(qualityLevel), float(minDistance)
    if not (qualityLevel > 0 and minDistance >= 0 and maxCorners >= 0):
        _fail("qualityLevel > 0 && minDistance >= 0 && maxCorners >= 0 in function 'goodFeaturesToTrack'")
    eig, mx, mask = corner_min_eigen_val(images, blockSize, mask=mask, ctx=ctx, return_max=True)
    B, H, W = eig.shape
    ctx = ctx or _lib.default_context(eig.device.index or 0)
    L = _lib.load()
    cap = H * W
    keys = torch.empty((B, cap), dtype=torch.int64, device=eig.device)
    count = torch.zeros((B,), dtype=torch.int32, device=eig.device)
    m_ptr, m_pitch, m_bs = (None, 0, 0) if mask is None else (mask.data_ptr(), mask.stride(1), _batch_stride(mask))
    rc = L.klt_corner_candidates(ctx.handle, eig.data_ptr(), W, H * W, W, H, B, m_ptr, m_pitch, m_bs, mx.data_ptr(), qualityLevel,
                                 keys.data_ptr(), cap, cap, count.data_ptr(), _stream_ptr(eig))
    if rc != KLT_OK:
        _raise_status(rc, "klt_corner_candidates")
    counts = count.cpu().numpy()          # synchronises
    out = []
    n = ctypes.c_int(0)
    for b in range(B):
        k = keys[b, :int(counts[b])].cpu().numpy().view(np.uint64).copy()
        c_cap = maxCorners if maxCorners > 0 else max(len(k), 1)
        res = np.empty((c_cap, 2), np.float32)
        rc = L.klt_select_corners_host(k.ctypes.data, len(k), W, H, maxCorners, minDistance, res.ctypes.data, c_cap, ctypes.byref(n))
        if rc != KLT_OK:
            _raise_status(rc, "klt_select_corners_host")
        out.append(res[:n.value].reshape(-1, 1, 2).copy() if n.value else None)
    return out


def mask_from_points(points, radius, shape, ctx=None):
    """Detection mask of reference src/extractor/extractor.py:102-107 for (N, 2) float32 CUDA points -> (H, W) uint8 CUDA
    tensor: 255, with a filled cv2.circle of `radius` (value 0) around np.int32 of every point."""
    torch = _torch()
    if not (isinstance(points, torch.Tensor) and points.is_cuda and points.dtype == torch.float32):
        raise error("klt_b200: points must be a float32 CUDA tensor")
    pts = points.reshape(-1, 2).contiguous()
    h, w = int(shape[0]), int(shape[1])
    mask = torch.empty((h, w), dtype=torch.uint8, device=pts.device)
    ctx = ctx or _lib.default_context(pts.device.index or 0)
    rc = _lib.load().klt_corner_mask_from_points(ctx.handle, pts.data_ptr() if pts.numel() else None, pts.shape[0], int(radius), w, h,
                                                 mask.data_ptr(), w, _stream_ptr(mask))
    if rc != KLT_OK:
        _raise_status(rc, "klt_corner_mask_from_points")
    return mask
