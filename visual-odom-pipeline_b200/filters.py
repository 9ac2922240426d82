"""Drop-in replacement for the OpenCV call of the reference's loader (SURVEY.md s8f rank 3).

``bilateralFilter`` has the signature and return contract of ``cv2.bilateralFilter`` as the reference applies it to every
frame it reads (src/loader/loader.py:16-20,86):

    img = bilateralFilter(cv2.imread(path, cv2.IMREAD_GRAYSCALE), d=5, sigmaColor=1.5, sigmaSpace=1.5)

uint8 (h, w) numpy in -> fresh uint8 (h, w) out.  The arithmetic is OpenCV's own code path (oracle/bilateral_oracle.c
B.1-B.6, what an OpenCV build without IPP runs): identical to it except on exact rounding ties (< 1e-5 of the pixels, by 1)
and within 1 of the IPP-enabled wheel, whose closed-source primitive differs from OpenCV's own code by 1 on about half of
the pixels.  sm_100a kernel behind the C ABI (csrc/klt_bilateral.cu); no CPU fallback.
"""
import numpy as np

from . import _lib
from ._lib import KLT_OK
from .corners import _u8_image
from .lk import _addr, _fail, _raise_status, error

BORDER_REFLECT_101 = 4   # cv2.BORDER_DEFAULT


def _check_params(d, sigmaColor, sigmaSpace, borderType):
    if int(borderType) != BORDER_REFLECT_101:
        raise error("klt_b200: bilateralFilter: only BORDER_REFLECT_101 / BORDER_DEFAULT (what the reference uses, loader.py:86)")
    d = int(d)
    sigmaColor, sigmaSpace = float(sigmaColor), float(sigmaSpace)
    if not (np.isfinite(sigmaColor) and np.isfinite(sigmaSpace)):
        _fail("bilateralFilter: sigmaColor and sigmaSpace must be finite")
    return d, sigmaColor, sigmaSpace


def bilateralFilter(src, d, sigmaColor, sigmaSpace, dst=None, borderType=BORDER_REFLECT_101, device=0):
    """cv2.bilateralFilter(src, d, sigmaColor, sigmaSpace[, dst[, borderType]]) -> uint8 (h, w), on a B200."""
    d, sigmaColor, sigmaSpace = _check_params(d, sigmaColor, sigmaSpace, borderType)
    img = _u8_image(src, "src", "bilateralFilter")
    h, w = img.shape
    out = np.empty((h, w), np.uint8)
    ctx = _lib.default_context(device)
    rc = _lib.load().klt_bilateral_filter_host(ctx.handle, _addr(img), img.strides[0], w, h, d, sigmaColor, sigmaSpace,
                                               _addr(out), out.strides[0])
    if rc != KLT_OK:
        _raise_status(rc, "bilateralFilter")
    return out


def bilateral_filter(images, d=5, sigmaColor=1.5, sigmaSpace=1.5, out=None, ctx=None):
    """The same filter on a (B, H, W) / (H, W) uint8 CUDA tensor, one launch for the batch, asynchronous on the current
    torch stream.  `out`: optional (B, H, W) uint8 CUDA tensor (any row pitch); default: 128-byte-pitched storage, i.e. a
    frame batch the pyramid / LK kernels take on their fast path."""
    import ctypes

    import torch

    from .tracker import _as_image_batch, _batch_stride, _stream_ptr, alloc_image_batch
    d, sigmaColor, sigmaSpace = _check_params(d, sigmaColor, sigmaSpace, BORDER_REFLECT_101)
    img = _as_image_batch(images)
    B, H, W = img.shape
    if out is None:
        out = alloc_image_batch(B, H, W, device=img.device)
    if not (isinstance(out, torch.Tensor) and out.is_cuda and out.dtype == torch.uint8 and tuple(out.shape) == (B, H, W) and out.stride(2) == 1):
        raise error("klt_b200: bilateral_filter: `out` must be a (B, H, W) uint8 CUDA tensor with unit column stride")
    if out.data_ptr() == img.data_ptr():
        raise error("klt_b200: bilateral_filter: in-place filtering is not supported")
    ctx = ctx or _lib.default_context(img.device.index or 0)
    rc = _lib.load().klt_bilateral_filter(ctx.handle, img.data_ptr(), W, H, img.stride(1), _batch_stride(img),
                                          out.data_ptr(), out.stride(1), _batch_stride(out), B, d, sigmaColor, sigmaSpace,
                                          _stream_ptr(img))
    if rc != KLT_OK:
        _raise_status(rc, "klt_bilateral_filter")
    return out if images.dim() == 3 else out[0]
