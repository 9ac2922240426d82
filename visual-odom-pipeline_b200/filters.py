"""Drop-in replacements for the OpenCV pre-filters of a KLT front end: the reference's loader filter (SURVEY.md s8f
rank 3) and contrast-limited adaptive histogram equalisation.

``bilateralFilter`` has the signature and return contract of ``cv2.bilateralFilter`` as the reference applies it to every
frame it reads (src/loader/loader.py:16-20,86):

    img = bilateralFilter(cv2.imread(path, cv2.IMREAD_GRAYSCALE), d=5, sigmaColor=1.5, sigmaSpace=1.5)

uint8 (h, w) numpy in -> fresh uint8 (h, w) out.  The arithmetic is OpenCV's own code path (oracle/bilateral_oracle.c
B.1-B.6, what an OpenCV build without IPP runs): identical to it except on exact rounding ties (< 1e-5 of the pixels, by 1)
and within 1 of the IPP-enabled wheel, whose closed-source primitive differs from OpenCV's own code by 1 on about half of
the pixels.  sm_100a kernel behind the C ABI (csrc/klt_bilateral.cu); no CPU fallback.

``createCLAHE`` has the contract of ``cv2.createCLAHE`` for what a tracker needs of it, 8-bit single-channel frames:

    img = createCLAHE(clipLimit=3.0, tileGridSize=(8, 8)).apply(frame)

bit-identical to the cv2 wheel (oracle/clahe_oracle.py C.1-C.5); sm_100a kernels behind the C ABI (csrc/klt_clahe.cu).
16-bit images, which cv2 also takes, raise `error`: there is no fallback.
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


def check_clahe(clipLimit, tileGridSize, w=None, h=None, func="createCLAHE"):
    """clipLimit and tileGridSize checked as klt_clahe checks them (against a w x h image when given; before any device
    work) -> (clipLimit float, tiles_x, tiles_y)."""
    try:
        clip = float(clipLimit)
        tx, ty = (int(v) for v in tileGridSize)
    except (TypeError, ValueError):
        raise error("klt_b200: %s: clipLimit must be a number and tileGridSize a pair of ints" % func)
    if not np.isfinite(clip):
        raise error("klt_b200: %s: clipLimit must be finite" % func)
    if tx < 1 or ty < 1:
        _fail("tilesX_ > 0 && tilesY_ > 0 in function '%s'" % func)
    if tx * ty > _lib.KLT_MAX_CLAHE_TILES:
        raise error("klt_b200: %s: tileGridSize %r has more than KLT_MAX_CLAHE_TILES (%d) tiles" % (func, (tx, ty), _lib.KLT_MAX_CLAHE_TILES))
    if w is not None and clip > 0:
        pad = w % tx != 0 or h % ty != 0
        total = ((w + tx - w % tx) // tx if pad else w // tx) * ((h + ty - h % ty) // ty if pad else h // ty)
        if total > 2 ** 31 - 1 or clip * total / 256 >= 2.0 ** 31:
            raise error("klt_b200: %s: clipLimit %r is too large for %d x %d tiles of a %d x %d image (the clip count must fit "
                        "an int32)" % (func, clip, tx, ty, w, h))
    return clip, tx, ty


class CLAHE:
    """What cv2.createCLAHE returns, for 8-bit single-channel images: apply(src[, dst]) and the clip / grid accessors."""

    def __init__(self, clipLimit=40.0, tileGridSize=(8, 8), device=0):
        self.device = device
        self.setClipLimit(clipLimit)
        self.setTilesGridSize(tileGridSize)

    def getClipLimit(self):
        return self._clip

    def setClipLimit(self, clipLimit):
        self._clip = check_clahe(clipLimit, (1, 1))[0]

    def getTilesGridSize(self):
        return self._tiles

    def setTilesGridSize(self, tileGridSize):
        self._tiles = check_clahe(0.0, tileGridSize)[1:]

    def apply(self, src, dst=None):
        """uint8 (h, w) numpy (any row stride) -> equalized uint8 (h, w): written into `dst` when it is a uint8 (h, w) array
        (which may be `src`), else a fresh array.  clipLimit <= 0: no clipping."""
        if isinstance(src, np.ndarray) and src.dtype == np.uint16:
            raise error("klt_b200: CLAHE.apply: 16-bit images are not supported (8-bit single-channel frames only)")
        if not isinstance(src, np.ndarray) or src.dtype != np.uint8 or not (src.ndim == 2 or (src.ndim == 3 and src.shape[2] == 1)):
            _fail("_src.type() == CV_8UC1 || _src.type() == CV_16UC1 in function 'apply'")
        img = _u8_image(src, "src", "apply")
        h, w = img.shape
        clip, tx, ty = check_clahe(self._clip, self._tiles, w, h, "CLAHE.apply")
        out = dst if (isinstance(dst, np.ndarray) and dst.dtype == np.uint8 and dst.shape == (h, w) and dst.strides[1] == 1
                      and dst.strides[0] >= w and dst.flags.writeable) else np.empty((h, w), np.uint8)
        ctx = _lib.default_context(self.device)
        rc = _lib.load().klt_clahe_host(ctx.handle, _addr(img), img.strides[0], w, h, clip, tx, ty, _addr(out), out.strides[0])
        if rc != KLT_OK:
            _raise_status(rc, "CLAHE.apply")
        if dst is not None and out is not dst and isinstance(dst, np.ndarray) and dst.dtype == np.uint8 and dst.shape == (h, w):
            dst[...] = out
            return dst
        return out


def createCLAHE(clipLimit=40.0, tileGridSize=(8, 8)):
    """cv2.createCLAHE([clipLimit[, tileGridSize]]) -> CLAHE, on a B200 (8-bit single-channel images)."""
    return CLAHE(clipLimit, tileGridSize)


def clahe_launch(img, out, clip, tiles, ws, ctx, stream):
    """klt_clahe on (B, H, W) uint8 CUDA tensors with a workspace tensor of klt_clahe_ws_bytes; arguments checked."""
    from .tracker import _batch_stride
    B, H, W = img.shape
    rc = _lib.load().klt_clahe(ctx.handle, img.data_ptr(), W, H, img.stride(1), _batch_stride(img), out.data_ptr(), out.stride(1),
                               _batch_stride(out), B, clip, tiles[0], tiles[1], ws.data_ptr(), ws.numel(), stream)
    if rc != KLT_OK:
        _raise_status(rc, "klt_clahe")


def clahe(images, clipLimit=40.0, tileGridSize=(8, 8), out=None, ctx=None):
    """createCLAHE(clipLimit, tileGridSize).apply on every image of a (B, H, W) / (H, W) uint8 CUDA tensor: two launches
    for the batch, asynchronous on the current torch stream.  `out`: optional uint8 CUDA tensor shaped like `images` (any
    row pitch; `images` itself equalizes in place), returned as given; default: 128-byte-pitched storage, as
    bilateral_filter."""
    import torch

    from .tracker import _as_image_batch, _batch_stride, _stream_ptr, alloc_image_batch
    if isinstance(images, torch.Tensor) and images.is_cuda and images.dtype == torch.uint16:
        raise error("klt_b200: clahe: 16-bit images are not supported (8-bit single-channel frames only)")
    img = _as_image_batch(images)
    B, H, W = img.shape
    clip, tx, ty = check_clahe(clipLimit, tileGridSize, W, H, "clahe")
    given = out
    if out is None:
        out = alloc_image_batch(B, H, W, device=img.device)
    elif isinstance(out, torch.Tensor) and out.dim() == 2 and images.dim() == 2:
        out = out.unsqueeze(0)
    if not (isinstance(out, torch.Tensor) and out.is_cuda and out.dtype == torch.uint8 and tuple(out.shape) == (B, H, W) and out.stride(2) == 1):
        raise error("klt_b200: clahe: `out` must be a uint8 CUDA tensor shaped like `images`, with unit column stride")
    if out.data_ptr() == img.data_ptr() and (out.stride(1) != img.stride(1) or _batch_stride(out) != _batch_stride(img)):
        raise error("klt_b200: clahe: in place, `out` must be `images` itself")
    ctx = ctx or _lib.default_context(img.device.index or 0)
    ws = torch.empty((int(_lib.load().klt_clahe_ws_bytes(B, tx, ty)),), dtype=torch.uint8, device=img.device)
    clahe_launch(img, out, clip, (tx, ty), ws, ctx, _stream_ptr(img))
    if given is not None:
        return given
    return out if images.dim() == 3 else out[0]
