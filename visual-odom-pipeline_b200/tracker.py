"""Device-resident API: batched pyramids and LK on torch CUDA tensors (no host round trips).

PyTorch is used for device memory and streams only; every kernel is libklt_b200's.  This is the
path the batched configs use (BASELINE.json configs[3]: many independent KITTI-shape sequences) and
the caller-side fusion of the reference's tracking step (SURVEY.md s8f rank 1): one frame's
pyramid is built once and reused as the next pair's `prev`.
"""
import ctypes

from . import _lib
from ._lib import KLT_OK, klt_pyr_layout
from .lk import _check_win_level, _fail, _raise_status, error, make_params


def _torch():
    import torch
    return torch


def _stream_ptr(t):
    torch = _torch()
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _as_image_batch(img):
    torch = _torch()
    if not (isinstance(img, torch.Tensor) and img.is_cuda):
        raise error("klt_b200: expected a CUDA uint8 tensor")
    if img.dtype != torch.uint8:
        _fail("img.depth() == CV_8U in function 'buildOpticalFlowPyramid'")
    if img.dim() == 2:
        img = img.unsqueeze(0)
    if img.dim() != 3 or img.numel() == 0:
        raise error("klt_b200: images must be (H, W) or (B, H, W) uint8")
    if img.stride(2) != 1 or img.stride(1) < img.shape[2] or (img.shape[0] > 1 and img.stride(0) < img.stride(1) * img.shape[1]):
        img = img.contiguous()
    return img


def _batch_stride(t):
    """Bytes between the items of a (B, H, W) tensor; a batch of one may carry any stride(0), so its item is its H rows."""
    return t.stride(0) if t.shape[0] > 1 else t.stride(1) * t.shape[1]


def alloc_image_batch(batch, h, w, device="cuda"):
    """(B, H, W) uint8 view into 128-byte-pitched storage: rows start 16-byte aligned so the pyramid
    kernel takes its 128-bit load path (a plain contiguous tensor with odd W falls back to byte loads)."""
    torch = _torch()
    pitch = (w + 127) // 128 * 128
    store = torch.zeros((batch, h, pitch), dtype=torch.uint8, device=device)   # padding columns are read by 16-byte granule copies
    return store[:, :, :w]


class DevicePyramid:
    """Gaussian pyramid of a batch of images on the device (levels >= 1 in one buffer).

    Level 0 is the caller's tensor itself unless `copy=True`: without a copy the caller must leave the tensor unmodified
    for as long as the pyramid is used (levels 1..top would otherwise belong to another image than level 0).
    `copy=True` moves level 0 into storage owned by the pyramid (128-byte pitch: the kernels' 128-bit load path)."""

    def __init__(self, images, winSize=(21, 21), maxLevel=3, ctx=None, out=None, copy=False, prefilter=None):
        torch = _torch()
        win_w, win_h, maxLevel = _check_win_level(winSize, maxLevel)
        self.images = _as_image_batch(images)
        if prefilter is not None:
            # the loader's bilateral filter (loader.py:16-20,86) writes the pyramid's own level 0: the raw frame is read
            # once and no separate copy is made
            from .filters import bilateral_filter
            self.images = bilateral_filter(self.images, *prefilter, ctx=ctx)
        elif copy:
            own = alloc_image_batch(self.images.shape[0], self.images.shape[1], self.images.shape[2], device=self.images.device)
            own.copy_(self.images)
            self.images = own
        B, H, W = self.images.shape
        self.ctx = ctx or _lib.default_context(self.images.device.index or 0)
        self.win = (win_w, win_h)
        self.layout = klt_pyr_layout()
        L = _lib.load()
        rc = L.klt_pyr_plan(W, H, win_w, win_h, maxLevel, B, ctypes.byref(self.layout))
        if rc != KLT_OK:
            _raise_status(rc, "klt_pyr_plan")
        self.layout.level[0].pitch = self.images.stride(1)
        self.layout.level[0].batch_stride = _batch_stride(self.images)
        nbytes = max(int(self.layout.bytes), 1)
        if out is not None:
            if out.numel() < nbytes or out.dtype != torch.uint8 or not out.is_cuda:
                raise error("klt_b200: pyramid buffer too small")
            self.buffer = out
        else:
            # zeros: the pitch padding of a level is read (never used) by the 16-byte granule copies of the next step
            self.buffer = torch.zeros(nbytes, dtype=torch.uint8, device=self.images.device)
        self.build()

    @property
    def top(self):
        return int(self.layout.top)

    def build(self):
        """(Re)build levels 1..top from self.images on the current torch stream."""
        L = _lib.load()
        rc = L.klt_pyr_build(self.ctx.handle, self.images.data_ptr(), ctypes.byref(self.layout), self.buffer.data_ptr(),
                             0, 0, _stream_ptr(self.images))
        if rc != KLT_OK:
            _raise_status(rc, "klt_pyr_build")
        return self

    def level(self, l):
        """(B, h_l, w_l) uint8 view of level l."""
        torch = _torch()
        if l == 0:
            return self.images
        lv = self.layout.level[l]
        B = self.images.shape[0]
        flat = self.buffer[lv.offset: lv.offset + lv.batch_stride * B]
        return torch.as_strided(flat, (B, lv.h, lv.w), (lv.batch_stride, lv.pitch, 1))

    def algorithmic_bytes(self):
        """SURVEY.md s8d: each source level read once + each produced level written once (u8)."""
        B = self.images.shape[0]
        tot = 0
        for l in range(self.top):
            a, b = self.layout.level[l], self.layout.level[l + 1]
            tot += a.w * a.h + b.w * b.h
        return tot * B


def lk_track(prev, nxt, prevPts, nextPts=None, criteria=(3, 30, 0.01), flags=0, minEigThreshold=1e-4,
             return_iters=False):
    """Track (B, N, 2) float32 CUDA points from pyramid `prev` to pyramid `nxt` (one kernel launch).

    -> nextPts (B, N, 2) float32, status (B, N) uint8, err (B, N) float32 [, iters (B, N) int32]
    """
    torch = _torch()
    if prev.layout.top != nxt.layout.top or prev.images.shape != nxt.images.shape or prev.win != nxt.win:
        _fail("prevPyr[level * lvlStep1].size() == nextPyr[level * lvlStep2].size() in function 'calc'")
    B = prev.images.shape[0]
    if not (isinstance(prevPts, torch.Tensor) and prevPts.is_cuda and prevPts.dtype == torch.float32
            and prevPts.dim() == 3 and prevPts.shape[0] == B and prevPts.shape[2] == 2):
        _fail("(npoints = prevPts.checkVector(2, CV_32F, true)) >= 0 in function 'calc'")
    pts = prevPts.contiguous()
    N = pts.shape[1]
    dev = pts.device
    if int(flags) & _lib.OPTFLOW_USE_INITIAL_FLOW:
        if nextPts is None or tuple(nextPts.shape) != tuple(pts.shape):
            _fail("nextPts.checkVector(2, CV_32F, true) == npoints in function 'calc'")
        out = nextPts.to(torch.float32).contiguous().clone()
    else:
        out = torch.empty_like(pts)
    status = torch.empty((B, N), dtype=torch.uint8, device=dev)
    err = torch.empty((B, N), dtype=torch.float32, device=dev)
    iters = torch.zeros((B, N), dtype=torch.int32, device=dev) if return_iters else None
    if N > 0:
        params = make_params(prev.win, criteria, flags, minEigThreshold)
        L = _lib.load()
        rc = L.klt_lk_track(prev.ctx.handle, prev.images.data_ptr(), prev.buffer.data_ptr(), nxt.images.data_ptr(),
                            nxt.buffer.data_ptr(), ctypes.byref(prev.layout), 0, 0, 1, B, pts.data_ptr(), out.data_ptr(),
                            status.data_ptr(), err.data_ptr(), iters.data_ptr() if return_iters else None, N,
                            ctypes.byref(params), _stream_ptr(pts))
        if rc != KLT_OK:
            _raise_status(rc, "klt_lk_track")
    return (out, status, err, iters) if return_iters else (out, status, err)


def calc_optical_flow_pyr_lk_device(prevImg, nextImg, prevPts, nextPts=None, winSize=(21, 21), maxLevel=3,
                                    criteria=(3, 30, 0.01), flags=0, minEigThreshold=1e-4):
    """cv2.calcOpticalFlowPyrLK contract on CUDA tensors; outputs are CUDA tensors shaped like cv2's."""
    torch = _torch()
    prev = DevicePyramid(prevImg, winSize, maxLevel)
    nxt = DevicePyramid(nextImg, winSize, maxLevel, ctx=prev.ctx)
    B = prev.images.shape[0]
    shape = tuple(prevPts.shape)
    if B == 1 and prevPts.dim() in (2, 3) and not (prevPts.dim() == 3 and prevPts.shape[0] == 1 and prevImg.dim() == 3):
        pts = prevPts.reshape(1, -1, 2)
        nin = nextPts.reshape(1, -1, 2) if nextPts is not None else None
    else:
        pts, nin = prevPts, nextPts
    if pts.numel() == 0:
        return None, None, None
    out, st, er = lk_track(prev, nxt, pts, nin, criteria, flags, minEigThreshold)
    if prevImg.dim() == 2:
        return out.reshape(shape), st.reshape(-1, 1), er.reshape(-1, 1)
    return out, st, er


def track_filter(p0, p1, p0r, max_bidir_error, w, h, ctx=None):
    """Bidirectional-error / bounds filter of reference src/extractor/extractor.py:46-47,53 on CUDA tensors.
    p0, p1, p0r: (..., 2) float32 -> keep (...) bool, bidir (...) float32."""
    torch = _torch()
    a, b, c = p0.contiguous(), p1.contiguous(), p0r.contiguous()
    n = a.numel() // 2
    keep = torch.empty(a.shape[:-1], dtype=torch.uint8, device=a.device)
    bidir = torch.empty(a.shape[:-1], dtype=torch.float32, device=a.device)
    if n:
        ctx = ctx or _lib.default_context(a.device.index or 0)
        rc = _lib.load().klt_track_filter(ctx.handle, a.data_ptr(), b.data_ptr(), c.data_ptr(), n, float(max_bidir_error), int(w), int(h),
                                          keep.data_ptr(), bidir.data_ptr(), _stream_ptr(a))
        if rc != KLT_OK:
            _raise_status(rc, "klt_track_filter")
    return keep.bool(), bidir


class KLTTracker:
    """Frame-to-frame tracker that keeps the last frame's pyramid on the device.

    Caller-side fusion of the reference's tracking step (src/extractor/extractor.py:38-88 and
    src/pipeline/pipeline.py:98-103): the reference calls cv2.calcOpticalFlowPyrLK four times per
    frame on the same image pair, i.e. OpenCV builds 8 pyramids per frame; here each frame's pyramid
    is built exactly once and reused as the next pair's `prev`.  The tracker copies every frame into storage of its
    own, so the caller may overwrite its frame tensor (e.g. upload frame t+1 into the same buffer) as soon as a call
    returns.
    """

    def __init__(self, winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03), flags=0, minEigThreshold=1e-4, prefilter=None):
        """prefilter = (d, sigmaColor, sigmaSpace): apply the loader's cv2.bilateralFilter (loader.py:16-20,86) to every raw
        frame on the device while it is copied into the tracker's storage (None: frames arrive filtered)."""
        self.winSize, self.maxLevel, self.criteria = winSize, maxLevel, criteria
        self.flags, self.minEigThreshold = flags, minEigThreshold
        self.prefilter = prefilter
        self.prev = None

    def reset(self, images):
        self.prev = DevicePyramid(images, self.winSize, self.maxLevel, copy=True, prefilter=self.prefilter)
        return self

    def track(self, images, prevPts, bidirectional=False):
        """Track prevPts (B, N, 2) from the stored frame into `images`; the new frame becomes `prev`.

        bidirectional=True repeats the reference's second call (extractor.py:45: same image pair,
        started from the forward result) and returns it as a 4th output."""
        if self.prev is None:
            raise error("klt_b200: KLTTracker.track() before reset()")
        nxt = DevicePyramid(images, self.winSize, self.maxLevel, ctx=self.prev.ctx, copy=True, prefilter=self.prefilter)
        out = lk_track(self.prev, nxt, prevPts, None, self.criteria, self.flags, self.minEigThreshold)
        if bidirectional:
            back = lk_track(self.prev, nxt, out[0], None, self.criteria, self.flags, self.minEigThreshold)
            out = out + (back[0],)
        self.prev = nxt
        return out

    def track_filtered(self, images, prevPts, max_bidir_error=30):
        """The reference's whole KLT step for a batch of sequences (extractor.py:43-53): forward pass, the second pass
        started from the forward result, bidirectional-error and inclusive-bounds filter -- all on the device, the
        new frame's pyramid built once and kept as the next `prev`.
        -> p1 (B, N, 2), keep (B, N) bool, bidir (B, N) float32, status (B, N) uint8, err (B, N) float32"""
        p1, st, er, p0r = self.track(images, prevPts, bidirectional=True)
        H, W = self.prev.images.shape[1], self.prev.images.shape[2]
        keep, bidir = track_filter(prevPts, p1, p0r, max_bidir_error, W, H, ctx=self.prev.ctx)
        return p1, keep, bidir, st, er

    def step(self, image, points, max_bidir_error=30, mask_radius=10, maxCorners=1000, qualityLevel=0.03, minDistance=10,
             blockSize=31):
        """One frame of the reference's data-parallel work for ONE sequence, everything on the device
        (src/pipeline/pipeline.py:98-103,159-163 with src/extractor/extractor.py:38-88,102-111): track `points`
        (N, 2) float32 CUDA tensor from the stored frame into `image` (forward pass + the reference's second pass),
        drop them by bidirectional error and the inclusive bounds test, rasterise the detection mask around the
        survivors, detect new Shi-Tomasi corners.  One upload (the new frame, by the caller) and one small download
        (candidate keys for the sequential selection) per frame.
        -> survivors (M, 2) float32 CUDA, keep (N,) bool CUDA, new corners float32 (K, 1, 2) numpy or None"""
        torch = _torch()
        from . import detector as D
        img = _as_image_batch(image)
        if img.shape[0] != 1:
            raise error("klt_b200: KLTTracker.step() takes one frame")
        pts = points.reshape(1, -1, 2)
        if pts.shape[1]:
            p1, keep, _bidir, _st, _er = self.track_filtered(img, pts, max_bidir_error)
            survivors = p1[0][keep[0]]
            keep = keep[0]
        else:
            self.prev = DevicePyramid(img, self.winSize, self.maxLevel, ctx=self.prev.ctx if self.prev is not None else None, copy=True,
                                      prefilter=self.prefilter)
            survivors = torch.zeros((0, 2), dtype=torch.float32, device=img.device)
            keep = torch.zeros((0,), dtype=torch.bool, device=img.device)
        if self.prefilter is not None:
            img = self.prev.images            # detection runs on the filtered frame, as in the reference (loader.py:86)
        H, W = img.shape[1], img.shape[2]
        mask = D.mask_from_points(survivors, mask_radius, (H, W), ctx=self.prev.ctx)
        new = D.good_features_to_track(img, maxCorners, qualityLevel, minDistance, mask=mask.unsqueeze(0), blockSize=blockSize,
                                       ctx=self.prev.ctx)[0]
        return survivors, keep, new
