"""Device-resident API: batched pyramids and LK on torch CUDA tensors (no host round trips).

PyTorch is used for device memory and streams only; every kernel is libklt_b200's.  This is the
path the batched configs use (BASELINE.json configs[3]: many independent KITTI-shape sequences) and
the caller-side fusion of the reference's tracking step (SURVEY.md s8f rank 1): one frame's
pyramid is built once and reused as the next pair's `prev`.
"""
import collections
import ctypes
import numbers

from . import _lib
from ._lib import KLT_OK, klt_pyr_layout
from .lk import _check_win_level, _fail, _raise_status, check_second_pass, error, make_params


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


def check_equalize(equalize, w=None, h=None, func="equalize"):
    """equalize = (clipLimit, tileGridSize) checked as klt_clahe checks it (against w x h frames when given) ->
    (clipLimit, (tiles_x, tiles_y)), or None."""
    if equalize is None:
        return None
    from .filters import check_clahe
    if not (isinstance(equalize, (tuple, list)) and len(equalize) == 2):
        raise error("klt_b200: %s must be None or (clipLimit, tileGridSize)" % func)
    clip, tx, ty = check_clahe(equalize[0], equalize[1], w, h, func)
    return clip, (tx, ty)


class DevicePyramid:
    """Gaussian pyramid of a batch of images on the device (levels >= 1 in one buffer).

    Level 0 is the caller's tensor itself unless `copy=True`: without a copy the caller must leave the tensor unmodified
    for as long as the pyramid is used (levels 1..top would otherwise belong to another image than level 0).
    `copy=True` moves level 0 into storage owned by the pyramid (128-byte pitch: the kernels' 128-bit load path).
    equalize = (clipLimit, tileGridSize): level 0 is createCLAHE(clipLimit, tileGridSize).apply of the (pre-filtered) frame,
    equalized in the pyramid's own storage (a fresh one when the level would otherwise be the caller's tensor)."""

    def __init__(self, images, winSize=(21, 21), maxLevel=3, ctx=None, out=None, copy=False, prefilter=None, equalize=None):
        torch = _torch()
        win_w, win_h, maxLevel = _check_win_level(winSize, maxLevel)
        self.images = _as_image_batch(images)
        equalize = check_equalize(equalize, self.images.shape[2], self.images.shape[1])
        if prefilter is not None:
            # the loader's bilateral filter (loader.py:16-20,86) writes the pyramid's own level 0: the raw frame is read
            # once and no separate copy is made
            from .filters import bilateral_filter
            self.images = bilateral_filter(self.images, *prefilter, ctx=ctx)
        elif copy:
            own = alloc_image_batch(self.images.shape[0], self.images.shape[1], self.images.shape[2], device=self.images.device)
            own.copy_(self.images)
            self.images = own
        if equalize is not None:
            from .filters import clahe
            owned = prefilter is not None or copy
            self.images = clahe(self.images, *equalize, out=self.images if owned else None, ctx=ctx)
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

    def __init__(self, winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03), flags=0, minEigThreshold=1e-4, prefilter=None,
                 equalize=None):
        """prefilter = (d, sigmaColor, sigmaSpace): apply the loader's cv2.bilateralFilter (loader.py:16-20,86) to every raw
        frame on the device while it is copied into the tracker's storage (None: frames arrive filtered).
        equalize = (clipLimit, tileGridSize), e.g. (3.0, (8, 8)): equalize every frame on the device with
        createCLAHE(clipLimit, tileGridSize).apply, after prefilter when both are set, before its pyramid is built; LK
        and detection (and its mask) then run on the equalized frame.  None (the default) launches nothing of this."""
        self.winSize, self.maxLevel, self.criteria = winSize, maxLevel, criteria
        self.flags, self.minEigThreshold = flags, minEigThreshold
        self.prefilter = prefilter
        check_equalize(equalize, func="KLTTracker equalize")
        self.equalize = equalize
        self.prev = None

    def reset(self, images):
        self.prev = DevicePyramid(images, self.winSize, self.maxLevel, copy=True, prefilter=self.prefilter,
                                  equalize=self.equalize)
        return self

    def track(self, images, prevPts, bidirectional=False, second_pass="reference"):
        """Track prevPts (B, N, 2) from the stored frame into `images`; the new frame becomes `prev`.

        bidirectional=True repeats the reference's second call (extractor.py:45: same image pair,
        started from the forward result) and returns it as a 4th output.  second_pass="reverse" makes that call the
        forward-backward check instead: the forward result tracked from `images` back into the stored frame."""
        check_second_pass(second_pass)
        if self.prev is None:
            raise error("klt_b200: KLTTracker.track() before reset()")
        nxt = DevicePyramid(images, self.winSize, self.maxLevel, ctx=self.prev.ctx, copy=True, prefilter=self.prefilter,
                            equalize=self.equalize)
        out = lk_track(self.prev, nxt, prevPts, None, self.criteria, self.flags, self.minEigThreshold)
        if bidirectional:
            a, b = (nxt, self.prev) if second_pass == "reverse" else (self.prev, nxt)
            back = lk_track(a, b, out[0], None, self.criteria, self.flags, self.minEigThreshold)
            out = out + (back[0],)
        self.prev = nxt
        return out

    def track_filtered(self, images, prevPts, max_bidir_error=30, second_pass="reference"):
        """The reference's whole KLT step for a batch of sequences (extractor.py:43-53): forward pass, the second pass
        started from the forward result, bidirectional-error and inclusive-bounds filter -- all on the device, the
        new frame's pyramid built once and kept as the next `prev`.  second_pass="reverse": the forward-backward check
        (see track); a useful max_bidir_error is then about 1 px.
        -> p1 (B, N, 2), keep (B, N) bool, bidir (B, N) float32, status (B, N) uint8, err (B, N) float32"""
        p1, st, er, p0r = self.track(images, prevPts, bidirectional=True, second_pass=second_pass)
        H, W = self.prev.images.shape[1], self.prev.images.shape[2]
        keep, bidir = track_filter(prevPts, p1, p0r, max_bidir_error, W, H, ctx=self.prev.ctx)
        return p1, keep, bidir, st, er

    def step(self, image, points, max_bidir_error=30, mask_radius=10, maxCorners=1000, qualityLevel=0.03, minDistance=10,
             blockSize=31, second_pass="reference"):
        """One frame of the reference's data-parallel work for ONE sequence, everything on the device
        (src/pipeline/pipeline.py:98-103,159-163 with src/extractor/extractor.py:38-88,102-111): track `points`
        (N, 2) float32 CUDA tensor from the stored frame into `image` (forward pass + the reference's second pass),
        drop them by bidirectional error and the inclusive bounds test, rasterise the detection mask around the
        survivors, detect new Shi-Tomasi corners.  One upload (the new frame, by the caller) and one small download
        (candidate keys for the sequential selection) per frame.  second_pass="reverse": the forward-backward check
        (see track); a useful max_bidir_error is then about 1 px.
        -> survivors (M, 2) float32 CUDA, keep (N,) bool CUDA, new corners float32 (K, 1, 2) numpy or None"""
        torch = _torch()
        from . import detector as D
        check_second_pass(second_pass)
        img = _as_image_batch(image)
        if img.shape[0] != 1:
            raise error("klt_b200: KLTTracker.step() takes one frame")
        pts = points.reshape(1, -1, 2)
        if pts.shape[1]:
            p1, keep, _bidir, _st, _er = self.track_filtered(img, pts, max_bidir_error, second_pass)
            survivors = p1[0][keep[0]]
            keep = keep[0]
        else:
            self.prev = DevicePyramid(img, self.winSize, self.maxLevel, ctx=self.prev.ctx if self.prev is not None else None, copy=True,
                                      prefilter=self.prefilter, equalize=self.equalize)
            survivors = torch.zeros((0, 2), dtype=torch.float32, device=img.device)
            keep = torch.zeros((0,), dtype=torch.bool, device=img.device)
        if self.prefilter is not None or self.equalize is not None:
            img = self.prev.images            # detection runs on the filtered / equalized frame, as LK does (loader.py:86)
        H, W = img.shape[1], img.shape[2]
        mask = D.mask_from_points(survivors, mask_radius, (H, W), ctx=self.prev.ctx)
        new = D.good_features_to_track(img, maxCorners, qualityLevel, minDistance, mask=mask.unsqueeze(0), blockSize=blockSize,
                                       ctx=self.prev.ctx)[0]
        return survivors, keep, new

    def step_batch(self, images, points, counts, max_bidir_error=30, mask_radius=10, maxCorners=1000, qualityLevel=0.03,
                   minDistance=10, blockSize=31, second_pass="reference"):
        """`step` for B sequences at once, with a different point count per sequence (klt_frame_step_batch: one launch
        sequence for the whole batch, one host synchronisation).  images: (B, H, W) uint8 CUDA, B as in `reset`;
        points: (B, N, 2) float32 CUDA; counts: (B,) int32 CUDA, sequence b owns points[b, :counts[b]].
        -> next_points (B, M, 2) float32, next_counts (B,) int32, keep (B, N) bool, n_new (B,) int32, all CUDA, with
        M = max(next_counts): next_points[b, :s_b] are sequence b's survivors in input order (s_b = keep[b].sum()), then its
        n_new[b] new corners strongest first.  Per sequence, bit-identical to `step` on points[b, :counts[b]].
        second_pass="reverse": the forward-backward check (see track; klt_frame_step_batch_fb_async, then one
        synchronisation for the counts and the flag word); a useful max_bidir_error is then about 1 px."""
        torch = _torch()
        import numpy as np
        check_second_pass(second_pass)
        if self.prev is None:
            raise error("klt_b200: KLTTracker.step_batch() before reset()")
        img = _as_image_batch(images)
        B, H, W = self.prev.images.shape
        if tuple(img.shape) != (B, H, W) or img.device != self.prev.images.device:
            raise error("klt_b200: step_batch() takes (B, H, W) frames of the batch and size the tracker was reset with")
        if not (isinstance(points, torch.Tensor) and points.device == img.device and points.dtype == torch.float32
                and points.dim() == 3 and points.shape[0] == B and points.shape[2] == 2):
            raise error("klt_b200: step_batch() points must be a (B, N, 2) float32 tensor on the frames' device")
        if not (isinstance(counts, torch.Tensor) and counts.device == img.device and counts.dtype == torch.int32
                and tuple(counts.shape) == (B,)):
            raise error("klt_b200: step_batch() counts must be a (B,) int32 tensor on the frames' device")
        maxCorners = int(maxCorners)
        if maxCorners < 1:
            raise error("klt_b200: step_batch() needs maxCorners >= 1 (the output width is N + maxCorners)")
        pts, cnt = points.contiguous(), counts.contiguous()
        N = pts.shape[1]
        nxt = DevicePyramid(img, self.winSize, self.maxLevel, ctx=self.prev.ctx, copy=True, prefilter=self.prefilter,
                            equalize=self.equalize)
        dev = img.device
        out = torch.empty((B, N + maxCorners, 2), dtype=torch.float32, device=dev)
        keep = torch.empty((B, N), dtype=torch.bool, device=dev)
        next_counts = torch.empty((B,), dtype=torch.int32, device=dev)
        n_new = torch.empty((B,), dtype=torch.int32, device=dev)
        host_counts = np.zeros(B, np.int32)
        L = _lib.load()
        ws_bytes = int(L.klt_frame_step_ws_bytes(W, H, B, N))
        ws = torch.empty((ws_bytes + 256,), dtype=torch.uint8, device=dev)
        ws_ptr = (ws.data_ptr() + 255) // 256 * 256
        params = make_params(self.prev.win, self.criteria, self.flags, self.minEigThreshold)
        # detection runs on the next pyramid's level 0: the frame as given, or the pre-filtered / equalized frame, as in step
        args = (self.prev.ctx.handle, self.prev.images.data_ptr(), self.prev.buffer.data_ptr(), nxt.images.data_ptr(),
                nxt.buffer.data_ptr(), ctypes.byref(self.prev.layout), 0, 0, 1, B, pts.data_ptr() if N else None, cnt.data_ptr(), N,
                ctypes.byref(params), float(max_bidir_error), int(mask_radius), maxCorners, float(qualityLevel), float(minDistance),
                int(blockSize), out.data_ptr(), N + maxCorners, keep.data_ptr() if N else None, next_counts.data_ptr(), n_new.data_ptr())
        if second_pass == "reverse":
            flags = torch.zeros((1,), dtype=torch.int32, device=dev)
            rc = L.klt_frame_step_batch_fb_async(*args, None, None, None, flags.data_ptr(), ws_ptr, ws_bytes, None, None, None,
                                                 _stream_ptr(img))
            if rc == KLT_OK:
                host = torch.cat([next_counts, flags]).cpu().numpy()     # the one synchronisation
                host_counts[:] = host[:B]
                if host[B]:
                    rc = _lib.KLT_ERR_INVALID_ARG                          # a count outside [0, N], as klt_frame_step_batch
        else:
            rc = L.klt_frame_step_batch(*args, host_counts.ctypes.data, ws_ptr, ws_bytes, _stream_ptr(img))
        if rc != KLT_OK:
            _raise_status(rc, "klt_frame_step_batch")
        self.prev = nxt
        M = int(host_counts.max())
        return out[:, :M], next_counts, keep, n_new


TrackHistory = collections.namedtuple("TrackHistory", "counts frames points ids src")


# include/klt_b200.h: a larger distance thins as this one does on every image the step accepts
MAX_TRACK_DISTANCE = 131072.0


def check_min_track_distance(d):
    """None, or a finite float in (0, MAX_TRACK_DISTANCE] -> the value as a float; anything else raises `error`."""
    if d is None:
        return None
    if isinstance(d, bool) or not isinstance(d, numbers.Real):
        raise error("klt_b200: min_track_distance must be None or a number")
    d = float(d)
    if not (0.0 < d <= MAX_TRACK_DISTANCE):
        raise error("klt_b200: min_track_distance must be finite and in (0, %g], got %r" % (MAX_TRACK_DISTANCE, d))
    return d


def check_detect_grid(grid, per_cell):
    """detect_grid (cols, rows) and tracks_per_cell, both None or both given -> None or ((cols, rows), q) as ints; the
    frame size is checked by the caller.  Anything else raises `error`."""
    if grid is None and per_cell is None:
        return None
    if grid is None or per_cell is None:
        raise error("klt_b200: detect_grid and tracks_per_cell go together")

    def whole(v):
        return isinstance(v, numbers.Integral) and not isinstance(v, bool)
    if not (isinstance(grid, (tuple, list)) and len(grid) == 2 and all(whole(v) for v in grid)):
        raise error("klt_b200: detect_grid must be a pair of ints (cols, rows)")
    cols, rows = int(grid[0]), int(grid[1])
    if cols < 1 or rows < 1 or cols * rows > _lib.KLT_MAX_GRID_CELLS:
        raise error("klt_b200: detect_grid needs cols, rows >= 1 and cols * rows <= %d, got %r" % (_lib.KLT_MAX_GRID_CELLS, (cols, rows)))
    if not whole(per_cell) or int(per_cell) < 1:
        raise error("klt_b200: tracks_per_cell must be an int >= 1, got %r" % (per_cell,))
    return (cols, rows), int(per_cell)


def history_rows(frames, depth):
    """Which ring rows history() returns: frames (B,), each sequence's current frame, and the ring depth R ->
    (frames (T, B) int32, rows (T, B) int64) with T = min(R, max(frames) + 1), frames[t, b] = frames[b] - T + 1 + t (oldest
    first) and rows = frames mod R.  A sequence that started over has fewer valid rows than T: its negative frames."""
    import numpy as np
    f = np.asarray(frames, np.int64).reshape(-1)
    T = min(int(depth), int(f.max()) + 1)
    fr = f[None, :] - T + 1 + np.arange(T)[:, None]
    return fr.astype(np.int32), fr % int(depth)


def history_from_ring(ring, frames):
    """A whole ring (TrackHistory of numpy arrays shaped (R, B, ...)) and each sequence's current frame -> history():
    per sequence its own last rows (history_rows), count 0 in the rows of a negative frame."""
    import numpy as np
    counts, _, points, ids, src = (np.asarray(a) for a in ring)
    fr, rows = history_rows(frames, counts.shape[0])
    b = np.arange(counts.shape[1])[None, :]
    return TrackHistory(np.where(fr >= 0, counts[rows, b], 0).astype(np.int32), fr, points[rows, b], ids[rows, b], src[rows, b])


def tracks_from_history(hist):
    """KLTSequenceBatch.history() (or a TrackHistory of numpy arrays shaped like it) -> per sequence, a dict
    id -> (frames (n,) int32, points (n, 2) float32) of every track with a position in those frames, oldest first."""
    import numpy as np
    counts, frames, points, ids = (np.asarray(a) for a in hist[:4])
    T_, B = counts.shape
    out = []
    for b in range(B):
        n = [int(counts[t, b]) for t in range(T_)]
        tid = np.concatenate([ids[t, b, :n[t]] for t in range(T_)] + [np.zeros(0, np.int32)]).astype(np.int32)
        tfr = np.concatenate([np.full(n[t], frames[t, b], np.int32) for t in range(T_)] + [np.zeros(0, np.int32)])
        tpt = np.concatenate([points[t, b, :n[t]].reshape(-1, 2) for t in range(T_)] + [np.zeros((0, 2), np.float32)]).astype(np.float32)
        order = np.argsort(tid, kind="stable")       # rows are oldest first, so each track's frames stay in order
        uid, start = np.unique(tid[order], return_index=True)
        end = list(start[1:]) + [len(order)]
        out.append({int(u): (tfr[order[s:e]], tpt[order[s:e]]) for u, s, e in zip(uid, start, end)})
    return out


class KLTSequenceBatch:
    """B sequences stepped frame after frame on the device with no host synchronisation between frames
    (klt_frame_step_batch_async), eagerly or replayed from CUDA graphs.

    The same step as KLTTracker.step_batch, with a fixed capacity C per sequence: sequence b keeps its survivors and
    takes at most min(maxCorners, C - survivors_b) new corners, i.e. the first ones cv2.goodFeaturesToTrack(...,
    maxCorners=min(maxCorners, C - survivors_b)) returns (none when that is 0).  Every point carries a track id: a survivor
    keeps its id, and the new corners of sequence b get consecutive ids from a per-sequence counter, strongest first.

    frames0: (B, H, W) uint8 CUDA, the first frame of each sequence.  points: (B, N, 2) float32 and counts: (B,) int32 on
    the same device, N <= capacity: sequence b starts with points[b, :counts[b]].  ids: optional (B, N) int32 ids of those
    points (default 0 .. counts[b] - 1); the id counter of sequence b starts after the largest of them.  prefilter:
    (d, sigmaColor, sigmaSpace), the loader's bilateral filter applied to every frame on the device, as in KLTTracker.

    Everything is allocated here: two pyramid slots with their own level-0 storage (the current frame and the next one),
    two point / id rows of width C per sequence, counts, id counters, keep flags, new-corner counts, a flag word, the
    workspace, a frame staging tensor and a private CUDA stream.  The initial counts are checked on the host here, the
    only time counts come from outside; after that the step writes them itself, within [0, C].  The caller's current
    stream waits for each step (on the device), so the properties can be read on it as soon as step() returns.

    history=R >= 1 also keeps per-track records on the device (klt_track_records_step, one more launch per step, in the
    graphs too): frames0 is frame 0 and each step advances `frame` by one.  Each slot carries `first_points` / `first_frames`,
    where and in which frame its track was first seen (the initial points: frame 0 and their position, unless
    first_points (B, N, 2) float32 and first_frames (B, N) int32 are given, together; a new corner: its own position and
    the frame it was born in).  A ring of the last R frames keeps, per sequence, every row's positions, ids and the slot
    each track had in the frame before (`src`, -1 when born there); window(k) reads the last k positions of every slot
    from it on the device, history() downloads it.  history=0 allocates and launches nothing of this.

    control=True lets a back end steer the batch between steps (klt_frame_step_batch_control_async, the same launches):
    drop(mask) ends chosen tracks at the next step, restart(seqs, ...) starts chosen sequences over at the next step, and
    `restarted` tells which did.  Both requests are written on the device in stream order, so they may be computed
    there and need no host synchronisation, eagerly or between graph replays.  control=False allocates and launches
    nothing of this.

    motion_prior starts each track's forward LK pass at a predicted position instead of where the track is
    (klt_track_predict, one more launch per step before the new frame's pyramid, then klt_frame_step_batch_init_async;
    in the graphs too).  Per sequence and slot j < counts[b], the start is: the position a back end gave with
    predict(points, mask) since the last step; else, with "velocity", p + (p - q) for a track with a position q in its
    sequence's previous frame (p its current position, float32 like numpy); else p, which changes nothing.  Per frame this
    is cv2.calcOpticalFlowPyrLK(im0, im1, p0, starts, flags=cv2.OPTFLOW_USE_INITIAL_FLOW) in the forward pass; the second
    pass, the filter and the detection are unchanged.  None (the default) allocates and launches nothing of this; "given"
    enables predict() alone; "velocity" also needs history >= 2.

    second_pass="reverse" replaces the reference's second LK pass (same frame pair, started from the forward result) by
    the forward-backward check (klt_frame_step_batch_fb_async, the same launches): p1 is tracked from the new frame back
    into the old one, p0r = cv2.calcOpticalFlowPyrLK(im1, im0, p1, None), and d = max |p0 - p0r| is the tracking error
    of a correct track rather than about twice the frame's motion, so a useful max_bidir_error is about 1 px.  With a
    motion_prior the reverse pass starts at the mirrored start p1 - (s - p0), s the forward pass's start, with
    OPTFLOW_USE_INITIAL_FLOW.  `bidir_error` holds each step's d.  "reference" (the default) is the reference's pass.

    min_track_distance=d (a float > 0) keeps the tracks apart (klt_frame_step_batch_thin_async, the same launches): at
    every step the survivors of the filter that are not dropped are visited in slot order, and one that lies closer than
    d to an earlier one that was kept is thinned: dx * dx + dy * dy < d * d in float64 on the float32 positions, each
    operation rounded once, as numpy float64 computes it.  A thinned track ends like a dropped one: keep False, no place in
    the output row or the detection mask, no record.  Slot order is birth order, because every row the step writes holds
    its survivors in input order, then the new corners strongest first; so the older track wins, and within one birth
    frame the stronger corner.  For the initial points and the staged points of a restart it is the order the caller
    gives them in, and a sequence restarted at a step thins nothing at that step.  `thinned` marks each step's thinned
    slots.  None (the default) allocates nothing and calls the entry points it calls without the option.

    detect_grid=(cols, rows) with tracks_per_cell=q (always together) tops up each cell of a cols x rows grid instead of
    detecting on the whole frame (klt_frame_step_batch_grid_async): with the global rule the strongest corners come first,
    so where contrast is uneven every new track goes to the textured part of the image.  Column edges are
    X_i = floor(i * W / cols), row edges Y_j = floor(j * H / rows); s_k counts the points of the row before detection (the
    kept survivors, or a restarted sequence's staged points) in cell k (a point counts in the last column / row whose edge
    is at or below it, clamped to the grid; NaN nowhere), and cell k gets cv2.goodFeaturesToTrack(frame, maxCorners =
    max(0, q - s_k), qualityLevel, minDistance, mask = M & cell, blockSize), M the usual mask around the survivors: the
    cell's own quality threshold, minDistance within the cell.  The new corners follow the survivors interleaved by rank
    (the strongest of every cell, then the second of every cell, ...) and are cut to min(maxCorners, C - survivors), so
    ids, records and the slot order within one birth frame are rank, then cell.  detect_grid=(1, 1) with
    tracks_per_cell=C is the step without the option.  Works with every other option, eagerly and from the graphs.
    cols <= W, rows <= H, cols * rows <= 1024.  None (the default) allocates and launches nothing of this.

    subpix=(winSize, zeroZone, criteria), e.g. ((5, 5), (-1, -1), (3, 40, 0.001)), refines each step's new corners to
    sub-pixel positions (klt_corner_sub_pix, one more launch per step after the frame step and before the records; in the
    graphs too): per sequence, the new corners of the row (the n_new slots behind the survivors, or behind a restart's
    staged points) are replaced by cv2.cornerSubPix(frame, new, winSize, zeroZone, criteria) on the frame detection ran
    on (pre-filtered when prefilter is set), bit for bit as OpenCV's own code computes it (without IPP).  Ids, records and
    first_points then hold the refined positions, and the next step starts from them: its LK pass, velocity prior,
    thinning, detection mask and grid cell counts (a corner moves by at most winSize from its pixel).  Survivors and
    staged points are never touched.  The window is checked against the frame size here (W >= 2 wx + 5, H >= 2 wy + 5,
    wx, wy <= 15).  None (the default) allocates and launches nothing of this.

    equalize=(clipLimit, tileGridSize), e.g. (3.0, (8, 8)), equalizes every frame the object takes (frames0 and every
    step's) on the device before its pyramid is built: level 0 of the frame's slot is createCLAHE(clipLimit,
    tileGridSize).apply(frame), or of the bilateral output when prefilter is set (equalized in place there), bit for bit
    as cv2 computes it (klt_clahe, two launches per step before the pyramid build; in the graphs too).  LK, detection, the
    mask, the grid cell counts and subpix all run on the equalized frame.  A change of exposure between two frames then
    mostly cancels out, where LK's brightness constancy would otherwise fail.  Checked against the frame size here, as
    klt_clahe checks it.  None (the default) allocates and launches nothing of this."""

    def __init__(self, frames0, points, counts, capacity, ids=None, winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03),
                 max_bidir_error=30, mask_radius=10, maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31,
                 prefilter=None, history=0, first_points=None, first_frames=None, control=False, motion_prior=None,
                 second_pass="reference", min_track_distance=None, detect_grid=None, tracks_per_cell=None, subpix=None,
                 equalize=None):
        torch = _torch()
        self.second_pass = check_second_pass(second_pass)
        self.min_track_distance = check_min_track_distance(min_track_distance)
        grid = check_detect_grid(detect_grid, tracks_per_cell)
        img = _as_image_batch(frames0)
        B, H, W = img.shape
        if grid is not None and (grid[0][0] > W or grid[0][1] > H):
            raise error("klt_b200: detect_grid %r does not fit %d x %d frames (cols <= W, rows <= H)" % (grid[0], W, H))
        self.detect_grid, self.tracks_per_cell = (None, None) if grid is None else grid
        if subpix is not None:
            from .corners import check_subpix
            if not (isinstance(subpix, (tuple, list)) and len(subpix) == 3):
                raise error("klt_b200: KLTSequenceBatch subpix must be None or (winSize, zeroZone, criteria)")
            subpix = check_subpix(*subpix, W, H, func="KLTSequenceBatch subpix")
        self.subpix = subpix
        self.equalize = check_equalize(equalize, W, H, "KLTSequenceBatch equalize")
        dev = img.device
        C = int(capacity)
        if C < 1:
            raise error("klt_b200: KLTSequenceBatch needs capacity >= 1")
        if not (isinstance(points, torch.Tensor) and points.device == dev and points.dtype == torch.float32
                and points.dim() == 3 and points.shape[0] == B and points.shape[2] == 2 and points.shape[1] <= C):
            raise error("klt_b200: KLTSequenceBatch points must be a (B, N, 2) float32 tensor on the frames' device, N <= capacity")
        if not (isinstance(counts, torch.Tensor) and counts.device == dev and counts.dtype == torch.int32
                and tuple(counts.shape) == (B,)):
            raise error("klt_b200: KLTSequenceBatch counts must be a (B,) int32 tensor on the frames' device")
        N = points.shape[1]
        host_counts = counts.cpu()
        if bool(((host_counts < 0) | (host_counts > N)).any()):
            raise error("klt_b200: KLTSequenceBatch counts must lie in [0, %d]" % N)
        if ids is not None and not (isinstance(ids, torch.Tensor) and ids.device == dev and ids.dtype == torch.int32
                                    and tuple(ids.shape) == (B, N)):
            raise error("klt_b200: KLTSequenceBatch ids must be a (B, N) int32 tensor on the frames' device")
        self.maxCorners = int(maxCorners)
        if self.maxCorners < 1:
            raise error("klt_b200: KLTSequenceBatch needs maxCorners >= 1")
        R = int(history)
        if R < 0:
            raise error("klt_b200: KLTSequenceBatch needs history >= 0")
        if (first_points is None) != (first_frames is None):
            raise error("klt_b200: KLTSequenceBatch first_points and first_frames go together")
        if first_points is not None:
            if R < 1:
                raise error("klt_b200: KLTSequenceBatch first_points / first_frames need history >= 1")
            if not (isinstance(first_points, torch.Tensor) and first_points.device == dev and first_points.dtype == torch.float32
                    and tuple(first_points.shape) == tuple(points.shape)):
                raise error("klt_b200: KLTSequenceBatch first_points must be a float32 tensor shaped like points on the frames' device")
            if not (isinstance(first_frames, torch.Tensor) and first_frames.device == dev and first_frames.dtype == torch.int32
                    and tuple(first_frames.shape) == (B, N)):
                raise error("klt_b200: KLTSequenceBatch first_frames must be a (B, N) int32 tensor on the frames' device")
        self.depth = R
        if motion_prior not in (None, "given", "velocity"):
            raise error("klt_b200: KLTSequenceBatch motion_prior must be None, 'given' or 'velocity'")
        if motion_prior == "velocity" and R < 2:
            raise error("klt_b200: KLTSequenceBatch motion_prior='velocity' needs history >= 2")
        self.motion_prior = motion_prior
        win_w, win_h, _ = _check_win_level(winSize, maxLevel)
        self.capacity, self.prefilter = C, prefilter
        self.max_bidir_error, self.mask_radius = float(max_bidir_error), int(mask_radius)
        self.qualityLevel, self.minDistance, self.blockSize = float(qualityLevel), float(minDistance), int(blockSize)
        self.params = make_params((win_w, win_h), criteria, 0, 1e-4)
        self.ctx = _lib.default_context(dev.index or 0)
        self.stream = torch.cuda.Stream(device=dev)
        self.stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self.stream):
            self._slots = [DevicePyramid(alloc_image_batch(B, H, W, device=dev), winSize, maxLevel, ctx=self.ctx) for _ in range(2)]
            self._stage = alloc_image_batch(B, H, W, device=dev)
            if self.equalize is not None:
                tiles = self.equalize[1]
                self._clahe_ws = torch.empty((int(_lib.load().klt_clahe_ws_bytes(B, *tiles)),), dtype=torch.uint8, device=dev)
            self._fill(self._slots[0], img)
            self._pts = torch.zeros((2, B, C, 2), dtype=torch.float32, device=dev)
            self._ids = torch.zeros((2, B, C), dtype=torch.int32, device=dev)
            self._counts = torch.zeros((2, B), dtype=torch.int32, device=dev)
            self._pts[0, :, :N] = points
            self._counts[0] = counts
            if ids is None:
                ids = torch.arange(N, dtype=torch.int32, device=dev).expand(B, N)
            self._ids[0, :, :N] = ids
            valid = torch.arange(N, device=dev)[None, :] < counts[:, None].long()
            lo = torch.iinfo(torch.int32).min
            self._next_id = (torch.where(valid, ids, torch.full_like(ids, lo)).max(1).values.clamp_min(-1) + 1).int() if N else \
                torch.zeros((B,), dtype=torch.int32, device=dev)
            self._keep = torch.zeros((B, C), dtype=torch.uint8, device=dev)
            self._n_new = torch.zeros((B,), dtype=torch.int32, device=dev)
            self._flags = torch.zeros((1,), dtype=torch.int32, device=dev)
            self._ws_bytes = int(_lib.load().klt_frame_step_ws_bytes(W, H, B, C)) if grid is None else \
                int(_lib.load().klt_frame_step_grid_ws_bytes(W, H, B, C, *grid[0]))
            self._ws = torch.empty((self._ws_bytes + 256,), dtype=torch.uint8, device=dev)
            if R:
                # per-slot state, ping-ponged with the point rows; the ring (layout: include/klt_b200.h) holds frame 0
                self._first_pts = torch.zeros((2, B, C, 2), dtype=torch.float32, device=dev)
                self._first_frames = torch.zeros((2, B, C), dtype=torch.int32, device=dev)
                self._first_pts[0, :, :N] = points if first_points is None else first_points
                if first_frames is not None:
                    self._first_frames[0, :, :N] = first_frames
                self._frame = torch.zeros((B,), dtype=torch.int32, device=dev)
                self._ring_pts = torch.zeros((R, B, C, 2), dtype=torch.float32, device=dev)
                self._ring_ids = torch.zeros((R, B, C), dtype=torch.int32, device=dev)
                self._ring_src = torch.full((R, B, C), -1, dtype=torch.int32, device=dev)
                self._ring_counts = torch.zeros((R, B), dtype=torch.int32, device=dev)
                self._ring_frames = torch.zeros((R, B), dtype=torch.int32, device=dev)
                self._ring_pts[0, :, :N] = points
                self._ring_ids[0, :, :N] = ids
                self._ring_counts[0] = counts
            self.control = bool(control)
            if self.control:
                # pending drops and restarts (cleared by the step), the staged rows of a restart, and the step's `restarted`
                self._drop = torch.zeros((B, C), dtype=torch.uint8, device=dev)
                self._rs_flag = torch.zeros((B,), dtype=torch.uint8, device=dev)
                self._rs_pts = torch.zeros((B, C, 2), dtype=torch.float32, device=dev)
                self._rs_counts = torch.zeros((B,), dtype=torch.int32, device=dev)
                self._rs_ids = torch.zeros((B, C), dtype=torch.int32, device=dev)
                self._rs_next_id = torch.zeros((B,), dtype=torch.int32, device=dev)
                self._restarted = torch.zeros((B,), dtype=torch.uint8, device=dev)
                if R:
                    self._rs_first_pts = torch.zeros((B, C, 2), dtype=torch.float32, device=dev)
                    self._rs_first_frames = torch.zeros((B, C), dtype=torch.int32, device=dev)
                self._ctl = _lib.klt_step_control(self._drop.data_ptr(), self._rs_flag.data_ptr(), self._rs_pts.data_ptr(),
                                                  self._rs_counts.data_ptr(), self._rs_ids.data_ptr(), self._rs_next_id.data_ptr(),
                                                  self._restarted.data_ptr())
            if motion_prior is not None:
                # positions given by predict() (pending until the step clears the mask), and the forward pass's starts
                self._guess_pts = torch.zeros((B, C, 2), dtype=torch.float32, device=dev)
                self._guess_mask = torch.zeros((B, C), dtype=torch.uint8, device=dev)
                self._init = torch.zeros((B, C, 2), dtype=torch.float32, device=dev)
            if self.second_pass == "reverse":
                self._bidir = torch.full((B, C), float("nan"), dtype=torch.float32, device=dev)
            if self.min_track_distance is not None:
                self._thinned = torch.zeros((B, C), dtype=torch.uint8, device=dev)
        torch.cuda.current_stream(dev).wait_stream(self.stream)
        self._ws_ptr = (self._ws.data_ptr() + 255) // 256 * 256
        self._cur = 0          # slot / row of the current frame
        self._frame_host = 0
        self._eager_steps = 0
        self._graphs = None

    def _fill(self, slot, frames):
        """frames -> the slot's level 0 (bilateral-filtered when prefilter is set, then equalized in place when equalize is
        set), then its pyramid; current stream."""
        if self.prefilter is not None:
            from .filters import bilateral_filter
            bilateral_filter(frames, *self.prefilter, out=slot.images, ctx=self.ctx)
        else:
            slot.images.copy_(frames)
        if self.equalize is not None:
            from .filters import clahe_launch
            clahe_launch(slot.images, slot.images, *self.equalize, self._clahe_ws, self.ctx, _stream_ptr(slot.images))
        slot.build()

    def _enqueue(self, cur, frames):
        """The step from slot / row `cur` to the other one, on the current stream (self.stream)."""
        nxt = 1 - cur
        prev, new = self._slots[cur], self._slots[nxt]
        B, C = self._pts.shape[1], self.capacity
        L = _lib.load()
        if self.motion_prior is not None:
            # reads only the previous step's state, so it goes before the pyramid build, off the path to the forward pass
            vel = self.motion_prior == "velocity"
            rc = L.klt_track_predict(self.ctx.handle, B, C, self._pts[cur].data_ptr(), self._counts[cur].data_ptr(),
                                     self._guess_pts.data_ptr(), self._guess_mask.data_ptr(), self.depth if vel else 0,
                                     self._ring_pts.data_ptr() if vel else None, self._ring_src.data_ptr() if vel else None,
                                     self._ring_counts.data_ptr() if vel else None, self._frame.data_ptr() if vel else None,
                                     self._init.data_ptr(), ctypes.c_void_p(self.stream.cuda_stream))
            if rc != KLT_OK:
                _raise_status(rc, "klt_track_predict")
        self._fill(new, frames)
        args = (self.ctx.handle, prev.images.data_ptr(), prev.buffer.data_ptr(), new.images.data_ptr(), new.buffer.data_ptr(),
                ctypes.byref(prev.layout), 0, 0, 1, B, self._pts[cur].data_ptr(), self._counts[cur].data_ptr(), C, ctypes.byref(self.params),
                self.max_bidir_error, self.mask_radius, self.maxCorners, self.qualityLevel, self.minDistance, self.blockSize,
                self._pts[nxt].data_ptr(), C, self._keep.data_ptr(), self._counts[nxt].data_ptr(), self._n_new.data_ptr(),
                self._ids[cur].data_ptr(), self._ids[nxt].data_ptr(), self._next_id.data_ptr(), self._flags.data_ptr(), self._ws_ptr,
                self._ws_bytes)
        if self.detect_grid is not None:
            thin = self.min_track_distance is not None
            rc = L.klt_frame_step_batch_grid_async(*args, self._init.data_ptr() if self.motion_prior is not None else None,
                                                   ctypes.byref(self._ctl) if self.control else None,
                                                   self._bidir.data_ptr() if self.second_pass == "reverse" else None,
                                                   int(self.second_pass == "reverse"), self.min_track_distance if thin else 0.0,
                                                   self._thinned.data_ptr() if thin else None, self.detect_grid[0], self.detect_grid[1],
                                                   self.tracks_per_cell, ctypes.c_void_p(self.stream.cuda_stream))
        elif self.min_track_distance is not None:
            rc = L.klt_frame_step_batch_thin_async(*args, self._init.data_ptr() if self.motion_prior is not None else None,
                                                   ctypes.byref(self._ctl) if self.control else None,
                                                   self._bidir.data_ptr() if self.second_pass == "reverse" else None,
                                                   int(self.second_pass == "reverse"), self.min_track_distance,
                                                   self._thinned.data_ptr(), ctypes.c_void_p(self.stream.cuda_stream))
        elif self.second_pass == "reverse":
            rc = L.klt_frame_step_batch_fb_async(*args, self._init.data_ptr() if self.motion_prior is not None else None,
                                                 ctypes.byref(self._ctl) if self.control else None, self._bidir.data_ptr(),
                                                 ctypes.c_void_p(self.stream.cuda_stream))
        elif self.motion_prior is not None:
            rc = L.klt_frame_step_batch_init_async(*args, self._init.data_ptr(), ctypes.byref(self._ctl) if self.control else None,
                                                   ctypes.c_void_p(self.stream.cuda_stream))
        elif self.control:
            rc = L.klt_frame_step_batch_control_async(*args, ctypes.byref(self._ctl), ctypes.c_void_p(self.stream.cuda_stream))
        else:
            rc = L.klt_frame_step_batch_async(*args, ctypes.c_void_p(self.stream.cuda_stream))
        if rc != KLT_OK:
            _raise_status(rc, "klt_frame_step_batch_async")
        if self.subpix is not None:
            # the new corners are the slots [next_counts - n_new, next_counts) of each row, refined on the frame detection saw
            img = new.images
            rc = L.klt_corner_sub_pix(self.ctx.handle, img.data_ptr(), img.shape[2], img.shape[1], img.stride(1), _batch_stride(img), B,
                                      self._pts[nxt].data_ptr(), C, self._counts[nxt].data_ptr(), self._n_new.data_ptr(), *self.subpix,
                                      ctypes.c_void_p(self.stream.cuda_stream))
            if rc != KLT_OK:
                _raise_status(rc, "klt_corner_sub_pix")
        if self.depth:
            args = (self.ctx.handle, B, C, C, self._keep.data_ptr(), self._pts[nxt].data_ptr(), self._ids[nxt].data_ptr(),
                    self._counts[nxt].data_ptr(), self._first_pts[cur].data_ptr(), self._first_frames[cur].data_ptr(),
                    self._first_pts[nxt].data_ptr(), self._first_frames[nxt].data_ptr(), self._frame.data_ptr(), self.depth,
                    self._ring_pts.data_ptr(), self._ring_ids.data_ptr(), self._ring_src.data_ptr(), self._ring_counts.data_ptr(),
                    self._ring_frames.data_ptr())
            if self.control:
                rc = L.klt_track_records_step_control(*args, self._restarted.data_ptr(), self._rs_counts.data_ptr(),
                                                      self._rs_first_pts.data_ptr(), self._rs_first_frames.data_ptr(),
                                                      ctypes.c_void_p(self.stream.cuda_stream))
            else:
                rc = L.klt_track_records_step(*args, ctypes.c_void_p(self.stream.cuda_stream))
            if rc != KLT_OK:
                _raise_status(rc, "klt_track_records_step")

    def step(self, frames):
        """Enqueue one frame for every sequence: frames (B, H, W) uint8 CUDA.  Does not synchronise."""
        torch = _torch()
        img = _as_image_batch(frames)
        slot = self._slots[self._cur]
        if tuple(img.shape) != tuple(slot.images.shape) or img.device != slot.images.device:
            raise error("klt_b200: KLTSequenceBatch.step() takes (B, H, W) frames of the batch's size and device")
        caller = torch.cuda.current_stream(img.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            if self._graphs is None:
                self._enqueue(self._cur, img)
                self._eager_steps += 1
            else:
                self._stage.copy_(img)
                self._graphs[self._cur].replay()
        caller.wait_stream(self.stream)
        self._cur = 1 - self._cur
        self._frame_host += 1
        return self

    def capture(self):
        """Record the step into two CUDA graphs, one per parity of the slots, on the object's stream; later step() calls
        copy the frames into the staging tensor and replay the graph of the current parity.  Needs one eager step()
        first (it sets up the per-device kernel attributes and the pyramid build's scratch of this stream)."""
        torch = _torch()
        if self._eager_steps < 1:
            raise error("klt_b200: KLTSequenceBatch.capture() needs one eager step() first")
        if self._graphs is not None:
            return self
        graphs = []
        for cur in (0, 1):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.stream):
                self._enqueue(cur, self._stage)
            graphs.append(g)
        self._graphs = graphs
        return self

    @property
    def points(self):
        """(B, C, 2) float32: sequence b's points are points[b, :counts[b]] (survivors in input order, then new corners)."""
        return self._pts[self._cur]

    @property
    def counts(self):
        return self._counts[self._cur]

    @property
    def ids(self):
        """(B, C) int32 track ids of `points`."""
        return self._ids[self._cur]

    @property
    def keep(self):
        """(B, C) bool: which of the previous frame's points survived the last step (False behind its count)."""
        return self._keep.view(_torch().bool)

    @property
    def n_new(self):
        return self._n_new

    @property
    def bidir_error(self):
        """(B, C) float32: the last step's forward-backward error d of each of the previous frame's points, aligned with
        `keep`; NaN behind its count, for a sequence restarted at that step, and before the first step.  Needs
        second_pass="reverse"."""
        if self.second_pass != "reverse":
            raise error("klt_b200: KLTSequenceBatch.bidir_error needs second_pass='reverse'")
        return self._bidir

    @property
    def thinned(self):
        """(B, C) uint8: 1 where the last step thinned one of the previous frame's points (aligned with `keep`); 0 elsewhere,
        behind its count, for a sequence restarted at that step, and before the first step.  Needs min_track_distance."""
        if self.min_track_distance is None:
            raise error("klt_b200: KLTSequenceBatch.thinned needs min_track_distance")
        return self._thinned

    def _need_history(self, what):
        if not self.depth:
            raise error("klt_b200: KLTSequenceBatch.%s needs history >= 1" % what)

    @property
    def frame(self):
        """Number of steps since construction (frames0 is frame 0)."""
        return self._frame_host

    @property
    def frames(self):
        """(B,) int32 CUDA: each sequence's own current frame index (0 at construction and at a restart)."""
        self._need_history("frames")
        return self._frame

    @property
    def first_points(self):
        """(B, C, 2) float32: where the track in each slot was first seen (valid for slots [0, counts[b]))."""
        self._need_history("first_points")
        return self._first_pts[self._cur]

    @property
    def first_frames(self):
        """(B, C) int32: the frame in which the track in each slot was first seen."""
        self._need_history("first_frames")
        return self._first_frames[self._cur]

    @property
    def lengths(self):
        """(B, C) int32: frames the track in each slot has a position in, frame - first_frames + 1."""
        self._need_history("lengths")
        return self._frame[:, None] - self._first_frames[self._cur] + 1

    def window(self, k):
        """(B, C, k, 2) float32 CUDA, 1 <= k <= history: [b, j, k - 1 - d] is slot j's position d frames ago (the track's
        last k positions), NaN before the track was born, before frame 0 and for j >= counts[b].  Computed on the device
        (klt_track_window) on the object's stream; no synchronisation."""
        torch = _torch()
        self._need_history("window()")
        k = int(k)
        if not 1 <= k <= self.depth:
            raise error("klt_b200: KLTSequenceBatch.window(k) needs 1 <= k <= history (%d)" % self.depth)
        B, C = self._pts.shape[1], self.capacity
        out = torch.empty((B, C, k, 2), dtype=torch.float32, device=self._pts.device)
        caller = torch.cuda.current_stream(out.device)
        self.stream.wait_stream(caller)
        rc = _lib.load().klt_track_window(self.ctx.handle, B, C, self.depth, self._ring_pts.data_ptr(), self._ring_src.data_ptr(),
                                          self._ring_counts.data_ptr(), self._frame.data_ptr(), k, out.data_ptr(),
                                          ctypes.c_void_p(self.stream.cuda_stream))
        if rc != KLT_OK:
            _raise_status(rc, "klt_track_window")
        caller.wait_stream(self.stream)
        return out

    def history(self):
        """Synchronise and download the ring's valid rows, oldest first, as numpy: TrackHistory(counts (T, B) int32, frames
        (T, B) int32, points (T, B, C, 2) float32, ids (T, B, C) int32, src (T, B, C) int32).  Sequence b contributes its own
        last min(history, frames[b] + 1) frames: T = min(history, max(frames) + 1), frames[t, b] = frames[b] - T + 1 + t,
        count 0 where that is negative (a sequence restarted fewer than T - 1 frames ago).  Entries behind counts[t, b] are
        undefined.  tracks_from_history() groups them by track."""
        self._need_history("history()")
        self.stream.synchronize()
        ring = TrackHistory(*(t.cpu().numpy() for t in (self._ring_counts, self._ring_frames, self._ring_pts, self._ring_ids,
                                                        self._ring_src)))
        return history_from_ring(ring, self._frame.cpu().numpy())

    def _need_control(self, what):
        if not self.control:
            raise error("klt_b200: KLTSequenceBatch.%s needs control=True" % what)

    @property
    def restarted(self):
        """(B,) bool: which sequences started over at the current frame (written by every step)."""
        self._need_control("restarted")
        return self._restarted.view(_torch().bool)

    def _cuda_arg(self, name, t, dtype, shape):
        torch = _torch()
        if not (isinstance(t, torch.Tensor) and t.device == self._pts.device and t.dtype == dtype and tuple(t.shape) == tuple(shape)):
            raise error("klt_b200: KLTSequenceBatch: %s must be a %s %s tensor on the batch's device" % (name, tuple(shape), dtype))

    def drop(self, mask):
        """End the tracks marked in mask ((B, C) bool CUDA, aligned with `points` / `ids`) at the next step: they do not
        survive it (keep False), enter no detection mask and get no ring entry.  Slots at or behind counts[b] are ignored;
        calls before one step add up.  Enqueued on the object's stream after the caller's stream; no synchronisation."""
        torch = _torch()
        self._need_control("drop()")
        B, C = self._pts.shape[1], self.capacity
        self._cuda_arg("drop() mask", mask, torch.bool, (B, C))
        caller = torch.cuda.current_stream(mask.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            self._drop.bitwise_or_(mask.view(torch.uint8))
        caller.wait_stream(self.stream)
        return self

    def restart(self, seqs, points=None, counts=None, ids=None, first_points=None, first_frames=None):
        """Start the sequences marked in seqs ((B,) bool CUDA) over at the next step, whose frame becomes their frame 0:
        no old point survives, the row starts with points[b, :counts[b]] ((B, N, 2) float32, N <= C; counts (B,) int32,
        default N; no points: none), then the step's new corners.  ids (B, N) int32: their ids, the id counter restarts after
        the largest (as in the constructor); without ids they and the new corners continue the sequence's counter.  With
        history >= 1 the sequence's frame becomes 0, and first_points (B, N, 2) float32 / first_frames (B, N) int32 (together;
        default: their position and 0) are the points' first observations.  For each sequence the last call before a step
        wins, and a restart overrides drops of the same sequence.  A count outside [0, N] is clamped and flagged for
        check().  Enqueued on the object's stream after the caller's stream; no synchronisation."""
        torch = _torch()
        self._need_control("restart()")
        B, C = self._pts.shape[1], self.capacity
        dev = self._pts.device
        self._cuda_arg("restart() seqs", seqs, torch.bool, (B,))
        if points is None:
            if counts is not None or ids is not None or first_points is not None or first_frames is not None:
                raise error("klt_b200: KLTSequenceBatch.restart(): counts, ids, first_points and first_frames need points")
            N = 0
        else:
            if not (isinstance(points, torch.Tensor) and points.dim() == 3 and points.shape[0] == B and points.shape[1] <= C):
                raise error("klt_b200: KLTSequenceBatch.restart(): points must be a (B, N, 2) float32 tensor, N <= capacity")
            N = points.shape[1]
            self._cuda_arg("restart() points", points, torch.float32, (B, N, 2))
            if counts is not None:
                self._cuda_arg("restart() counts", counts, torch.int32, (B,))
            if ids is not None:
                self._cuda_arg("restart() ids", ids, torch.int32, (B, N))
            if (first_points is None) != (first_frames is None):
                raise error("klt_b200: KLTSequenceBatch.restart(): first_points and first_frames go together")
            if first_points is not None:
                self._need_history("restart(first_points=...)")
                self._cuda_arg("restart() first_points", first_points, torch.float32, (B, N, 2))
                self._cuda_arg("restart() first_frames", first_frames, torch.int32, (B, N))
        caller = torch.cuda.current_stream(dev)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            m1 = seqs
            m2, m3 = seqs[:, None], seqs[:, None, None]
            if N:
                cnt = counts if counts is not None else torch.full((B,), N, dtype=torch.int32, device=dev)
                self._flags.bitwise_or_((m1 & ((cnt < 0) | (cnt > N))).any().to(torch.int32))
                cnt = cnt.clamp(0, N)
                self._rs_pts[:, :N] = torch.where(m3, points, self._rs_pts[:, :N])
            else:
                cnt = torch.zeros((B,), dtype=torch.int32, device=dev)
            self._rs_counts.copy_(torch.where(m1, cnt, self._rs_counts))
            if ids is not None:
                valid = torch.arange(N, device=dev)[None, :] < cnt[:, None].long()
                lo = torch.iinfo(torch.int32).min
                nid = (torch.where(valid, ids, torch.full_like(ids, lo)).max(1).values.clamp_min(-1) + 1).int()
                self._rs_ids[:, :N] = torch.where(m2, ids, self._rs_ids[:, :N])
            else:
                self._rs_ids.copy_(torch.where(m2, self._next_id[:, None] + torch.arange(C, dtype=torch.int32, device=dev)[None, :],
                                               self._rs_ids))
                nid = self._next_id + cnt
            self._rs_next_id.copy_(torch.where(m1, nid, self._rs_next_id))
            if self.depth and N:
                fp = points if first_points is None else first_points
                ff = torch.zeros((B, N), dtype=torch.int32, device=dev) if first_frames is None else first_frames
                self._rs_first_pts[:, :N] = torch.where(m3, fp, self._rs_first_pts[:, :N])
                self._rs_first_frames[:, :N] = torch.where(m2, ff, self._rs_first_frames[:, :N])
            self._rs_flag.bitwise_or_(seqs.view(torch.uint8))
        caller.wait_stream(self.stream)
        return self

    def predict(self, points, mask):
        """Start the forward LK pass of the next step at points[b, j] ((B, C, 2) float32 CUDA, aligned with `points` /
        `ids`) for the slots marked in mask ((B, C) bool CUDA), as given: NaN, inf and positions outside the image too.
        With motion_prior="velocity" the marked slots override the velocity.  Slots at or behind counts[b] are ignored;
        for slots marked by several calls before one step, the last one wins; the step consumes the requests.  Needs a
        motion_prior.  Enqueued on the object's stream after the caller's stream; no synchronisation."""
        torch = _torch()
        if self.motion_prior is None:
            raise error("klt_b200: KLTSequenceBatch.predict() needs motion_prior='given' or 'velocity'")
        B, C = self._pts.shape[1], self.capacity
        self._cuda_arg("predict() points", points, torch.float32, (B, C, 2))
        self._cuda_arg("predict() mask", mask, torch.bool, (B, C))
        caller = torch.cuda.current_stream(mask.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            self._guess_pts.copy_(torch.where(mask[:, :, None], points, self._guess_pts))
            self._guess_mask.bitwise_or_(mask.view(torch.uint8))
        caller.wait_stream(self.stream)
        return self

    def check(self):
        """Synchronise and raise `error` if a step has seen a count outside [0, C] (clamped by the kernels); clears it."""
        self.stream.synchronize()
        if int(self._flags.item()):
            self._flags.zero_()
            raise error("klt_b200: KLTSequenceBatch: a point count outside [0, capacity] was clamped")
        return self
