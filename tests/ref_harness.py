"""Harness that runs the UNMODIFIED reference pipeline (src/pipeline/pipeline.py, src/extractor/extractor.py) on a
synthetic sequence, with `cv2.calcOpticalFlowPyrLK` either spied on (to record what the reference's own code passes
and receives at the boundary) or replaced by the B200 drop-in -- SURVEY.md s4 / s7 step 8, BASELINE configs[2].

TEST INFRASTRUCTURE.  Nothing here is product code; nothing here copies reference sources: the reference is imported
from the `src/` directory of a checkout of JonasFrey96/Visual-Odom-Pipeline named by the VO_REFERENCE_SRC environment
variable, and the tests that need it skip without it.  The repository keeps the recorded trace
(tests/golden/pipeline_trace.npz, made by tests/golden/make_pipeline_trace.py) and this file's deterministic frame
renderer, so that the other tests replay the reference's own call sequence without its sources.

Shims (no reference file is edited; all are attribute patches made from outside):
  * `matplotlib`, `matplotlib.pyplot`, `coloredlogs`: absent in this image -> stub modules in sys.modules
    (imports at extractor.py:6, visu.py:9, main.py:9);
  * `visu.Visualizer` -> no-op class (pipeline.py:30,38-39,166-167 only call update / render);
  * `cv2.waitKey` / `cv2.imshow`: headless OpenCV raises (pipeline.py:40) -> no-ops;
  * `cv2.circle`: OpenCV 4.13 rejects the 1-element-array coordinates of extractor.py:106-107 -> coercing wrapper;
  * `cv2.KeyPoint_convert`: rejects the (N, 1, 2) array of extractor.py:112 -> coercing wrapper.
"""
import os
import sys
import types
import zlib

import numpy as np

REFERENCE_SRC = os.environ.get("VO_REFERENCE_SRC", "")
REFERENCE_MISSING = "needs the original project's sources: set VO_REFERENCE_SRC to its src/ directory"


def reference_available():
    return bool(REFERENCE_SRC) and os.path.isdir(os.path.join(REFERENCE_SRC, "pipeline"))


# ------------------------------------------------------------------------------------------------------------------
# Deterministic synthetic sequence: a textured, slanted plane seen by a translating / slowly rotating pinhole camera.
# Pure numpy; the texture is integer arithmetic and the warp is float64 element-wise arithmetic followed by
# fixed-point bilinear sampling, so every machine renders the same bytes (checked against CRCs kept in the trace).
# ------------------------------------------------------------------------------------------------------------------
def _box_blur_int(a, r):
    """(2r+1)^2 box sum of an int64 image with wrap-around, via cumulative sums (exact)."""
    for ax in (0, 1):
        p = np.concatenate([a.take(range(-r - 1, 0), axis=ax), a, a.take(range(0, r), axis=ax)], axis=ax)
        c = np.cumsum(p, axis=ax, dtype=np.int64)
        n = a.shape[ax]
        hi = c.take(range(2 * r + 1, 2 * r + 1 + n), axis=ax)
        lo = c.take(range(0, n), axis=ax)
        a = hi - lo
    return a


def plane_texture(size=2048, seed=5):
    """uint8 (size, size) multi-scale texture (integer arithmetic only)."""
    rng = np.random.default_rng(seed)
    acc = np.zeros((size, size), np.int64)
    for r, amp in ((1, 3), (3, 4), (8, 5), (20, 4)):
        n = rng.integers(0, 256, (size, size), dtype=np.int64)
        b = _box_blur_int(_box_blur_int(n, r), r)                 # two passes: smoother than one box
        b = b - b.min()
        acc += amp * (b * 1024 // max(int(b.max()), 1))
    acc = acc - acc.min()
    return (acc * 255 // max(int(acc.max()), 1)).astype(np.uint8)


class SyntheticLoader:
    """Duck type of the reference's Loader as Pipeline uses it (pipeline.py:15,30,36,44-46,95,172):
    `_name`, `getCamera()`, `getInit()`, `getFrame(i)` -> (uint8 HxW, 4x4 pose), `getImage(i)`, `__len__`."""

    def __init__(self, h=480, w=640, n_frames=40, seed=5, init=(0, 3)):
        self._name = "synthetic_plane"
        self.h, self.w, self.n = int(h), int(w), int(n_frames)
        self._init = init
        f = 0.9 * w
        self.K = np.array([[f, 0, w / 2.0], [0, f, h / 2.0], [0, 0, 1]], np.float64)
        self._tex = plane_texture(2048, seed)
        self._cache = {}

    def __len__(self):
        return self.n

    def getCamera(self):
        return self.K.copy()

    def getInit(self):
        return self._init

    def pose(self, i):
        """world -> camera (4x4): the camera moves right and forward and yaws a little."""
        a = np.deg2rad(0.15 * i)
        R = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]], np.float64)
        c = np.array([0.06 * i, -0.01 * i, 0.03 * i], np.float64)       # camera centre in the world
        H = np.eye(4)
        H[:3, :3] = R
        H[:3, 3] = -R @ c
        return H

    def getImage(self, i):
        if not (0 <= i < self.n):
            raise AssertionError("frame id out of range")
        if i not in self._cache:
            self._cache[i] = self._render(i)
        return self._cache[i]

    def getFrame(self, i):
        return self.getImage(i), self.pose(i)

    def _render(self, i):
        # plane: points X = o + s*e1 + t*e2 (texture pixel (s, t) scaled by `mpp` metres per pixel), slanted about y
        mpp = 0.012
        th = np.deg2rad(25.0)
        e1 = np.array([np.cos(th), 0, np.sin(th)]) * mpp
        e2 = np.array([0, 1.0, 0]) * mpp
        o = np.array([-1024 * mpp * np.cos(th), -1024 * mpp, 9.0 - 1024 * mpp * np.sin(th)])
        H = self.pose(i)
        R, t = H[:3, :3], H[:3, 3]
        A = np.stack([e1, e2, o], axis=1)                 # texture (s, t, 1) -> world
        M = self.K @ (R @ A + np.outer(t, [0, 0, 1.0]))   # texture (s, t, 1) -> image (homogeneous)
        Mi = np.linalg.inv(M)
        ys, xs = np.mgrid[0:self.h, 0:self.w].astype(np.float64)
        d = Mi[2, 0] * xs + Mi[2, 1] * ys + Mi[2, 2]
        s = (Mi[0, 0] * xs + Mi[0, 1] * ys + Mi[0, 2]) / d
        tt = (Mi[1, 0] * xs + Mi[1, 1] * ys + Mi[1, 2]) / d
        # fixed-point bilinear (8 fractional bits) with wrap-around addressing
        sf = np.floor(s * 256.0).astype(np.int64)
        tf = np.floor(tt * 256.0).astype(np.int64)
        s0, fs = sf >> 8, sf & 255
        t0, ft = tf >> 8, tf & 255
        n = self._tex.shape[0]
        tex = self._tex.astype(np.int64)
        a = tex[t0 % n, s0 % n]
        b = tex[t0 % n, (s0 + 1) % n]
        c = tex[(t0 + 1) % n, s0 % n]
        e = tex[(t0 + 1) % n, (s0 + 1) % n]
        v = (a * (256 - fs) * (256 - ft) + b * fs * (256 - ft) + c * (256 - fs) * ft + e * fs * ft + 32768) >> 16
        return np.ascontiguousarray(v.astype(np.uint8))


def frame_crc(img):
    return zlib.crc32(np.ascontiguousarray(img).tobytes()) & 0xffffffff


# ------------------------------------------------------------------------------------------------------------------
# Import of the reference with the shims, spy and injection
# ------------------------------------------------------------------------------------------------------------------
class _NoopVisualizer:
    def __init__(self, *a, **k):
        pass

    def update(self, *a, **k):
        pass

    def render(self, *a, **k):
        pass


def import_reference():
    """-> (pipeline module, extractor module, cv2) with the shims installed.  Raises if the reference is absent."""
    if not reference_available():
        raise RuntimeError(REFERENCE_MISSING)
    import cv2
    for name in ("matplotlib", "matplotlib.pyplot", "coloredlogs"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                m = types.ModuleType(name)
                m.figure = lambda *a, **k: None
                m.install = lambda *a, **k: None
                sys.modules[name] = m
    if "matplotlib" in sys.modules and not hasattr(sys.modules["matplotlib"], "pyplot"):
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    if REFERENCE_SRC not in sys.path:
        sys.path.insert(0, REFERENCE_SRC)
    # OpenCV 4.13 API drift + headless build (SURVEY.md s4)
    if not getattr(cv2, "_klt_harness_shims", False):
        _circle, _kpc = cv2.circle, cv2.KeyPoint_convert

        def circle(img, center, radius, color, *a, **k):
            return _circle(img, (int(np.asarray(center[0]).ravel()[0]), int(np.asarray(center[1]).ravel()[0])), radius, color, *a, **k)

        def keypoint_convert(x, *a, **k):
            if isinstance(x, np.ndarray):
                x = np.ascontiguousarray(x.reshape(-1, 2), np.float32)
                return _kpc([tuple(map(float, p)) for p in x], *a, **k) if False else [cv2.KeyPoint(float(p[0]), float(p[1]), 1.0) for p in x]
            return _kpc(x, *a, **k)

        cv2.circle, cv2.KeyPoint_convert = circle, keypoint_convert
        cv2.waitKey = lambda *a, **k: -1
        cv2.imshow = lambda *a, **k: None
        cv2._klt_harness_shims = True
    import extractor.extractor as ext_mod
    import pipeline.pipeline as pipe_mod
    pipe_mod.Visualizer = _NoopVisualizer
    return pipe_mod, ext_mod, cv2


class LKSpy:
    """Stands in for cv2.calcOpticalFlowPyrLK (the attribute is looked up at call time, extractor.py:44): forwards to
    `impl` and records every call."""

    def __init__(self, impl, keep_images=False):
        self.impl = impl
        self.calls = []
        self.keep_images = keep_images
        self.seconds = 0.0

    def __call__(self, im0, im1, p0, p1, **kw):
        import time
        t = time.perf_counter()
        out = self.impl(im0, im1, p0, p1, **kw)
        self.seconds += time.perf_counter() - t
        rec = {"p0": np.array(p0, copy=True), "kw": dict(kw), "q": np.array(out[0], copy=True), "st": np.array(out[1], copy=True),
               "err": np.array(out[2], copy=True), "crc0": frame_crc(im0), "crc1": frame_crc(im1), "shape": tuple(im0.shape)}
        if self.keep_images:
            rec["im0"], rec["im1"] = im0, im1
        self.calls.append(rec)
        return out


def run_reference_pipeline(n_steps, lk_impl=None, loader=None, seed=12345):
    """Builds the reference Pipeline on the synthetic loader and runs `n_steps` Pipeline.step() calls with
    cv2.calcOpticalFlowPyrLK = LKSpy(lk_impl or the real cv2 function).
    -> dict(calls=[...], per_step=[(n_candidates, n_landmarks, landmark uv array)], step_seconds, lk_seconds)"""
    import time
    pipe_mod, ext_mod, cv2 = import_reference()
    real = getattr(cv2, "_klt_real_lk", None) or cv2.calcOpticalFlowPyrLK
    cv2._klt_real_lk = real
    spy = LKSpy(lk_impl or real)
    loader = loader or SyntheticLoader()
    cv2.setRNGSeed(seed)          # RANSAC in findEssentialMat / solvePnPRansac
    np.random.seed(seed)
    cv2.calcOpticalFlowPyrLK = spy
    try:
        pipe = pipe_mod.Pipeline(loader, headless=True)
        per_step, t_steps = [], []
        for _ in range(n_steps):
            t = time.perf_counter()
            pipe.step()
            t_steps.append(time.perf_counter() - t)
            st = pipe._state
            uv = np.array([k.uv.reshape(2) for k in st._landmarks_kp], np.float64).reshape(-1, 2)
            hist = np.array([len(k.uv_history) for k in st._landmarks_kp], np.int64)
            per_step.append({"n_candidates": len(st._candidates_kp), "n_landmarks": len(st._landmarks_kp), "landmark_uv": uv,
                             "landmark_hist_len": hist})
    finally:
        cv2.calcOpticalFlowPyrLK = real
    return {"calls": spy.calls, "per_step": per_step, "step_seconds": t_steps, "lk_seconds": spy.seconds}
