"""Inputs of the cornerSubPix tests (tests/test_subpix_cpu.py, tests/test_gpu_subpix.py): images, windows, zero zones,
criteria and the points to refine, all generated from seeds."""
import numpy as np

from visual_odom_pipeline_b200 import synth as S

CAP = 15                     # include/klt_b200.h KLT_MAX_SUBPIX_WIN
WINDOWS = [(1, 1), (3, 4), (5, 5), (7, 7), (10, 10), (CAP, CAP)]
ZERO_ZONES = [(-1, -1), (0, 0), (2, 1)]
CRITERIA = [(3, 40, 0.001), (1, 10, 0.0), (2, 0, 0.03), (3, 0, 0.01), (3, 1, 0.001), (1, 150, 0.0), (3, 30, -1.0)]


def checkerboard(h, w, square=9.0, ox=0.37, oy=0.71, ss=4):
    """A checkerboard whose corners sit at sub-pixel positions (square size, offsets in pixels), rendered by averaging
    ss x ss samples per pixel."""
    s = (np.arange(ss) + 0.5) / ss
    y = (np.arange(h)[:, None] + s[None, :]).reshape(-1) - oy
    x = (np.arange(w)[:, None] + s[None, :]).reshape(-1) - ox
    v = ((np.floor(y / square)[:, None] + np.floor(x / square)[None, :]) % 2).reshape(h, ss, w, ss).mean((1, 3))
    return np.clip(40 + 170 * v, 0, 255).astype(np.uint8)


def images():
    """name -> uint8 image"""
    rng = np.random.default_rng(11)
    return {
        "kitti": S.texture(376, 1241, seed=3).astype(np.uint8),
        "noise": rng.integers(0, 256, (97, 131), dtype=np.uint8),
        "checker": checkerboard(90, 120),
        "flat": np.full((60, 70), 93, np.uint8),
    }


def points(cv2, img, win, seed, n_free=24):
    """float32 (N, 1, 2): goodFeaturesToTrack corners with jitter, points in every border band [0, win + 2) of the four
    edges and at the far edge itself, and free points anywhere (some of which diverge or walk out of the image)."""
    rng = np.random.default_rng(seed)
    h, w = img.shape
    out = []
    c = cv2.goodFeaturesToTrack(img, 60, 0.01, 5, blockSize=7)
    if c is not None:
        c = c.reshape(-1, 2) + rng.uniform(-0.7, 0.7, (len(c), 2)).astype(np.float32)
        out.append(c)
    bx, by = win[0] + 2, win[1] + 2
    n = 6
    band = [np.stack([rng.uniform(0, bx, n), rng.uniform(0, h, n)], 1), np.stack([rng.uniform(w - bx, w, n), rng.uniform(0, h, n)], 1),
            np.stack([rng.uniform(0, w, n), rng.uniform(0, by, n)], 1), np.stack([rng.uniform(0, w, n), rng.uniform(h - by, h, n)], 1),
            np.array([[0, 0], [w - 1, h - 1], [0, h - 1], [w - 1, 0], [0.25, 0.5], [w - 0.75, h - 0.5]])]
    out += band
    out.append(np.stack([rng.uniform(0, w, n_free), rng.uniform(0, h, n_free)], 1))
    p = np.concatenate(out).astype(np.float32)
    p = np.stack([np.clip(p[:, 0], 0, np.nextafter(np.float32(w), 0)), np.clip(p[:, 1], 0, np.nextafter(np.float32(h), 0))], 1)
    return p.astype(np.float32).reshape(-1, 1, 2)


def cases(cv2):
    """(name, image, points (N, 1, 2), winSize, zeroZone, criteria): every window with every image that fits it, the
    default criteria and zero zone, then the other zero zones and criteria on a rotating subset, the zero zone too large to
    apply, and an image of exactly 2w + 5 per window."""
    imgs = images()
    k = 0
    for win in WINDOWS:
        for name, img in imgs.items():
            if img.shape[1] < 2 * win[0] + 5 or img.shape[0] < 2 * win[1] + 5:
                continue
            pts = points(cv2, img, win, seed=k)
            yield "%s win%r" % (name, win), img, pts, win, (-1, -1), (3, 40, 0.001)
            zz = ZERO_ZONES[k % len(ZERO_ZONES)]
            crit = CRITERIA[k % len(CRITERIA)]
            yield "%s win%r zz%r crit%r" % (name, win, zz, crit), img, pts, win, zz, crit
            k += 1
        big = (win[0], win[1])                       # 2 * zz + 1 == W: not applied
        yield "kitti win%r zz too large" % (win,), imgs["kitti"], points(cv2, imgs["kitti"], win, seed=k), win, big, (3, 40, 0.001)
        h, w = 2 * win[1] + 5, 2 * win[0] + 5
        small = S.texture(h, w, seed=k).astype(np.uint8)
        yield "exact %dx%d win%r" % (w, h, win), small, points(cv2, small, win, seed=k, n_free=8), win, (-1, -1), (3, 40, 0.001)
        k += 1
    for crit in CRITERIA:
        yield "kitti crit%r" % (crit,), imgs["kitti"], points(cv2, imgs["kitti"], (5, 5), seed=100), (5, 5), (-1, -1), crit
