"""Deterministic synthetic inputs for parity tests and benchmarks (SURVEY.md s8d).

Frames are multi-scale band-limited noise; the second frame is an affine warp of the first.  There
are no datasets in the image (no network), so every test / bench input comes from here.  cv2 is
used only as an image-synthesis utility (GaussianBlur / warpAffine), never on the tracking path.
"""
import numpy as np

BENIGN = (3.3, -1.7, 0.4, 1.01)   # tx, ty, rot_deg, scale
HARD = (14.2, 5.3, 1.5, 1.03)


def texture(h, w, seed=7):
    """float32 (h, w) in [0, 255]: sum of 4 octaves of blurred white noise."""
    import cv2
    rng = np.random.default_rng(seed)
    img = np.zeros((h, w), np.float32)
    for sigma, amp in [(1.0, 40), (2.5, 60), (6, 80), (15, 60)]:
        n = rng.standard_normal((h, w)).astype(np.float32)
        n = cv2.GaussianBlur(n, (0, 0), sigma)
        n /= n.std()
        img += amp * n
    img = (img - img.min()) / (img.max() - img.min()) * 255.0
    return img.astype(np.float32)


def warp(img_f32, motion=BENIGN):
    import cv2
    h, w = img_f32.shape
    tx, ty, rot, scale = motion
    M = cv2.getRotationMatrix2D((w / 2, h / 2), rot, scale)
    M[0, 2] += tx
    M[1, 2] += ty
    return cv2.warpAffine(img_f32, M, (w, h), flags=cv2.INTER_CUBIC, borderMode=cv2.BORDER_REFLECT_101)


def frame_pair(h, w, seed=7, motion=BENIGN, noise_sigma=0.0, flat_cols=None):
    """-> (prev uint8 (h,w), next uint8 (h,w))."""
    f0 = texture(h, w, seed)
    if flat_cols is not None:
        f0[:, flat_cols[0]:flat_cols[1]] = 128.0
    f1 = warp(f0, motion)
    if noise_sigma > 0:
        rng = np.random.default_rng(seed + 1000)
        f1 = f1 + rng.normal(0, noise_sigma, f1.shape).astype(np.float32)
    return np.clip(f0, 0, 255).astype(np.uint8), np.clip(f1, 0, 255).astype(np.uint8)


def sequence(h, w, n_frames, seed=7, motion=(1.1, -0.6, 0.15, 1.003)):
    """list of n_frames uint8 frames, each the same small warp of the previous one."""
    f = texture(h, w, seed)
    out = [np.clip(f, 0, 255).astype(np.uint8)]
    for _ in range(n_frames - 1):
        f = warp(f, motion)
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return out


def uniform_points(n, h, w, seed=3, margin=0.0):
    """float32 (n,1,2) uniform in [-margin, w+margin) x [-margin, h+margin)."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-margin, w + margin, n)
    y = rng.uniform(-margin, h + margin, n)
    return np.stack([x, y], -1).astype(np.float32).reshape(-1, 1, 2)


def grid_points(nx, ny, h, w):
    xs = (np.arange(nx, dtype=np.float32) + 0.5) * (w / nx)
    ys = (np.arange(ny, dtype=np.float32) + 0.5) * (h / ny)
    gx, gy = np.meshgrid(xs, ys)
    return np.stack([gx, gy], -1).astype(np.float32).reshape(-1, 1, 2)


def shade(frame, left_gain, frac=1.0 / 3.0):
    """uint8 frame with the contrast of its left `frac` of columns scaled by left_gain about 128 (a fixed shadow-like gain
    map: g(x) = left_gain for x < frac * w, 1 elsewhere), in float32, rounded and clipped back to uint8."""
    f = np.asarray(frame, np.float32)
    g = np.ones(f.shape[1], np.float32)
    g[:int(f.shape[1] * frac)] = np.float32(left_gain)
    return np.clip(np.rint(128.0 + (f - 128.0) * g[None, :]), 0, 255).astype(np.uint8)


def uneven_sequence(h, w, n_frames, seed=100, left_gain=0.1, motion=(1.1, -0.6, 0.15, 1.003)):
    """sequence() with the fixed gain map of shade() applied after each warp: the left third of every frame has
    left_gain times the contrast of the rest, as under a shadow that stays in place while the scene moves."""
    f = texture(h, w, seed)
    out = [shade(np.clip(f, 0, 255), left_gain)]
    for _ in range(n_frames - 1):
        f = warp(f, motion)
        out.append(shade(np.clip(f, 0, 255), left_gain))
    return out


def exposure_sequence(h, w, n_frames, gains, seed=7, motion=(1.1, -0.6, 0.15, 1.003)):
    """sequence() under a changing exposure: frame t is clip(rint(f_t * gains[t])) of the float frame f_t (the same small
    warp of the previous one), as when a camera's auto-exposure changes its gain between frames."""
    if len(gains) != n_frames:
        raise ValueError("exposure_sequence needs one gain per frame")
    f = texture(h, w, seed)
    out = []
    for t in range(n_frames):
        if t:
            f = warp(f, motion)
        out.append(np.clip(np.rint(f * np.float32(gains[t])), 0, 255).astype(np.uint8))
    return out
