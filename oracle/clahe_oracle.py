"""Restatement of OpenCV 4.13's CLAHE_Impl::apply for 8-bit single-channel images (modules/imgproc/src/clahe.cpp) in
numpy -- TEST INFRASTRUCTURE ONLY.  tests/test_clahe_cpu.py pins it to the cv2 wheel bit for bit (IPP does not change
this function); the device kernels (visual-odom-pipeline_b200/csrc/klt_clahe.cu) implement the same steps.

For a w x h image, tiles = (tx, ty) and clipLimit:
  C.1 padding: none when w % tx == 0 and h % ty == 0; otherwise BORDER_REFLECT_101 on the right by tx - w % tx and at
      the bottom by ty - h % ty -- an axis that divides evenly still gets a whole extra tile when the other does not.
      The padding may be larger than the image (several bounces; a 1-pixel axis repeats its pixel).
  C.2 tile tw x th = padded size / tiles, total = tw * th, lutScale = float32(255) / float32(total).
  C.3 clip = max(int(clipLimit * total / 256), 1) in double when clipLimit > 0, else 0 (no clipping).
  C.4 per tile k = j * tx + i: the 256-bin histogram of the padded tile; when clip > 0 every bin is cut at clip, the
      excess e is spread as e // 256 to every bin, and one more goes to bins 0, s, 2s, ... (s = max(256 // r, 1)), the
      first r = e % 256 of them; lut[k][v] = saturate_u8(round_half_even(float32(cumsum[v]) * lutScale)).
  C.5 per pixel of the unpadded image: tyf = float32(y) * (1.0f / th) - 0.5f, ty1 = floor(tyf), ya = tyf - ty1,
      ya1 = 1 - ya, ty2 = min(ty1 + 1, ty - 1), ty1 = max(ty1, 0); the same along x; res = (L[ty1,tx1][v] * xa1 +
      L[ty1,tx2][v] * xa) * ya1 + (L[ty2,tx1][v] * xa1 + L[ty2,tx2][v] * xa) * ya in float32, each operation rounded
      once, left to right; dst = saturate_u8(round_half_even(res)).
"""
import numpy as np

f32 = np.float32


def reflect101(p, n):
    """BORDER_REFLECT_101 index of p into [0, n), as many bounces as it takes (csrc/klt_common.cuh reflect101)."""
    p = np.array(p, np.int64)
    if n == 1:
        return np.zeros_like(p)
    period = 2 * n - 2
    p = np.abs(p) % period
    return np.where(p < n, p, period - p)


def plan(w, h, clip_limit, tiles):
    """C.1-C.3 -> (padded width, padded height, tw, th, clip, lutScale)."""
    tx, ty = int(tiles[0]), int(tiles[1])
    if tx < 1 or ty < 1:
        raise ValueError("tiles must be >= 1")
    if w % tx == 0 and h % ty == 0:
        wext, hext = w, h
    else:
        wext, hext = w + tx - w % tx, h + ty - h % ty
    tw, th = wext // tx, hext // ty
    total = tw * th
    clip = max(int(float(clip_limit) * total / 256), 1) if clip_limit > 0 else 0
    return wext, hext, tw, th, clip, f32(255) / f32(total)


def luts(img, clip_limit=40.0, tiles=(8, 8)):
    """C.1-C.4 -> uint8 (ty * tx, 256), the tables of the tiles in row-major order."""
    img = np.asarray(img)
    assert img.dtype == np.uint8 and img.ndim == 2
    h, w = img.shape
    tx, ty = int(tiles[0]), int(tiles[1])
    wext, hext, tw, th, clip, lut_scale = plan(w, h, clip_limit, tiles)
    ext = img[reflect101(np.arange(hext), h)[:, None], reflect101(np.arange(wext), w)[None, :]]
    tile = (np.arange(hext) // th)[:, None] * tx + (np.arange(wext) // tw)[None, :]
    hist = np.bincount((tile * 256 + ext).ravel(), minlength=tx * ty * 256).reshape(tx * ty, 256).astype(np.int64)
    if clip > 0:
        excess = np.maximum(hist - clip, 0).sum(1)
        hist = np.minimum(hist, clip) + (excess // 256)[:, None]
        r = excess % 256
        s = np.maximum(256 // np.maximum(r, 1), 1)
        i = np.arange(256)[None, :]
        hist += ((r[:, None] > 0) & (i % s[:, None] == 0) & (i // s[:, None] < r[:, None])).astype(np.int64)
    cum = np.cumsum(hist, 1).astype(f32)
    return np.clip(np.rint(cum * lut_scale), 0, 255).astype(np.uint8)


def _axis(n, t, tiles):
    c = np.arange(n).astype(f32) * (f32(1) / f32(t)) - f32(0.5)
    i1 = np.floor(c).astype(np.int64)
    a = (c - i1.astype(f32)).astype(f32)
    a1 = (f32(1) - a).astype(f32)
    return np.maximum(i1, 0), np.minimum(i1 + 1, tiles - 1), a, a1


def clahe(img, clip_limit=40.0, tiles=(8, 8)):
    """cv2.createCLAHE(clip_limit, tiles).apply(img) for uint8 (h, w) -> uint8 (h, w)."""
    img = np.asarray(img)
    h, w = img.shape
    tx, ty = int(tiles[0]), int(tiles[1])
    _, _, tw, th, _, _ = plan(w, h, clip_limit, tiles)
    L = luts(img, clip_limit, tiles).astype(f32)
    x1, x2, xa, xa1 = _axis(w, tw, tx)
    y1, y2, ya, ya1 = _axis(h, th, ty)
    v = img.astype(np.int64)

    def at(ty_, tx_):
        return L[ty_[:, None] * tx + tx_[None, :], v]
    top = at(y1, x1) * xa1 + at(y1, x2) * xa
    bot = at(y2, x1) * xa1 + at(y2, x2) * xa
    res = top * ya1[:, None] + bot * ya[:, None]
    assert res.dtype == f32
    return np.clip(np.rint(res), 0, 255).astype(np.uint8)
