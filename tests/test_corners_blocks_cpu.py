"""CPU tier of the detection step away from the reference's blockSize 31: the C oracle (oracle/gftt_oracle.c) against
live cv2.cornerMinEigenVal / cv2.goodFeaturesToTrack at every small block size, on the images where the box sums'
rounding shows (uniform noise, 0/255 noise) and on the shapes where the row filter and the reflection change regime
(W % 32 on both sides of 0, W < 32, H and W down to 1).  cornerMinEigenVal and goodFeaturesToTrack are public drop-ins
whose default is blockSize=3, so every block size a caller may pass must be exact, not just 31.

A second test pins rule G.5 where it lives: the box sums restated in numpy against cv2.boxFilter on cv2's own Sobel
products.  When a cv2 wheel changes the box order, that test fails next to the eigenvalue test and names the stage.

Bar: eigenvalue maps equal as uint32, corners equal in value and order."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

BLOCKS = list(range(1, 18)) + [31, 32, 33, 63, 64, 65]
KINDS = ["noise", "binary", "smooth", "constant", "spot"]
# (h, w): W % 32 on both sides of 0 and W < 32 (the scalar tail of the y-derivative's row filter, G.3), H and W down to 1
SHAPES = [(1, 1), (1, 37), (29, 1), (2, 2), (2, 64), (3, 31), (7, 33), (16, 5), (31, 32), (33, 63), (40, 65), (57, 96),
          (64, 97), (100, 129), (376, 1241)]
SEEDS = 3        # images per shape and kind (noise, binary, spot); the 1-4 ulp box-sum differences are sparse
GFTT_PARAMS = [(0, 0.01, 0.0, False), (40, 0.03, 3.5, True)]   # (maxCorners, qualityLevel, minDistance, masked)


def image(kind, h, w, seed):
    """Deterministic uint8 (h, w) image of one kind."""
    rng = np.random.default_rng(1000003 * seed + 1009 * h + w)
    if kind == "noise":
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "binary":         # the largest gradients the arithmetic can see, everywhere
        return (rng.integers(0, 2, (h, w)) * 255).astype(np.uint8)
    if kind == "constant":       # all products 0: the map must be exactly 0
        return np.full((h, w), 37 + seed, np.uint8)
    if kind == "spot":           # one bright pixel on a constant image
        img = np.full((h, w), 20, np.uint8)
        img[int(rng.integers(0, h)), int(rng.integers(0, w))] = 255
        return img
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    ph = rng.uniform(0, 6.283, 3)
    img = 128 + 60 * np.sin(xx / 4.3 + ph[0]) * np.cos(yy / 6.1 + ph[1]) + 50 * np.sin((xx + yy) / 11.7 + ph[2])
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


def images(h, w):
    for kind in KINDS:
        for seed in range(1 if kind in ("smooth", "constant") else SEEDS):
            yield kind, seed, image(kind, h, w, seed)


def accepted(block, h, w):
    """The library refuses block / 2 >= min(h, w) (the border would reach past the reflected image)."""
    return block // 2 < min(h, w)


def corner_mask(h, w, seed):
    rng = np.random.default_rng(seed)
    m = np.full((h, w), 255, np.uint8)
    m[rng.integers(0, h, max(1, h * w // 7)), rng.integers(0, w, max(1, h * w // 7))] = 0
    return m


def eig_mismatch(got, want):
    bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
    if bad.size == 0:
        return None
    i = tuple(bad[0])
    return "%d / %d differ, first at %s: %r vs cv2 %r" % (len(bad), got.size, i, got[i], want[i])


def same_corners(a, b):
    if a is None or b is None:
        return a is None and b is None
    return a.shape == b.shape and np.array_equal(a, b)


def _check_block(oracle, block, shapes):
    failures = []
    for (h, w) in shapes:
        for kind, seed, img in images(h, w):
            what = "block %d, %dx%d %s seed %d" % (block, h, w, kind, seed)
            msg = eig_mismatch(oracle.corner_min_eigen_val(img, block), cv2.cornerMinEigenVal(img, block, ksize=3))
            if msg:
                failures.append("%s: eigenvalues: %s" % (what, msg))
            for (mc, ql, md, masked) in GFTT_PARAMS:
                m = corner_mask(h, w, seed) if masked else None
                c = oracle.good_features_to_track(img, mc, ql, md, mask=m, block_size=block)
                k = cv2.goodFeaturesToTrack(img, mc, ql, md, mask=m, blockSize=block)
                if not same_corners(c, k):
                    failures.append("%s: corners differ for maxCorners=%d quality=%g minDistance=%g masked=%s" % (what, mc, ql, md, masked))
    assert not failures, "%d cases differ from cv2:\n%s" % (len(failures), "\n".join(failures[:25]))


@pytest.mark.parametrize("block", BLOCKS)
def test_oracle_equals_cv2_at_block_size(oracle, block):
    shapes = [s for s in SHAPES if accepted(block, *s)]
    assert shapes
    _check_block(oracle, block, shapes)


@pytest.mark.parametrize("hw", SHAPES)
def test_oracle_equals_cv2_at_the_largest_accepted_block(oracle, hw):
    block = 2 * min(hw) - 1
    assert accepted(block, *hw) and not accepted(block + 1, *hw)
    _check_block(oracle, block, [hw])


def _refl101(p, n):
    while p < 0 or p >= n:
        p = -p if p < 0 else 2 * n - 2 - p
    return p


def box_sums_g5(plane, block):
    """G.5 of oracle/gftt_oracle.c restated in numpy: unnormalised block x block box sums of a float32 plane, reflect-101
    border, anchor block / 2, in double precision and OpenCV's order, then rounded to float32.
    Rows: fresh left-to-right sums of `block` values for block <= 5; a running sum for larger blocks (the sum of the first
    `block` values, then s += (double)new - (double)old per step).  Columns: a running sum (the first block - 1 row sums
    top to bottom, then per output row s0 = SUM + entering, out = (float)s0, SUM = s0 - leaving)."""
    h, w = plane.shape
    an = block // 2
    xs = [_refl101(i - an, w) for i in range(w + block - 1)]
    ys = [_refl101(i - an, h) for i in range(h + block - 1)]
    p = plane.astype(np.float64)
    rows = np.empty((h, w))
    if block <= 5:
        for x in range(w):
            s = p[:, xs[x]].copy()
            for k in range(1, block):
                s = s + p[:, xs[x + k]]
            rows[:, x] = s
    else:
        s = np.zeros(h)
        for i in range(block):
            s = s + p[:, xs[i]]
        rows[:, 0] = s
        for x in range(w - 1):
            s = s + (p[:, xs[x + block]] - p[:, xs[x]])
            rows[:, x + 1] = s
    out = np.empty((h, w), np.float32)
    acc = np.zeros(w)
    for i in range(block - 1):
        acc = acc + rows[ys[i]]
    for y in range(h):
        s0 = acc + rows[ys[y + block - 1]]
        out[y] = s0.astype(np.float32)
        acc = s0 - rows[ys[y]]
    return out


def _box_inputs(block):
    """(name, float32 plane) pairs: cv2's own products (Sobel with the G.1 scale, float32 products), so that a mismatch
    is the box filter's and not the derivatives'; and planes of sparse values about 2^30 above a floor, where a running
    sum's rounding error outlives the value that caused it and a fresh sum has none."""
    for (h, w) in [(37, 41), (100, 129), (376, 1241)]:
        if not accepted(block, h, w):
            continue
        for kind in ("noise", "binary"):
            for seed in range(2):
                img = image(kind, h, w, seed)
                scale = 1.0 / (4 * block * 255.0)
                dx = cv2.Sobel(img, cv2.CV_32F, 1, 0, ksize=3, scale=scale, borderType=cv2.BORDER_REFLECT_101)
                dy = cv2.Sobel(img, cv2.CV_32F, 0, 1, ksize=3, scale=scale, borderType=cv2.BORDER_REFLECT_101)
                for name, prod in (("Dx*Dx", dx * dx), ("Dx*Dy", dx * dy), ("Dy*Dy", dy * dy)):
                    yield "%dx%d %s seed %d %s" % (h, w, kind, seed, name), prod
    for (h, w) in [(37, 41), (70, 129)]:
        if accepted(block, h, w):
            rng = np.random.default_rng(h * w)
            floor = np.where(rng.random((h, w)) < 0.1, 1.0, 2.0 ** -30)
            yield "%dx%d sparse values" % (h, w), (rng.uniform(-2, 2, (h, w)) * floor).astype(np.float32)


@pytest.mark.parametrize("block", BLOCKS)
def test_box_sum_order_equals_cv2_box_filter(block):
    """Stage G.5 alone against cv2.boxFilter(normalize=False, BORDER_REFLECT_101) on float32 planes."""
    failures = []
    for what, plane in _box_inputs(block):
        want = cv2.boxFilter(plane, -1, (block, block), normalize=False, borderType=cv2.BORDER_REFLECT_101)
        msg = eig_mismatch(box_sums_g5(plane, block), want)
        if msg:
            failures.append("%s: %s" % (what, msg))
    assert not failures, "\n".join(failures[:20])
