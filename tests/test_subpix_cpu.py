"""cornerSubPix, CPU tier: the restatement of cv2.cornerSubPix and getRectSubPix (oracle/subpix_oracle.c) against the live
cv2 wheel, and the drop-in's argument checks that need no device.

What "matches OpenCV" means for this call: the wheel routes getRectSubPix to a closed-source IPP primitive by default;
with cv2.ipp.setUseIPP(False) OpenCV's own code runs.  The oracle restates OpenCV's own code and must agree with it bit
for bit on every point of every case (tests/subpix_cases.py: four images, an image of exactly 2w + 5 per window, windows
up to the cap, zero zones, criteria, corners with jitter, every border band, diverging points).  Against the IPP default
the patch differs in its last bits; most points still agree to 1e-4 px, the others take another branch of the iteration
(a revert, an out-of-image stop, the convergence test) and may land anywhere within the window."""
import numpy as np
import pytest

from subpix_cases import cases, images

IPP_FAR = 1e-4            # px
IPP_FAR_FRACTION = 0.01   # of all points may lie farther than IPP_FAR from the IPP default (0.83 % measured)


@pytest.fixture(scope="module")
def subpix_oracle():
    """oracle/subpix_oracle.c through its ctypes front-end (compiled with gcc on first use)."""
    from oracle import subpix_oracle
    subpix_oracle.build()
    return subpix_oracle


@pytest.fixture()
def cv2_generic():
    cv2 = pytest.importorskip("cv2")
    was = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield cv2
    cv2.ipp.setUseIPP(was)


def test_rect_sub_pix_restates_opencv_interior_and_border(subpix_oracle, cv2_generic):
    cv2 = cv2_generic
    rng = np.random.default_rng(2)
    img = rng.integers(0, 256, (40, 50), dtype=np.uint8)
    border = 0
    for _ in range(3000):
        pw, ph = int(rng.integers(3, 36)), int(rng.integers(3, 36))
        cx, cy = np.float32(rng.uniform(-2, 52)), np.float32(rng.uniform(-2, 42))
        ref = cv2.getRectSubPix(img, (pw, ph), (float(cx), float(cy)), patchType=cv2.CV_32F)
        got = subpix_oracle.rect_sub_pix(img, (pw, ph), (cx, cy))
        assert np.array_equal(ref.view(np.uint32), got.view(np.uint32)), (pw, ph, cx, cy)
        ix, iy = np.floor(cx - (pw - 1) * 0.5), np.floor(cy - (ph - 1) * 0.5)
        border += not (0 <= ix and ix + pw < 50 and 0 <= iy and iy + ph < 40)
    assert border > 1000


def test_mask_uses_the_c_librarys_expf(subpix_oracle):
    import ctypes
    libm = ctypes.CDLL("libm.so.6")
    libm.expf.restype, libm.expf.argtypes = ctypes.c_float, [ctypes.c_float]
    f = np.float32
    for wx, wy in [(1, 1), (3, 4), (5, 5), (15, 15)]:
        m = subpix_oracle.subpix_mask((wx, wy))
        for i in range(2 * wy + 1):
            y = f(f(i - wy) / f(wy))
            for j in range(2 * wx + 1):
                x = f(f(j - wx) / f(wx))
                assert m[i, j] == f(f(libm.expf(float(f(-y * y)))) * f(libm.expf(float(f(-x * x)))))


def test_oracle_restates_opencvs_own_corner_sub_pix(subpix_oracle, cv2_generic):
    cv2 = cv2_generic
    n_cases = n_pts = moved = reverted = 0
    for name, img, pts, win, zz, crit in cases(cv2):
        ref = cv2.cornerSubPix(img, pts.copy(), win, zz, crit)
        got = subpix_oracle.corner_sub_pix(img, pts, win, zz, crit)
        bad = np.nonzero((got.view(np.uint32) != ref.view(np.uint32)).any(-1).ravel())[0]
        assert bad.size == 0, "%s: %d of %d points differ, first %s -> want %s got %s" % (
            name, bad.size, len(pts), pts[bad[0], 0], ref[bad[0], 0], got[bad[0], 0])
        n_cases += 1
        n_pts += len(pts)
        moved += int((got != pts).any(-1).sum())
        reverted += int(((got == pts).all(-1) & ~np.isin(name.split()[0], ["flat"])).sum())
    assert n_cases >= 60 and n_pts >= 6000
    assert moved > n_pts // 2 and reverted > 0


def test_flat_image_stops_at_the_determinant(subpix_oracle, cv2_generic):
    img = images()["flat"]
    pts = np.array([[[10.3, 20.7]], [[35.0, 30.5]]], np.float32)
    got, iters = subpix_oracle.corner_sub_pix(img, pts, (5, 5), (-1, -1), (3, 40, 0.001), return_iters=True)
    assert np.array_equal(got, pts) and list(iters) == [1, 1]
    assert np.array_equal(cv2_generic.cornerSubPix(img, pts.copy(), (5, 5), (-1, -1), (3, 40, 0.001)), pts)


def test_oracle_within_tolerance_of_the_ipp_wheel(subpix_oracle):
    cv2 = pytest.importorskip("cv2")
    if not cv2.ipp.useIPP():
        pytest.skip("this cv2 build has no IPP path")
    far = total = 0
    for name, img, pts, win, zz, crit in cases(cv2):
        ref = cv2.cornerSubPix(img, pts.copy(), win, zz, crit)
        got = subpix_oracle.corner_sub_pix(img, pts, win, zz, crit)
        d = np.abs(got - ref).reshape(-1, 2).max(1)
        assert (d <= max(win) + 1).all(), name
        far += int((d > IPP_FAR).sum())
        total += len(d)
    assert far <= IPP_FAR_FRACTION * total, "%d of %d points farther than %g px from the IPP default" % (far, total, IPP_FAR)


def test_oracle_rejects_what_cv2_rejects(subpix_oracle):
    img = images()["noise"]
    p = np.array([[20.0, 30.0]], np.float32)
    for bad_pts in ([[131.0, 5.0]], [[-0.01, 5.0]], [[np.nan, 5.0]], [[5.0, 97.0]]):
        with pytest.raises(ValueError):
            subpix_oracle.corner_sub_pix(img, np.array(bad_pts, np.float32), (5, 5), (-1, -1), (3, 40, 0.001))
    for win in ((0, 5), (5, -1)):
        with pytest.raises(ValueError):
            subpix_oracle.corner_sub_pix(img, p, win, (-1, -1), (3, 40, 0.001))
    with pytest.raises(ValueError):
        subpix_oracle.corner_sub_pix(img[:14, :14], p * 0 + 5, (5, 5), (-1, -1), (3, 40, 0.001))
    subpix_oracle.corner_sub_pix(img[:15, :15], p * 0 + 5, (5, 5), (-1, -1), (3, 40, 0.001))


# ---- the drop-in's checks, all on the host before any device call --------------------------------------------------------

def _err(klt, *args, match):
    with pytest.raises(klt.error, match=match):
        klt.cornerSubPix(*args)


def test_drop_in_argument_errors_need_no_device(klt):
    img = images()["noise"]
    p = np.array([[[20.3, 30.1]], [[40.0, 12.5]]], np.float32)
    crit = (3, 40, 0.001)
    _err(klt, img, p.astype(np.float64), (5, 5), (-1, -1), crit, match="count >= 0")
    _err(klt, img, p.reshape(-1, 2).astype(np.int32), (5, 5), (-1, -1), crit, match="count >= 0")
    _err(klt, img, np.zeros((2, 3), np.float32) + 20, (5, 5), (-1, -1), crit, match="count >= 0")
    _err(klt, img, (np.zeros((4, 2), np.float32) + 20)[::2], (5, 5), (-1, -1), crit, match="count >= 0")
    _err(klt, img, p.copy(), (0, 5), (-1, -1), crit, match="win.width > 0 && win.height > 0")
    _err(klt, img[:14, :14], p * 0 + 5, (5, 5), (-1, -1), crit, match="src.cols >= win.width\\*2 \\+ 5")
    _err(klt, img, p.copy(), (klt.KLT_MAX_SUBPIX_WIN + 1, 5), (-1, -1), crit, match="KLT_MAX_SUBPIX_WIN")
    for bad in ([[131.0, 5.0]], [[-0.01, 5.0]], [[np.nan, 5.0]], [[5.0, np.inf]]):
        q = np.array(bad, np.float32)
        _err(klt, img, q, (5, 5), (-1, -1), crit, match="contains\\(cT\\)")
        assert np.array_equal(q, np.array(bad, np.float32), equal_nan=True)
    _err(klt, img.astype(np.float32), p.copy(), (5, 5), (-1, -1), crit, match="float32 images are not supported")
    _err(klt, "img", p.copy(), (5, 5), (-1, -1), crit, match="not a numpy array")
    empty = np.zeros((0, 1, 2), np.float32)
    assert klt.cornerSubPix(img, empty, (5, 5), (-1, -1), crit) is empty
