"""CPU tier of contrast-limited adaptive histogram equalisation: the restatement oracle/clahe_oracle.py of OpenCV 4.13's
CLAHE_Impl::apply against the live cv2 wheel, bit for bit (IPP does not change this function), and the checks of the
createCLAHE drop-in and of the tracker option that run on the host before any device work."""
import numpy as np
import pytest

from clahe_cases import CLIPS, GRIDS, cases, image
from oracle import clahe_oracle as O
from visual_odom_pipeline_b200 import synth as S


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def test_oracle_bit_exact_with_opencv(cv2):
    n = 0
    for name, img, clip, grid in cases():
        ref = cv2.createCLAHE(clip, grid).apply(img)
        got = O.clahe(img, clip, grid)
        bad = int((got != ref).sum())
        assert bad == 0, "%s: %d of %d pixels differ" % (name, bad, ref.size)
        n += ref.size
    assert n > 20_000_000


def test_oracle_on_exposure_sequence_frames(cv2):
    """The frames of the tracker tests: (3.0, (8, 8)) and the defaults on every gain."""
    seq = S.exposure_sequence(376, 1241, 4, [1.0, 0.5, 1.4, 0.6], seed=11)
    for f in seq:
        for clip, grid in [(3.0, (8, 8)), (40.0, (8, 8)), (2.0, (4, 6))]:
            assert np.array_equal(O.clahe(f, clip, grid), cv2.createCLAHE(clip, grid).apply(f))


def test_padding_quirk_and_reflection():
    """An axis that divides still gets a whole tile of padding when the other does not; padding larger than the image
    reflects with several bounces (and repeats a 1-pixel axis)."""
    assert O.plan(1241, 376, 3.0, (8, 8))[:4] == (1248, 384, 156, 48)
    assert O.plan(1240, 376, 3.0, (8, 8))[:4] == (1240, 376, 155, 47)
    assert O.plan(1240, 377, 3.0, (8, 8))[:4] == (1248, 384, 156, 48)
    assert O.plan(3, 3, 3.0, (20, 20))[:4] == (20, 20, 1, 1)
    assert list(O.reflect101(np.arange(10), 3)) == [0, 1, 2, 1, 0, 1, 2, 1, 0, 1]
    assert list(O.reflect101(np.arange(4), 1)) == [0, 0, 0, 0]


def test_tile_index_of_every_pixel_is_in_range():
    """The device blend looks up tiles tx1 = floor(float32(x) * (1.0f / tw) - 0.5f) and tx1 + 1 (clamped from above) for
    x < w only; for those the float32 index never passes the last tile, with or without padding, so only pixels past the
    row's end (which the kernel skips) could reach a table outside the workspace."""
    f32 = np.float32
    for w, tx in [(1241, 8), (1241, 1241), (1241, 1), (9, 9), (1, 1), (13, 13), (30, 10), (1241, 20), (3, 20), (2048, 512),
                  (4096, 1024), (1920, 7)]:
        for h, ty in [(376, 47), (376, 8), (8, 8)]:
            wext = O.plan(w, h, 1.0, (tx, ty))[0]
            tw = wext // tx
            x = np.arange(w).astype(f32)
            t1 = np.floor(x * (f32(1) / f32(tw)) - f32(0.5)).astype(np.int64)
            assert t1.max() <= tx - 1 and t1.min() >= -1, (w, tx, h, ty)
            beyond = np.floor(np.arange(w, w + 4).astype(f32) * (f32(1) / f32(tw)) - f32(0.5)).astype(np.int64)
            if wext == w and tw <= 4 and w % 4:
                assert beyond.max() > tx - 1       # what an unguarded 4-pixel group would have read


def test_clip_count_and_remainder():
    """clip = max(int(clipLimit * total / 256), 1) in double, 0 for clipLimit <= 0; the remainder of the excess goes to
    bins 0, s, 2s, ... (s = max(256 // r, 1)), the first r of them."""
    assert O.plan(1241, 376, 3.0, (8, 8))[4] == int(3.0 * 7488 / 256)
    assert O.plan(1241, 376, 1e-9, (8, 8))[4] == 1
    assert O.plan(1241, 376, 0.0, (8, 8))[4] == 0 and O.plan(1241, 376, -5.0, (8, 8))[4] == 0
    # one tile of 256 pixels, all of value 0 -> clip = 3, excess 253 = 0 * 256 + 253: bins 0..252 get one each
    img = np.zeros((16, 16), np.uint8)
    lut = O.luts(img, 3.0, (1, 1))[0].astype(int)
    hist = np.zeros(256, int)
    hist[0] = 3
    hist[:253] += 1
    want = np.clip(np.rint(np.cumsum(hist).astype(np.float32) * (np.float32(255) / np.float32(256))), 0, 255)
    assert np.array_equal(lut, want)


def test_cases_cover_the_matrix():
    cs = cases()
    assert {c[3] for c in cs} == set(GRIDS) and {c[2] for c in cs} == set(CLIPS)
    assert any(c[1].shape[1] < c[3][0] for c in cs)         # more tiles than columns
    assert len(np.unique(image("levels", 50, 50, 3))) <= 4


# ---- the front end's checks, all on the host before any device call -----------------------------------------------------

def test_drop_in_defaults_and_accessors(klt):
    c = klt.createCLAHE()
    assert c.getClipLimit() == 40.0 and c.getTilesGridSize() == (8, 8)
    c.setClipLimit(3)
    c.setTilesGridSize((4, 6))
    assert c.getClipLimit() == 3.0 and c.getTilesGridSize() == (4, 6)
    c = klt.createCLAHE(2.0, (16, 3))
    assert c.getClipLimit() == 2.0 and c.getTilesGridSize() == (16, 3)


def test_drop_in_argument_errors_need_no_device(klt):
    img = image("noise", 40, 50, 1)
    for grid in [(0, 8), (8, 0), (-1, 8)]:
        with pytest.raises(klt.error, match="tilesX_ > 0"):
            klt.createCLAHE(3.0, grid)
    with pytest.raises(klt.error, match="KLT_MAX_CLAHE_TILES"):
        klt.createCLAHE(3.0, (257, 256))
    for bad in (float("nan"), float("inf"), -float("inf")):
        with pytest.raises(klt.error, match="finite"):
            klt.createCLAHE(bad, (8, 8))
    with pytest.raises(klt.error, match="pair of ints"):
        klt.createCLAHE(3.0, 8)
    c = klt.createCLAHE(3.0, (8, 8))
    with pytest.raises(klt.error, match="16-bit"):
        c.apply(img.astype(np.uint16))
    for bad in (np.dstack([img] * 3), img.astype(np.float32), img.astype(np.int8)):
        with pytest.raises(klt.error, match="CV_8UC1"):
            c.apply(bad)
    with pytest.raises(klt.error, match="CV_8UC1"):
        c.apply("img")
    with pytest.raises(klt.error, match="empty"):
        c.apply(np.zeros((0, 5), np.uint8))
    # clip_limit * total / 256 must fit an int32: one tile, no padding (1241 x 376 divides by (1, 1)), total = 1241 * 376
    big = np.zeros((376, 1241), np.uint8)
    with pytest.raises(klt.error, match="int32"):
        klt.createCLAHE(2.0 ** 31 * 256 / (1241 * 376) * 1.01, (1, 1)).apply(big)
    assert issubclass(klt.error, Exception)


def test_tracker_option_checks_need_no_device(klt):
    from visual_odom_pipeline_b200 import tracker as T
    assert T.check_equalize(None) is None
    assert T.check_equalize((3, [8, 8]), 1241, 376) == (3.0, (8, 8))
    for bad in [3.0, (3.0,), (3.0, (0, 8)), (float("nan"), (8, 8)), (3.0, (300, 300)), (1e12, (8, 8))]:
        with pytest.raises(klt.error):
            T.check_equalize(bad, 1241, 376)
    for bad in [(3.0, (0, 8)), (float("inf"), (8, 8))]:
        with pytest.raises(klt.error):
            T.KLTTracker(equalize=bad)


def test_ws_bytes(klt):
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    assert L.klt_clahe_ws_bytes(1, 8, 8) == 64 * 256
    assert L.klt_clahe_ws_bytes(64, 16, 3) == 64 * 48 * 256
    assert L.klt_clahe_ws_bytes(0, 8, 8) == 0 and L.klt_clahe_ws_bytes(1, 0, 8) == 0 and L.klt_clahe_ws_bytes(1, 8, -1) == 0


def test_exposure_sequence():
    gains = [1.0, 0.7, 1.4]
    seq = S.exposure_sequence(60, 80, 3, gains, seed=5, motion=(1.0, 0.0, 0.0, 1.0))
    f = S.texture(60, 80, 5)
    assert np.array_equal(seq[0], np.clip(np.rint(f), 0, 255).astype(np.uint8))
    f2 = S.warp(S.warp(f, (1.0, 0.0, 0.0, 1.0)), (1.0, 0.0, 0.0, 1.0))
    assert np.array_equal(seq[2], np.clip(np.rint(f2 * np.float32(1.4)), 0, 255).astype(np.uint8))
    with pytest.raises(ValueError):
        S.exposure_sequence(60, 80, 3, [1.0], seed=5)
