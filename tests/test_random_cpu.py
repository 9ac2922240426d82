"""Randomised parity (hypothesis, derandomised so that every run sees the same cases): the CPU oracle against live cv2 on
ragged shapes, windows, level counts, criteria, point sets and detection block sizes the hand-written cases do not
enumerate.  Same bar as tests/test_oracle.py: bit-exact."""
import numpy as np
from hypothesis import given, settings, strategies as st

from conftest import assert_lk_equal

SETTINGS = dict(max_examples=80, deadline=None, derandomize=True)


def _image(h, w, seed, kind):
    rng = np.random.default_rng(seed)
    if kind == 0:       # white noise
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == 3:       # checkerboards of 0 / 255 with cells of 1..4 pixels: the largest gradients the arithmetic can see
        c = 1 + seed % 4
        return ((((xx // c) + (yy // c)) % 2) * 255).astype(np.uint8)
    if kind == 4:       # constant image (zero gradients: the min-eigenvalue gate) with one bright pixel
        img = np.full((h, w), seed % 256, np.uint8)
        img[(seed // 7) % h, (seed // 3) % w] = 255 - seed % 256
        return img
    if kind == 1:       # smooth blobs + noise
        img = 128 + 70 * np.sin(xx / 5.0 + seed) * np.cos(yy / 7.0) + rng.normal(0, 6, (h, w))
    else:               # steps and flat areas
        img = ((xx // 9 + yy // 6) % 5) * 50 + rng.integers(0, 4, (h, w))
    return np.clip(img, 0, 255).astype(np.uint8)


@settings(**SETTINGS)
@given(h=st.integers(12, 90), w=st.integers(12, 130), seed=st.integers(0, 10 ** 6), kind=st.integers(0, 4),
       win_w=st.integers(3, 25), win_h=st.integers(3, 25), max_level=st.integers(0, 4), n=st.integers(1, 60),
       crit=st.sampled_from([(3, 30, 0.01), (3, 5, 0.03), (1, 7, 0.0), (2, 0, 0.05), (3, 100, 1e-4)]),
       flags=st.sampled_from([0, 8]), shift=st.tuples(st.integers(-4, 4), st.integers(-4, 4)))
def test_lk_oracle_equals_cv2_on_random_inputs(oracle, h, w, seed, kind, win_w, win_h, max_level, n, crit, flags, shift):
    import cv2
    a = _image(h, w, seed, kind)
    b = np.roll(a, shift, axis=(0, 1))
    rng = np.random.default_rng(seed + 1)
    p = np.stack([rng.uniform(-6, w + 6, n), rng.uniform(-6, h + 6, n)], -1).astype(np.float32).reshape(-1, 1, 2)
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=(win_w, win_h), maxLevel=max_level, criteria=crit, flags=flags)
    got = oracle.calc_optical_flow_pyr_lk(a, b, p, None, (win_w, win_h), max_level, crit, flags=flags)
    assert_lk_equal(got, ref, "h=%d w=%d win=%dx%d lvl=%d" % (h, w, win_w, win_h, max_level))


@settings(**SETTINGS)
@given(h=st.integers(1, 70), w=st.integers(1, 90), seed=st.integers(0, 10 ** 6))
def test_pyrdown_oracle_equals_cv2_on_random_shapes(oracle, h, w, seed):
    import cv2
    if h < 3 or w < 3:      # OpenCV's pyrDown handles them; the reflect-101 distances exceed the image: still must match
        pass
    a = _image(h, w, seed, 0)
    assert np.array_equal(oracle.pyr_down(a), cv2.pyrDown(a))


@settings(**SETTINGS)
@given(h=st.integers(3, 160), w=st.integers(3, 220), seed=st.integers(0, 10 ** 6), kind=st.integers(0, 4),
       block=st.sampled_from([1, 2, 3, 4, 5, 6, 15, 31]), max_corners=st.sampled_from([0, 10, 1000]),
       q=st.sampled_from([0.01, 0.03, 0.2]), min_dist=st.sampled_from([0.0, 1.0, 7.5, 10.0]), masked=st.booleans())
def test_good_features_oracle_equals_cv2_on_random_inputs(oracle, h, w, seed, kind, block, max_corners, q, min_dist, masked):
    import cv2
    if block // 2 >= min(h, w):
        block = 2 * min(h, w) - 1
    a = _image(h, w, seed, kind)
    eig = oracle.corner_min_eigen_val(a, block)
    assert np.array_equal(eig.view(np.uint32), cv2.cornerMinEigenVal(a, block, ksize=3).view(np.uint32)), (h, w, block)
    mask = None
    if masked:
        mask = np.full((h, w), 255, np.uint8)
        mask[h // 4: h // 2, w // 3: 2 * w // 3] = 0
    ref = cv2.goodFeaturesToTrack(a, max_corners, q, min_dist, mask=mask, blockSize=block)
    got = oracle.good_features_to_track(a, max_corners, q, min_dist, mask=mask, block_size=block)
    assert (ref is None) == (got is None)
    if ref is not None:
        assert got.shape == ref.shape and np.array_equal(got, ref), (h, w, block, max_corners, q, min_dist)
