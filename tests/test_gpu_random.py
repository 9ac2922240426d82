"""Randomised GPU parity (hypothesis, derandomised): the CUDA path through the public drop-ins against live cv2 on ragged
shapes, windows (generic and specialised kernels), level counts, criteria, flags and point sets -- bit-exact, like the
hand-written cases of tests/test_gpu_parity.py / test_gpu_corners.py / test_gpu_bilateral.py."""
import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from conftest import assert_lk_equal
from test_random_cpu import _image

pytestmark = pytest.mark.gpu
SETTINGS = dict(max_examples=250, deadline=None, derandomize=True)


@settings(**SETTINGS)
@given(h=st.integers(12, 200), w=st.integers(12, 260), seed=st.integers(0, 10 ** 6), kind=st.integers(0, 4),
       win=st.one_of(st.sampled_from([(21, 21), (31, 31)]), st.tuples(st.integers(3, 41), st.integers(3, 41))),
       max_level=st.integers(0, 5), n=st.integers(1, 300),
       crit=st.sampled_from([(3, 30, 0.01), (3, 30, 0.03), (3, 5, 0.03), (1, 7, 0.0), (2, 0, 0.05), (3, 100, 1e-4)]),
       flags=st.sampled_from([0, 8, 4]), shift=st.tuples(st.integers(-6, 6), st.integers(-6, 6)))
def test_lk_equals_cv2_on_random_inputs(klt, h, w, seed, kind, win, max_level, n, crit, flags, shift):
    import cv2
    a = _image(h, w, seed, kind)
    b = np.roll(a, shift, axis=(0, 1))
    rng = np.random.default_rng(seed + 1)
    p = np.stack([rng.uniform(-8, w + 8, n), rng.uniform(-8, h + 8, n)], -1).astype(np.float32).reshape(-1, 1, 2)
    init = (p + rng.normal(0, 1.5, p.shape)).astype(np.float32) if flags == 4 else None
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None if init is None else init.copy(), winSize=win, maxLevel=max_level, criteria=crit, flags=flags)
    got = klt.calcOpticalFlowPyrLK(a, b, p, init, winSize=win, maxLevel=max_level, criteria=crit, flags=flags)
    assert_lk_equal(got, ref, "h=%d w=%d win=%s lvl=%d flags=%d" % (h, w, win, max_level, flags))


@settings(**SETTINGS)
@given(h=st.integers(1, 150), w=st.integers(1, 300), seed=st.integers(0, 10 ** 6), levels=st.integers(1, 4))
def test_pyramid_equals_cv2_on_random_shapes(klt, h, w, seed, levels):
    import cv2
    a = _image(h, w, seed, 0)
    top, got = klt.buildOpticalFlowPyramid(a, (3, 3), levels)
    ref = a
    assert np.array_equal(got[0], a)
    for l in range(1, top + 1):
        ref = cv2.pyrDown(ref)
        assert np.array_equal(got[l], ref), (h, w, l)


@settings(max_examples=80, deadline=None, derandomize=True)
@given(h=st.integers(40, 160), w=st.integers(40, 220), seed=st.integers(0, 10 ** 6), kind=st.integers(0, 4),
       block=st.sampled_from([1, 2, 3, 4, 5, 6, 15, 31]), max_corners=st.sampled_from([0, 10, 1000]), q=st.sampled_from([0.01, 0.03, 0.2]),
       min_dist=st.sampled_from([0.0, 1.0, 7.5, 10.0]), masked=st.booleans())
def test_good_features_equals_cv2_on_random_inputs(klt, h, w, seed, kind, block, max_corners, q, min_dist, masked):
    import cv2
    a = _image(h, w, seed, kind)
    mask = None
    if masked:
        mask = np.full((h, w), 255, np.uint8)
        mask[h // 4: h // 2, w // 3: 2 * w // 3] = 0
    ref = cv2.goodFeaturesToTrack(a, max_corners, q, min_dist, mask=mask, blockSize=block)
    got = klt.goodFeaturesToTrack(a, max_corners, q, min_dist, mask=mask, blockSize=block)
    assert (ref is None) == (got is None)
    if ref is not None:
        assert got.shape == ref.shape and np.array_equal(got, ref), (h, w, block, max_corners, q, min_dist)


@settings(max_examples=80, deadline=None, derandomize=True)
@given(h=st.integers(5, 150), w=st.integers(5, 260), seed=st.integers(0, 10 ** 6), kind=st.integers(0, 4),
       params=st.sampled_from([(5, 1.5, 1.5), (3, 12.0, 1.0), (9, 30.0, 4.0), (0, 5.0, 1.1)]))
def test_bilateral_equals_the_oracle_on_random_inputs(klt, oracle, h, w, seed, kind, params):
    a = _image(h, w, seed, kind)
    d, sc, ss = params
    assert np.array_equal(klt.bilateralFilter(a, d, sc, ss), oracle.bilateral_filter(a, d, sc, ss)), (h, w, params)
