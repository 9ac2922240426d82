"""GPU tier for BASELINE configs[2]: the drop-in behind the reference's own call sequence.

The reference sources are not part of the repository, so the calls are replayed from tests/golden/pipeline_trace.npz (every
cv2.calcOpticalFlowPyrLK call of the unmodified Pipeline.step / Extractor.extend_tracks / extend_landmarks on the synthetic
sequence, recorded by tests/golden/make_pipeline_trace.py and re-derived from the reference in tests/test_pipeline_trace.py).
The drop-in is injected the way INTEGRATION.md s3 does it -- `cv2.calcOpticalFlowPyrLK = klt.calcOpticalFlowPyrLK` -- and
called through the cv2 attribute with the reference's positional / keyword arguments.  Where the reference sources are
given (VO_REFERENCE_SRC), the live test runs Pipeline.step() itself on the drop-in."""
import numpy as np
import pytest

import ref_harness as H
from conftest import assert_lk_equal, load_golden

pytestmark = pytest.mark.gpu
LK = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))   # reference src/extractor/extractor.py:16-19


@pytest.fixture(scope="module")
def injected(klt):
    import cv2
    real = cv2.calcOpticalFlowPyrLK
    cv2.calcOpticalFlowPyrLK = klt.calcOpticalFlowPyrLK
    yield cv2
    cv2.calcOpticalFlowPyrLK = real


def test_reference_call_sequence_replayed_through_the_injected_dropin(klt, injected):
    cv2 = injected
    tr = load_golden("pipeline_trace")
    loader = H.SyntheticLoader(int(tr["shape"][0]), int(tr["shape"][1]), n_frames=int(tr["n_frames"]))
    n = int(tr["n_calls"])
    points = 0
    for k in range(n):
        t0, t1 = (int(v) for v in tr["c%d_t" % k])
        im0, im1 = loader.getImage(t0), loader.getImage(t1).copy()      # pipeline.py:103 hands over a copy
        assert H.frame_crc(im0) == int(tr["frame_crc"][t0]) and H.frame_crc(im1) == int(tr["frame_crc"][t1])
        p0 = tr["c%d_p0" % k]
        p1, _st, _err = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **LK)            # extractor.py:44 / :65, verbatim call form
        assert isinstance(p1, np.ndarray) and p1.shape == p0.shape and p1.dtype == np.float32
        assert_lk_equal((p1, _st, _err), (tr["c%d_q" % k], tr["c%d_st" % k], tr["c%d_err" % k]), "call %d" % k)
        if k % 2 == 1:
            # what the reference computes from the couple (extractor.py:46-53): same survivors as with cv2
            pa, pr = tr["c%d_p0" % (k - 1)], p1
            d = abs(pa - pr).reshape(-1, 2).max(-1)
            dref = abs(pa - tr["c%d_q" % k]).reshape(-1, 2).max(-1)
            assert np.array_equal(d < np.inf, dref < np.inf)
        points += p0.shape[0]
    assert points > 20000


@pytest.mark.skipif(not H.reference_available(), reason=H.REFERENCE_MISSING)
def test_unmodified_reference_pipeline_on_the_dropin(klt):
    """Pipeline.step() (pipeline.py:92-167) with cv2 and with the drop-in: identical keypoints every frame."""
    loader = H.SyntheticLoader(480, 640, n_frames=14)
    a = H.run_reference_pipeline(4, loader=loader)
    b = H.run_reference_pipeline(4, loader=loader, lk_impl=klt.calcOpticalFlowPyrLK)
    assert len(a["calls"]) == len(b["calls"]) == 16
    for x, y in zip(a["calls"], b["calls"]):
        assert_lk_equal((y["q"], y["st"], y["err"]), (x["q"], x["st"], x["err"]))
    for sa, sb in zip(a["per_step"], b["per_step"]):
        assert np.array_equal(sa["landmark_uv"], sb["landmark_uv"]) and np.array_equal(sa["landmark_hist_len"], sb["landmark_hist_len"])
