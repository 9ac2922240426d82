"""CPU tier for BASELINE configs[2] (the reference's own Pipeline / Extractor code at the LK boundary):
tests/golden/pipeline_trace.npz holds every cv2.calcOpticalFlowPyrLK call the unmodified reference made on the synthetic
sequence of tests/ref_harness.py.  Here: (1) the renderer reproduces the sequence byte for byte, (2) where the reference
sources are given (VO_REFERENCE_SRC) the trace is re-derived from a fresh run of the reference's code,
(3) the C oracle reproduces what cv2 returned to the reference."""
import numpy as np
import pytest

import ref_harness as H
from conftest import assert_lk_equal, load_golden

LK = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))   # reference src/extractor/extractor.py:16-19


@pytest.fixture(scope="module")
def trace():
    return load_golden("pipeline_trace")


@pytest.fixture(scope="module")
def loader(trace):
    return H.SyntheticLoader(int(trace["shape"][0]), int(trace["shape"][1]), n_frames=int(trace["n_frames"]))


def test_renderer_reproduces_the_traced_frames(trace, loader):
    used = sorted({int(t) for k in range(int(trace["n_calls"])) for t in trace["c%d_t" % k]})
    for t in used:
        assert H.frame_crc(loader.getImage(t)) == int(trace["frame_crc"][t]), "frame %d renders differently on this machine" % t


def test_trace_structure_is_the_references_call_pattern(trace):
    """extend_tracks (extractor.py:44,45) then extend_landmarks (:65,66): 4 calls per frame on the same image pair, the
    second of each couple started from the first one's result."""
    n = int(trace["n_calls"])
    assert n == 4 * int(trace["n_steps"])
    for k in range(0, n, 2):
        assert np.array_equal(trace["c%d_t" % k], trace["c%d_t" % (k + 1)])
        assert np.array_equal(trace["c%d_q" % k].view(np.uint32), trace["c%d_p0" % (k + 1)].view(np.uint32))
    for k in range(0, n, 4):
        assert np.array_equal(trace["c%d_t" % k], trace["c%d_t" % (k + 2)])
        t0, t1 = trace["c%d_t" % k]
        assert t1 == t0 + 1                       # pipeline.py:94,103: im becomes im_prev


@pytest.mark.skipif(not H.reference_available(), reason=H.REFERENCE_MISSING)
def test_trace_is_what_the_unmodified_reference_does(trace, loader):
    run = H.run_reference_pipeline(2, loader=loader)
    assert len(run["calls"]) == 8
    for k, c in enumerate(run["calls"]):
        assert c["kw"] == LK
        assert np.array_equal(c["p0"].astype(np.float32).view(np.uint32), trace["c%d_p0" % k].view(np.uint32)), "inputs of call %d" % k
        assert_lk_equal((c["q"], c["st"], c["err"]), (trace["c%d_q" % k], trace["c%d_st" % k], trace["c%d_err" % k]), "call %d" % k)
    for s in range(2):
        assert np.array_equal(run["per_step"][s]["landmark_uv"], trace["s%d_landmark_uv" % s])


def test_oracle_reproduces_what_cv2_returned_to_the_reference(trace, loader, oracle):
    for k in (0, 2, 9, 18):
        t0, t1 = (int(v) for v in trace["c%d_t" % k])
        got = oracle.calc_optical_flow_pyr_lk(loader.getImage(t0), loader.getImage(t1), trace["c%d_p0" % k], None, LK["winSize"], LK["maxLevel"],
                                              LK["criteria"])
        assert_lk_equal(got, (trace["c%d_q" % k], trace["c%d_st" % k], trace["c%d_err" % k]), "call %d" % k)
