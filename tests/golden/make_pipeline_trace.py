"""Generates tests/golden/pipeline_trace.npz: every cv2.calcOpticalFlowPyrLK call the UNMODIFIED reference pipeline
(src/pipeline/pipeline.py:92-167 -> src/extractor/extractor.py:38-88) makes on the synthetic sequence of
tests/ref_harness.py, with its inputs and what the cv2 wheel returned.  Needs a checkout of the reference:

    VO_REFERENCE_SRC=<reference checkout>/src python tests/golden/make_pipeline_trace.py [n_steps]

The GPU tier replays these calls through the drop-in (tests/test_gpu_pipeline.py); the CPU tier re-runs the reference and
checks that the committed trace is still what its code produces (tests/test_pipeline_trace.py)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import ref_harness as H  # noqa: E402

N_STEPS = int(sys.argv[1]) if len(sys.argv) > 1 else 6
SHAPE = (480, 640)


def main():
    import cv2
    loader = H.SyntheticLoader(SHAPE[0], SHAPE[1], n_frames=N_STEPS + 8)
    run = H.run_reference_pipeline(N_STEPS, loader=loader)
    crc_to_t = {H.frame_crc(loader.getImage(t)): t for t in range(len(loader))}
    out = {"shape": np.array(SHAPE), "n_frames": np.array(len(loader)), "n_steps": np.array(N_STEPS), "n_calls": np.array(len(run["calls"])),
           "cv2_version": np.array(cv2.__version__), "frame_crc": np.array([H.frame_crc(loader.getImage(t)) for t in range(len(loader))], np.uint32)}
    for k, c in enumerate(run["calls"]):
        assert c["kw"] == {"winSize": (31, 31), "maxLevel": 3, "criteria": (3, 30, 0.03)}, c["kw"]   # extractor.py:16-19
        out["c%d_t" % k] = np.array([crc_to_t[c["crc0"]], crc_to_t[c["crc1"]]])
        out["c%d_p0" % k] = c["p0"].astype(np.float32)
        out["c%d_q" % k] = c["q"]
        out["c%d_st" % k] = c["st"]
        out["c%d_err" % k] = c["err"]
    for s, ps in enumerate(run["per_step"]):
        out["s%d_landmark_uv" % s] = ps["landmark_uv"]
        out["s%d_counts" % s] = np.array([ps["n_candidates"], ps["n_landmarks"]])
    path = os.path.join(HERE, "pipeline_trace.npz")
    np.savez_compressed(path, **out)
    n_pts = sum(c["p0"].shape[0] for c in run["calls"])
    print("wrote %s: %d steps, %d calls, %d points, %.0f KB; LK share of the reference's step time %.1f %% (%.3f of %.2f s)"
          % (path, N_STEPS, len(run["calls"]), n_pts, os.path.getsize(path) / 1e3, 100 * run["lk_seconds"] / sum(run["step_seconds"]),
             run["lk_seconds"], sum(run["step_seconds"])))


if __name__ == "__main__":
    main()
