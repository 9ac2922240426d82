#!/usr/bin/env python
"""bench.py -- KLT tracking hot path (pyramid build + pyramidal Lucas-Kanade) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload kitti|...|malaga_seq]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic frame pair of the workload: build both
Gaussian pyramids and track all keypoints coarse-to-fine (what the reference does inside ONE
cv2.calcOpticalFlowPyrLK call, src/extractor/extractor.py:44).  Default workload = BASELINE.json
configs[1]: KITTI-shape 1241x376, 2000 keypoints, winSize 21, maxLevel 3.

Printed JSON line (rank 0):
  value          tracked keypoints/s with inputs resident in HBM: exactly K timed steps after W warm-up steps (CUDA
                 events on the launching stream, barrier + synchronize on both sides, max over ranks);
  e2e            the same metric through the public drop-in `calcOpticalFlowPyrLK(numpy...)` with PINNED host buffers,
                 H2D + D2H inside the timed region; e2e_pageable: the same with ordinary (pageable) numpy arrays, which is
                 what the un-edited reference hands over (loader.py:86, pipeline.py:103);
  roofline       the HBM-bound kernel of the path (pyrDown, BASELINE `metric`: "pyramid HBM GB/s vs peak") on a batch larger
                 than L2, against MEASURED_PEAKS.json; lk_roofline: the dominant kernel of the step (LK) against the
                 resource it uses (int32 multiply-add issue), computed from this run;
  sharded_batch  BASELINE configs[3]: 256 independent KITTI-shape sequences block-partitioned over the ranks, one batched
                 pyramid build + one batched LK launch per rank and frame, results gathered in sequence order and a sample
                 bit-compared with cv2 on rank 0;
  cpu_baseline   cv2 (the reference's own implementation of the path) on this box's host cores.
`--impl reference` times only that cv2 path.  `--workload malaga_seq` = BASELINE configs[2]: the reference's per-frame call
sequence (4 LK calls on the frame pair + its numpy filters) over a 500-frame Malaga-shape sequence through the injected
drop-in.

`--dump-outputs DIR` (frame-pair workloads) writes what the last timed step of rank 0 handed its caller, as float32 .npy
files: next_pts (N, 2), status (N,), err (N,) and both pyramids, {prev,next}_pyramid_level<l> (h_l, w_l) for l >= 1.  The
inputs depend only on the arguments, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import ctypes
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs; criteria = cv2 defaults unless the config is the reference's own parameters
    "parking": dict(idx=0, h=480, w=640, n=500, win=(21, 21), max_level=3, criteria=(3, 30, 0.01)),
    "kitti": dict(idx=1, h=376, w=1241, n=2000, win=(21, 21), max_level=3, criteria=(3, 30, 0.01)),
    "kitti_ref_params": dict(idx=1, h=376, w=1241, n=2000, win=(31, 31), max_level=3, criteria=(3, 30, 0.03)),
    "malaga": dict(idx=2, h=768, w=1024, n=3000, win=(21, 21), max_level=3, criteria=(3, 30, 0.01)),
    "malaga_seq": dict(idx=2, h=768, w=1024, n=3000, win=(31, 31), max_level=3, criteria=(3, 30, 0.03), frames=500),
    "stress4k": dict(idx=4, h=2160, w=3840, n=100014, win=(31, 31), max_level=5, criteria=(3, 30, 0.01)),
}
L2_BYTES = 126 * 1024 * 1024
INT32_LANES_PER_SM = 128   # lanes an SM can issue integer multiply-adds on per clock (4 sub-partitions x 32)


def describe(wl_name, wl):
    if wl_name == "malaga_seq":
        return ("configs[2] malaga_seq: %dx%d synthetic sequence of %d frames, %d keypoints tracked frame to frame with the "
                "reference's call sequence (extractor.py:38-88: 4 calcOpticalFlowPyrLK calls per frame, winSize %d, maxLevel %d, "
                "criteria %s)" % (wl["w"], wl["h"], wl["frames"], wl["n"], wl["win"][0], wl["max_level"], tuple(wl["criteria"])))
    return ("configs[%d] %s: %dx%d frame pair, %d keypoints, winSize %d, maxLevel %d, criteria %s"
            % (wl["idx"], wl_name, wl["w"], wl["h"], wl["n"], wl["win"][0], wl["max_level"], tuple(wl["criteria"])))


class HostPool(list):
    """list of (prev, next, pts) host triples + `crop(i, extra_off)`: entry i moved `extra_off` more columns along its canvas"""
    crop = None


LEGACY_ROLL_POOL = False    # --legacy-roll-pool: the cyclic-shift pool of rounds 1-2, kept so that their numbers can be reproduced


def host_pool(wl, count, seed0, max_extra_off=0):
    """`count` distinct (prev, next, pts) host triples.  A few wide base pairs are synthesised with the SURVEY s8d generator
    (texture + affine warp) and every entry is a CROP of one of them at its own column offset: distinct bytes at distinct
    addresses for the cache behaviour, a different motion field per entry (the warp is about the canvas centre), and no
    seam.  (Rounds 1-2 used cyclic shifts: np.roll puts a motion discontinuity inside the image, and the windows that
    straddle it ran 60-77 iterations against 42 for the worst point of an unshifted pair -- the tail of every launch was
    an artefact of the generator.)"""
    from visual_odom_pipeline_b200 import synth as S
    h, w, n = wl["h"], wl["w"], wl["n"]
    n_base = min(count, 4)
    step = 37
    per = -(-count // n_base)
    canv = [S.frame_pair(h, w if LEGACY_ROLL_POOL else w + (per - 1) * step + max_extra_off, seed=seed0 + i) for i in range(n_base)]

    def crop(i, extra_off=0):
        a, b = canv[i % n_base]
        off = (i // n_base) * step + extra_off
        if LEGACY_ROLL_POOL:
            return np.ascontiguousarray(np.roll(a, off, axis=1)), np.ascontiguousarray(np.roll(b, off, axis=1))
        return np.ascontiguousarray(a[:, off:off + w]), np.ascontiguousarray(b[:, off:off + w])

    pool = HostPool()
    pool.crop = crop
    for i in range(count):
        a, b = crop(i)
        if wl["n"] == 100014:
            p = S.grid_points(422, 237, h, w)
        else:
            p = S.uniform_points(n, h, w, seed=seed0 + 1000 + i)
        pool.append((a, b, p))
    return pool


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(device_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            busy = [s for s in sm if s >= 0.5 * max(sm)]
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def csrc_sha16():
    """Hash of the kernel sources: profiler figures are only quoted when they were captured on the same sources."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "visual-odom-pipeline_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh")):
            with open(os.path.join(d, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def ncu_counters(report, pick_largest_grid=False):
    """Counters of the committed ncu capture of a kernel (profiles/r02/counters.json, written by
    scripts/summarize_profiles.py from `ncu --set full` runs of scripts/prof_target.py).  Returned only when the capture was
    made on the kernel sources of this checkout (csrc_sha16); profiler figures, labelled as such -- never timings of this run."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02", "counters.json")) as f:
            doc = json.load(f)
        if doc.get("csrc_sha16") != csrc_sha16():
            return None
        rows = doc.get(report) or []
        if not rows:
            return None

        def grid_size(r):
            try:
                return int(str(r.get("grid", "0")).strip("() ").split(",")[0])
            except ValueError:
                return 0
        return max(rows, key=grid_size) if pick_largest_grid else rows[-1]
    except Exception:
        return None


def time_cv2(wl, pool, reps, warm, threads=None):
    import cv2
    if threads is not None:
        cv2.setNumThreads(threads)
    lk = dict(winSize=wl["win"], maxLevel=wl["max_level"], criteria=wl["criteria"])
    for i in range(warm):
        a, b, p = pool[i % len(pool)]
        cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk)
    ts = []
    for i in range(reps):
        a, b, p = pool[i % len(pool)]
        t = time.perf_counter()
        cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk)
        ts.append(time.perf_counter() - t)
    return ts


# ------------------------------------------------------------------------------------------------------------------
# BASELINE configs[2]: the reference's per-frame call sequence on a sequence
# ------------------------------------------------------------------------------------------------------------------
def reference_tracking_step(lk_fn, im_prev, im, tracks, landmarks, lk_params, w, h, max_bidir_error=30):
    """What Pipeline.step hands to the extractor per frame (reference src/pipeline/pipeline.py:98-103) and what
    Extractor.extend_tracks / extend_landmarks do with it (src/extractor/extractor.py:38-88), restated: two LK calls per
    point set on the same image pair, the bidirectional-error test and the inclusive bounds test in numpy.
    -> (surviving tracks, surviving landmarks, seconds spent inside the 4 LK calls)"""
    t_lk = 0.0
    out = []
    for p0 in (tracks, landmarks):
        if p0.shape[0] == 0:
            out.append(p0)
            continue
        t = time.perf_counter()
        p1, _st, _err = lk_fn(im_prev, im, p0, None, **lk_params)          # extractor.py:44 / :65
        p0r, _st, _err = lk_fn(im_prev, im, p1, None, **lk_params)         # extractor.py:45 / :66
        t_lk += time.perf_counter() - t
        d = abs(p0 - p0r).reshape(-1, 2).max(-1)                           # extractor.py:46 / :67
        good = d < max_bidir_error                                         # :47 / :68
        q = p1.reshape(-1, 2)
        inb = (0 <= q[:, 0]) & (q[:, 0] <= w) & (0 <= q[:, 1]) & (q[:, 1] <= h)   # :53 / :75
        out.append(p1[good & inb])
    return out[0], out[1], t_lk


def run_malaga_seq(args, wl_name, wl):
    import torch
    import cv2
    import visual_odom_pipeline_b200 as K
    from visual_odom_pipeline_b200 import sharding, synth as S
    rank, local_rank, world = sharding.init_process_group()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    ctx = K.default_context(local_rank)
    h, w, n, n_frames = wl["h"], wl["w"], wl["n"], wl["frames"]
    lkp = dict(winSize=wl["win"], maxLevel=wl["max_level"], criteria=wl["criteria"])
    # 500 distinct frames: a base sequence of 25 wide frames (each a small warp of the previous one), replayed forwards
    # and backwards, every replay cropped 29 columns further along the canvas (distinct bytes, no seam: see host_pool)
    order = list(range(25)) + list(range(23, 0, -1))
    base = S.sequence(h, w + (n_frames // len(order) + 1) * 29, 25, seed=21 + rank)

    def frame(i):
        f = base[order[i % len(order)]]
        sh = (i // len(order)) * 29
        return f[:, sh:sh + w]

    def fresh_points(seed):
        p = S.uniform_points(n, h, w, seed=seed).astype(np.float32)
        return p[: n // 3].copy(), p[n // 3:].copy()        # candidate tracks, landmark keypoints

    def run(lk_fn, frames_to_run, replenish=True):
        tracks, landmarks = fresh_points(5)
        im_prev = frame(0).copy()
        t_lk = t_all = 0.0
        tracked = 0
        for i in range(1, frames_to_run + 1):
            im = frame(i).copy()                              # pipeline.py:103 hands over a copy (pageable numpy)
            tracked += tracks.shape[0] + landmarks.shape[0]
            t = time.perf_counter()
            tracks, landmarks, dt = reference_tracking_step(lk_fn, im_prev, im, tracks, landmarks, lkp, w, h)
            t_all += time.perf_counter() - t
            t_lk += dt
            if replenish and tracks.shape[0] + landmarks.shape[0] < 0.9 * n:
                # the reference re-detects features every frame (pipeline.py:159-163); here lost points are replaced by
                # fresh uniform ones so that the tracked count stays at the config's 3000
                ft, fl = fresh_points(1000 + i)
                tracks = np.concatenate([tracks, ft[: n // 3 - tracks.shape[0]]]) if tracks.shape[0] < n // 3 else tracks
                landmarks = np.concatenate([landmarks, fl[: n - n // 3 - landmarks.shape[0]]]) if landmarks.shape[0] < n - n // 3 else landmarks
            im_prev = im
        return t_lk, t_all, tracked, tracks, landmarks

    lk_b200 = lambda *a, **k: K.calcOpticalFlowPyrLK(*a, device=local_rank, **k)   # noqa: E731
    run(lk_b200, 5)
    sharding.barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_lk, t_all, tracked, tr_b, lm_b = run(lk_b200, n_frames)
    t_lk = sharding.max_over_ranks(t_lk)
    t_all = sharding.max_over_ranks(t_all)
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        # the same sequence of calls with cv2 on a bounded sample of frames, and a parity check of the survivors
        n_cpu = max(3, min(40, args.steps))
        c_lk, c_all, c_tracked, tr_c, lm_c = run(cv2.calcOpticalFlowPyrLK, n_cpu)
        _, _, _, tr_g, lm_g = run(lk_b200, n_cpu)
        parity = bool(np.array_equal(tr_c.view(np.uint32), tr_g.view(np.uint32)) and np.array_equal(lm_c.view(np.uint32), lm_g.view(np.uint32)))
        value = world * tracked / t_lk
        line = {
            "metric": "tracked_keypoints_per_sec", "value": value, "unit": "keypoints/s", "n_gpus": world, "steps": n_frames,
            "warmup": 5, "ms_per_step": 1e3 * t_lk / n_frames, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": describe(wl_name, wl),
                       "sharding": "each rank runs its own sequence; no collective on the data path"},
            "frames": n_frames, "keypoints_tracked": tracked,
            "lk_boundary_ms_per_frame": 1e3 * t_lk / n_frames,
            "tracking_step_ms_per_frame": 1e3 * t_all / n_frames,
            "note": "value = keypoints entering the frame's tracking step / time inside the 4 injected LK calls (pageable numpy in, "
                    "numpy out); tracking_step adds the reference's numpy filters.  Pose estimation, triangulation and bundle "
                    "adjustment (the rest of Pipeline.step) are not on this path and not timed here.",
            "e2e": {"value": value, "unit": "keypoints/s", "h2d_bytes_per_step": 4 * (2 * w * h) + 2 * n * 8, "d2h_bytes_per_step": 2 * n * 13,
                    "api": "cv2.calcOpticalFlowPyrLK = visual_odom_pipeline_b200.calcOpticalFlowPyrLK (INTEGRATION.md s3), pageable numpy arrays"},
            "gpu_launches": n_frames * 4 * 3,
            "clocks": clocks,
            "cpu_baseline": {"value": c_tracked / c_lk, "unit": "keypoints/s", "cores": cv2.getNumThreads(), "kind": "reference",
                             "sample": "the same call sequence with cv2 %s on the first %d frames: %.2f ms inside the LK calls per frame, "
                                       "%.2f ms per tracking step" % (cv2.__version__, n_cpu, 1e3 * c_lk / n_cpu, 1e3 * c_all / n_cpu)},
            "parity": {"survivors_identical_to_cv2_after_%d_frames" % n_cpu: parity},
            "device": ctx.name,
        }
        print(json.dumps(line), flush=True)
    sharding.barrier()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


def run_reference(args, wl_name, wl):
    """--impl reference: the reference's own CPU implementation of the path (cv2.calcOpticalFlowPyrLK as
    called at src/extractor/extractor.py:44) on this box's host cores, all threads OpenCV will use."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import cv2
    if wl_name == "malaga_seq":
        wl = dict(wl)
    pool = host_pool(wl, 8, seed0=7)
    per_call = time_cv2(wl, pool, 3, 2)
    est = statistics.median(per_call)
    steps = max(1, min(args.steps, int(60.0 / max(est, 1e-6))))   # bounded: at most ~1 min of CPU work
    ts = time_cv2(wl, pool, steps, args.warmup)
    total = sum(ts)
    value = wl["n"] * steps / total
    line = {
        "impl": "reference", "metric": "tracked_keypoints_per_sec", "value": value, "unit": "keypoints/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": describe(wl_name, wl)},
        "pairs_per_sec": steps / total,
        "cpu_baseline": {"value": value, "unit": "keypoints/s", "cores": cv2.getNumThreads(), "kind": "reference",
                         "sample": "%d cv2.calcOpticalFlowPyrLK calls (cv2 %s, %d OpenCV threads, os.cpu_count()=%s), median %.3f ms, min %.3f ms"
                                   % (steps, cv2.__version__, cv2.getNumThreads(), os.cpu_count(), 1e3 * statistics.median(ts), 1e3 * min(ts))},
        "e2e": {"value": value, "unit": "keypoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="kitti", choices=sorted(WORKLOADS))
    ap.add_argument("--pool", type=int, default=0, help="distinct device-resident pairs (0 = enough to exceed L2)")
    ap.add_argument("--legacy-roll-pool", action="store_true",
                    help="build the pool from cyclic column shifts as rounds 1-2 did (seam inside every shifted image); default: crops of wide canvases")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-detection", action="store_true", help="skip the Shi-Tomasi detection section (SURVEY s8f rank 2)")
    ap.add_argument("--no-sharded-batch", action="store_true", help="skip the configs[3] section (256 sharded sequences)")
    ap.add_argument("--sequences", type=int, default=256, help="configs[3]: independent sequences over all ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    global LEGACY_ROLL_POOL
    LEGACY_ROLL_POOL = bool(args.legacy_roll_pool)
    wl_name, wl = args.workload, WORKLOADS[args.workload]
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or wl_name == "malaga_seq"):
        ap.error("--dump-outputs covers the frame-pair workloads of --impl b200")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args, wl_name, wl)
    if wl_name == "malaga_seq":
        return run_malaga_seq(args, wl_name, wl)

    import torch
    import visual_odom_pipeline_b200 as K
    from visual_odom_pipeline_b200 import _lib, sharding
    from visual_odom_pipeline_b200.lk import make_params

    rank, local_rank, world = sharding.init_process_group()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    host_cores = [] if os.environ.get("KLT_NO_BIND") else sharding.bind_rank_to_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    dev = torch.device("cuda", local_rank)
    ctx = K.default_context(local_rank)
    L = _lib.load()
    stream = torch.cuda.current_stream(dev)
    sptr = ctypes.c_void_p(stream.cuda_stream)
    h, w, n = wl["h"], wl["w"], wl["n"]
    win, max_level = wl["win"], wl["max_level"]
    params = make_params(win, wl["criteria"], 0, 1e-4)
    K_steps = args.steps

    # ---- device-resident pool of distinct pairs, larger than L2 (no flush needed between steps) --------
    # ONE batched pyramid: item 2i = prev frame of pair i, item 2i+1 = its next frame.
    pitch = (w + 127) // 128 * 128
    lay1 = _lib.klt_pyr_layout()
    assert L.klt_pyr_plan(w, h, win[0], win[1], max_level, 1, ctypes.byref(lay1)) == 0
    pair_bytes = 2 * (pitch * h + int(lay1.bytes))
    P = args.pool or max(8, -(-int(1.5 * L2_BYTES) // pair_bytes))
    P = min(P, 1024)
    layB = _lib.klt_pyr_layout()
    assert L.klt_pyr_plan(w, h, win[0], win[1], max_level, 2 * P, ctypes.byref(layB)) == 0
    layB.level[0].pitch = pitch
    layB.level[0].batch_stride = pitch * h
    n_host = min(P, 16)
    dev_step = 53                                    # device entry i = host entry i % n_host, dev_step * (i // n_host) columns further
    hp = host_pool(wl, n_host, seed0=7 + 100 * rank, max_extra_off=((P - 1) // n_host) * dev_step)
    imgs = torch.empty((2 * P, h, pitch), dtype=torch.uint8, device=dev)
    pyrs = torch.empty(max(int(layB.bytes), 1), dtype=torch.uint8, device=dev)
    pts = torch.empty((P, n, 2), dtype=torch.float32, device=dev)
    for i in range(P):
        a, b = hp.crop(i % n_host, (i // n_host) * dev_step)
        p = hp[i % n_host][2]
        imgs[2 * i, :, :w].copy_(torch.from_numpy(a))
        imgs[2 * i + 1, :, :w].copy_(torch.from_numpy(b))
        pts[i].copy_(torch.from_numpy(p.reshape(n, 2)))
    out_q = torch.empty((P, n, 2), dtype=torch.float32, device=dev)
    out_s = torch.empty((P, n), dtype=torch.uint8, device=dev)
    out_e = torch.empty((P, n), dtype=torch.float32, device=dev)
    iters = torch.zeros((P, n), dtype=torch.int32, device=dev)
    img0, pyr0, pts0 = imgs.data_ptr(), pyrs.data_ptr(), pts.data_ptr()
    q0, s0, e0, it0 = out_q.data_ptr(), out_s.data_ptr(), out_e.data_ptr(), iters.data_ptr()
    h_ctx = ctx.handle
    layB_ref, params_ref = ctypes.byref(layB), ctypes.byref(params)

    def pyr_step(i):
        rc = L.klt_pyr_build(h_ctx, img0, layB_ref, pyr0, 2 * i, 2, sptr)
        assert rc == 0, _lib.status_string(rc)

    def lk_step(i, want_iters=False):
        rc = L.klt_lk_track(h_ctx, img0, pyr0, img0, pyr0, layB_ref, 2 * i, 2 * i + 1, 2, 1, pts0 + i * n * 8, q0 + i * n * 8,
                            s0 + i * n, e0 + i * n * 4, (it0 + i * n * 4) if want_iters else None, n, params_ref, sptr)
        assert rc == 0, _lib.status_string(rc)

    def step(i):
        pyr_step(i)
        lk_step(i)

    # kernels launched per step: the pyramid is one launch for all levels of both images when it has >= 2 levels built
    # (pyr_build_fused_kernel), else one launch per level; LK is one launch
    pyr_launches = 1 if int(layB.top) >= 2 else int(layB.top)
    launches_per_step = pyr_launches + 1

    def step_outputs(i):
        """What step(i) hands its caller, copied to the host as float32: nextPts / status / err and both pyramids."""
        out = {"next_pts": out_q[i], "status": out_s[i], "err": out_e[i]}
        for l in range(1, int(layB.top) + 1):
            lv = layB.level[l]
            for item, name in ((2 * i, "prev"), (2 * i + 1, "next")):
                base = lv.offset + item * lv.batch_stride
                out["%s_pyramid_level%d" % (name, l)] = pyrs[base:base + lv.h * lv.pitch].view(lv.h, lv.pitch)[:, :lv.w]
        return {k: v.float().cpu().numpy() for k, v in out.items()}

    # ---- headline: exactly K device-resident steps, right after the warm-up steps -------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    time.sleep(0.25)
    for s in range(args.warmup):
        step(s % P)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    sharding.barrier()
    ev0.record(stream)
    for s in range(K_steps):
        step((args.warmup + s) % P)
    ev1.record(stream)
    torch.cuda.synchronize()
    sharding.barrier()
    dev_ms = sharding.max_over_ranks(ev0.elapsed_time(ev1))
    value = world * n * K_steps / (dev_ms * 1e-3)
    # taken now: the sections below write the same pool entries again
    last_outputs = step_outputs((args.warmup + K_steps - 1) % P) if args.dump_outputs and rank == 0 else None

    # ---- the same steps pipelined over 4 streams: independent pairs overlap, the idle tail of one pair's LK launch is
    # filled by the next pair (throughput of a job of independent pairs; per-pair latency is the number above) -------
    n_str = 4
    side = [torch.cuda.Stream(device=dev) for _ in range(n_str)]
    sptrs = [ctypes.c_void_p(st_.cuda_stream) for st_ in side]
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pipe_steps = K_steps

    def step_on(i, sp):
        rc = L.klt_pyr_build(h_ctx, img0, layB_ref, pyr0, 2 * i, 2, sp)
        assert rc == 0, _lib.status_string(rc)
        rc = L.klt_lk_track(h_ctx, img0, pyr0, img0, pyr0, layB_ref, 2 * i, 2 * i + 1, 2, 1, pts0 + i * n * 8, q0 + i * n * 8,
                            s0 + i * n, e0 + i * n * 4, None, n, params_ref, sp)
        assert rc == 0, _lib.status_string(rc)

    for rep in range(2):      # first pass = warm-up
        torch.cuda.synchronize()
        sharding.barrier()
        pe0.record(stream)
        for st_ in side:
            st_.wait_event(pe0)
        for s_ in range(pipe_steps):
            step_on((args.warmup + s_) % P, sptrs[s_ % n_str])
        for st_ in side:
            ev = torch.cuda.Event()
            ev.record(st_)
            stream.wait_event(ev)
        pe1.record(stream)
        torch.cuda.synchronize()
    pipe_ms = sharding.max_over_ranks(pe0.elapsed_time(pe1))
    pipelined = {"streams": n_str, "steps": pipe_steps, "keypoints_per_sec": world * n * pipe_steps / (pipe_ms * 1e-3),
                 "pairs_per_sec": world * pipe_steps / (pipe_ms * 1e-3), "ms_per_step": pipe_ms / pipe_steps,
                 "note": "same steps, independent pairs issued round-robin on 4 streams"}

    # ---- per-kernel durations over the same steps (events on the launching stream) ---------------------------
    ksteps = K_steps
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(ksteps)]
    for s in range(ksteps):
        i = (args.warmup + s) % P
        evs[s][0].record(stream)
        pyr_step(i)
        evs[s][1].record(stream)
        lk_step(i, want_iters=True)
        evs[s][2].record(stream)
    torch.cuda.synchronize()
    pyr_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in evs)
    lk_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in evs)
    used = sorted(set((args.warmup + s) % P for s in range(ksteps)))
    it_mean = float(iters[used].float().mean().item())
    st_mean = float(out_s[used].float().mean().item())

    # ---- end to end through the public drop-in: host buffers in, numpy out -----------------------------------------
    hpin = []
    for (a, b, p) in hp:
        pa, pb, pp = K.pinned_empty(a.shape, np.uint8), K.pinned_empty(b.shape, np.uint8), K.pinned_empty(p.shape, np.float32)
        pa[...] = a; pb[...] = b; pp[...] = p
        hpin.append((pa, pb, pp))
    hpage = [(np.array(a), np.array(b), np.array(p)) for (a, b, p) in hp]     # ordinary numpy arrays (pageable)
    lk_kw = dict(winSize=win, maxLevel=max_level, criteria=wl["criteria"], device=local_rank)

    def e2e_seconds(bufs):
        for s in range(args.warmup):
            a, b, p = bufs[s % n_host]
            K.calcOpticalFlowPyrLK(a, b, p, None, **lk_kw)
        sharding.barrier()
        t0 = time.perf_counter()
        for s in range(K_steps):
            a, b, p = bufs[s % n_host]
            K.calcOpticalFlowPyrLK(a, b, p, None, **lk_kw)
        secs = sharding.max_over_ranks(time.perf_counter() - t0)
        sharding.barrier()
        return secs

    e2e_s = e2e_seconds(hpin)
    e2e_page_s = e2e_seconds(hpage)
    e2e_value = world * n * K_steps / e2e_s
    clocks = sampler.stop() if sampler else None

    # ---- BASELINE configs[3]: independent sequences block-partitioned over the ranks (every rank takes part) -------
    sharded = None
    if not args.no_sharded_batch and wl_name in ("kitti", "kitti_ref_params"):
        sharded = run_sharded_batch(args, wl, rank, local_rank, world, dev)

    line = None
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        sm_mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
        levels = int(layB.top) + 1
        # ---- LK: the dominant kernel of the step.  Its working set is L1/L2 resident, so the resource that bounds it is
        # integer multiply-add issue: MAC/pt = win^2 * (15 * levels + 7 * iterations + 6) (SURVEY.md s8d; iterations counted
        # by the kernel in this run) against sm_count * 128 lanes * f_sm (clock sampled during the timed region)
        mac_pt = win[0] * win[1] * (15 * levels + 7 * it_mean + 6)
        gmac = mac_pt * n / (lk_ms * 1e-3) / 1e9
        mac_peak = ctx.sm_count * INT32_LANES_PER_SM * sm_mhz * 1e6 / 1e9
        lk_bytes_pt = levels * (win[0] + 3) * (win[1] + 3) + it_mean * (win[0] + 1) * (win[1] + 1)
        c_lk = ncu_counters("prof_lk") if wl_name == "kitti" else None
        lk_roofline = {"kernel": "lk_fast_kernel (fused Scharr + pyramidal LK, all levels, 1 launch)", "bound": "int32_mac_issue",
                       "achieved": gmac, "peak": mac_peak, "unit": "GMAC/s", "frac": gmac / mac_peak,
                       "peak_formula": "%d SMs x %d int32 lanes x %.0f MHz (sampled under load)" % (ctx.sm_count, INT32_LANES_PER_SM, sm_mhz),
                       "launch_ms": lk_ms, "iters_per_point": it_mean, "int_mac_per_point": mac_pt,
                       "algorithmic_bytes_per_launch": lk_bytes_pt * n, "algorithmic_gbs": lk_bytes_pt * n / (lk_ms * 1e-3) / 1e9,
                       "traffic": (c_lk["dram_bytes_read"] + c_lk["dram_bytes_write"]) if c_lk else None,
                       "ncu": ({"source": "profiles/r02/counters.json (ncu --set full of the same launch shape on these kernel sources; profiler figures)",
                                "issue_slots_active_pct": c_lk["issue_active_pct"], "shared_mem_wavefronts_pct_of_peak": c_lk["smem_wavefronts_pct_of_peak"],
                                "sm_active_fraction_of_elapsed": (c_lk["sm_active_cycles_avg"] / c_lk["sm_elapsed_cycles_max"]) if c_lk.get("sm_elapsed_cycles_max") else None}
                               if c_lk else None),
                       "note": "working set is L2/L1-resident (DRAM traffic ~1.3 MB per launch): the kernel is issue/latency-bound, not HBM-bound"}

        # ---- the HBM-bound kernel: pyrDown over the whole pool (input larger than L2) ---------------------------
        nb = 2 * P
        l1 = layB.level[1] if layB.top >= 1 else None
        reps = 20
        pe = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(reps)]
        for r in range(3 + reps):
            k = r - 3
            if k >= 0:
                pe[k][0].record(stream)
            if l1 is not None:
                rc = L.klt_pyr_down(h_ctx, img0, w, h, pitch, pitch * h, pyr0 + l1.offset, l1.pitch, l1.batch_stride, nb, sptr)
                assert rc == 0
            if k >= 0:
                pe[k][1].record(stream)
            rc = L.klt_pyr_build(h_ctx, img0, layB_ref, pyr0, 0, 0, sptr)
            assert rc == 0
            if k >= 0:
                pe[k][2].record(stream)
        torch.cuda.synchronize()
        d01_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in pe)
        full_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in pe)
        b01 = nb * (w * h + ((w + 1) // 2) * ((h + 1) // 2))
        ball = 0
        for l in range(int(layB.top)):
            ball += nb * (layB.level[l].w * layB.level[l].h + layB.level[l + 1].w * layB.level[l + 1].h)
        c_pyr = ncu_counters("prof_pyr", True) if (w, h) == (1241, 376) else None
        roofline = {"kernel": "pyr_down_ring_kernel level 0->1, batch of %d images (%.0f MB read, > L2)" % (nb, nb * w * h / 1e6),
                    "bound": "hbm", "achieved": b01 / (d01_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": b01 / (d01_ms * 1e-3) / 1e9 / peak,
                    "traffic": (c_pyr["dram_bytes_read"] + c_pyr["dram_bytes_write"]) if c_pyr else None,
                    "traffic_note": "ncu dram__bytes_read+write of the same launch (310 KITTI images), profiles/r02/counters.json, quoted only when captured "
                                    "on these kernel sources; part of the output is still in L2 at kernel end",
                    "peak_source": peak_src, "launch_ms": d01_ms,
                    "algorithmic_bytes_per_launch": b01,
                    "whole_pyramid": {"levels_built": int(layB.top), "launches": pyr_launches, "ms": full_ms, "algorithmic_bytes": ball,
                                      "achieved": ball / (full_ms * 1e-3) / 1e9, "frac": ball / (full_ms * 1e-3) / 1e9 / peak}}

        # ---- batched LK throughput on this rank (all P independent pairs in ONE launch) --------------------------------
        be = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(3):
            if r == 2:
                be[0].record(stream)
            rc = L.klt_lk_track(h_ctx, img0, pyr0, img0, pyr0, layB_ref, 0, 1, 2, P, pts0, q0, s0, e0, None, n, params_ref, sptr)
            assert rc == 0, _lib.status_string(rc)
        be[1].record(stream)
        torch.cuda.synchronize()
        bms = be[0].elapsed_time(be[1])
        batched = {"pairs": P, "points": P * n, "ms": bms, "keypoints_per_sec": P * n / (bms * 1e-3), "pairs_per_sec": P / (bms * 1e-3),
                   "int32_mac_frac": (mac_pt * P * n / (bms * 1e-3) / 1e9) / mac_peak}

        # ---- one step recorded into a CUDA graph (pyramid build + LK of pool entry 0) and replayed: the device-pointer entry
        # points are plain launches once their scratch exists, the pyramid build switches to its device-side launch counter
        graph_replay = None
        try:
            gstream = torch.cuda.Stream(device=dev)
            gptr = ctypes.c_void_p(gstream.cuda_stream)
            gstream.wait_stream(stream)
            with torch.cuda.stream(gstream):
                for _ in range(2):       # scratch of this stream / geometry is allocated outside the capture
                    assert L.klt_pyr_build(h_ctx, img0, layB_ref, pyr0, 0, 2, gptr) == 0
                    assert L.klt_lk_track(h_ctx, img0, pyr0, img0, pyr0, layB_ref, 0, 1, 2, 1, pts0, q0, s0, e0, None, n, params_ref, gptr) == 0
            gstream.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=gstream):
                assert L.klt_pyr_build(h_ctx, img0, layB_ref, pyr0, 0, 2, gptr) == 0
                assert L.klt_lk_track(h_ctx, img0, pyr0, img0, pyr0, layB_ref, 0, 1, 2, 1, pts0, q0, s0, e0, None, n, params_ref, gptr) == 0
            greps = K_steps
            gev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            for _ in range(5):
                graph.replay()
            torch.cuda.synchronize()
            gev[0].record(torch.cuda.current_stream(dev))
            for _ in range(greps):
                graph.replay()
            gev[1].record(torch.cuda.current_stream(dev))
            torch.cuda.synchronize()
            first = out_q[0].clone()
            dev0 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            step(0)
            torch.cuda.synchronize()
            dev0[0].record(stream)
            for _ in range(greps):
                step(0)
            dev0[1].record(stream)
            torch.cuda.synchronize()
            graph_replay = {"ms_per_step": gev[0].elapsed_time(gev[1]) / greps, "replays": greps,
                            "direct_launches_same_pair_ms_per_step": dev0[0].elapsed_time(dev0[1]) / greps,
                            "identical_to_direct_launches": bool(torch.equal(first, out_q[0])),
                            "note": "pool entry 0 (one fixed pair, L2 resident): pyramid build + LK as one CUDA graph"}
        except Exception as ex:   # pragma: no cover
            graph_replay = {"error": repr(ex)}

        # ---- the generic kernel (any window other than 21x21 / 31x31): same pool, winSize 15x15 and 25x17 -----------------------
        generic = []
        for gwin in ((15, 15), (25, 17)):
            gparams = make_params(gwin, wl["criteria"], 0, 1e-4)
            ge = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            gpairs = min(P, 32)
            gq = torch.empty((gpairs, n, 2), dtype=torch.float32, device=dev)      # own outputs: the pool's are checked below
            gs = torch.empty((gpairs, n), dtype=torch.uint8, device=dev)
            gerr = torch.empty((gpairs, n), dtype=torch.float32, device=dev)
            for r in range(3):
                if r == 2:
                    ge[0].record(stream)
                rc = L.klt_lk_track(h_ctx, img0, pyr0, img0, pyr0, layB_ref, 0, 1, 2, gpairs, pts0, gq.data_ptr(), gs.data_ptr(), gerr.data_ptr(),
                                    None, n, ctypes.byref(gparams), sptr)
                assert rc == 0, _lib.status_string(rc)
            ge[1].record(stream)
            torch.cuda.synchronize()
            gms = ge[0].elapsed_time(ge[1])
            generic.append({"winSize": list(gwin), "pairs": gpairs, "points": gpairs * n, "ms": gms, "keypoints_per_sec": gpairs * n / (gms * 1e-3),
                            "kernel": "lk_kernel (klt_lk.cu: one warp per keypoint, runtime window geometry)"})

        detection = prefilter = None
        if not args.no_detection and h > 31 and w > 31:
            detection = run_detection(args, wl, K, L, hp, hpin, imgs, P, n_host, local_rank, world, dev, stream)
            prefilter = run_prefilter(args, wl, K, hp, imgs, P, local_rank, world, stream)

        # ---- parity spot check of pool entry used first, against live cv2 ------------------------------------
        parity = None
        try:
            import cv2
            i = args.warmup % P
            p = hp[i % n_host][2]
            a2, b2 = hp.crop(i % n_host, (i // n_host) * dev_step)
            rq, rs, re_ = cv2.calcOpticalFlowPyrLK(a2, b2, p, None, winSize=win, maxLevel=max_level,
                                                   criteria=wl["criteria"])
            gq, gs = out_q[i].cpu().numpy(), out_s[i].cpu().numpy()
            both = (rs.ravel() == 1) & (gs == 1)
            parity = {"points": int(n), "status_agree": float((rs.ravel() == gs).mean()),
                      "max_abs_diff_px": float(np.abs(rq.reshape(-1, 2)[both] - gq[both]).max()) if both.any() else 0.0,
                      "bit_exact": bool(np.array_equal(rq.reshape(-1, 2).view(np.uint32), gq.view(np.uint32)))}
        except Exception as ex:   # pragma: no cover
            parity = {"error": repr(ex)}

        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            import cv2
            hp_cpu = [(np.array(a), np.array(b), np.array(p)) for (a, b, p) in hp[:8]]
            est = statistics.median(time_cv2(wl, hp_cpu, 3, 2))
            reps_cpu = max(5, min(2000, int(12.0 / max(est, 1e-6))))
            ts = time_cv2(wl, hp_cpu, reps_cpu, 3)
            ts1 = time_cv2(wl, hp_cpu, max(3, min(200, int(4.0 / max(est * cv2.getNumThreads(), 1e-6)))), 1, threads=1)
            cv2.setNumThreads(-1)
            cpu = {"value": n * len(ts) / sum(ts), "unit": "keypoints/s", "cores": cv2.getNumThreads(), "kind": "reference",
                   "sample": "%d cv2.calcOpticalFlowPyrLK calls on the same workload (cv2 %s, %d OpenCV threads of os.cpu_count()=%s): "
                             "median %.3f ms, min %.3f ms per call; single thread: median %.3f ms"
                             % (len(ts), cv2.__version__, cv2.getNumThreads(), os.cpu_count(), 1e3 * statistics.median(ts), 1e3 * min(ts),
                                1e3 * statistics.median(ts1)),
                   "ms_per_call_median": 1e3 * statistics.median(ts), "ms_per_call_single_thread": 1e3 * statistics.median(ts1)}

        h2d, d2h = 2 * w * h + n * 8, n * 13
        line = {
            "metric": "tracked_keypoints_per_sec", "value": value, "unit": "keypoints/s", "n_gpus": world, "steps": K_steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / K_steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": describe(wl_name, wl),
                       "l2": "rotating pool of %d distinct device-resident pairs (%.0f MB) > 126 MB L2; no flush needed" % (P, P * pair_bytes / 1e6),
                       "pool": ("cyclic column shifts of 4 base pairs (the pool of rounds 1-2: a wrap-around seam inside every shifted image), %d point sets" % n_host)
                               if LEGACY_ROLL_POOL else
                               ("every pair is a crop of a wide synthetic canvas (texture + affine warp) at its own offset, %d point sets; "
                                "no wrap-around seams" % n_host),
                       "sharding": "each rank tracks its own independent sequences; no collective on the data path",
                       "host_cores_per_rank": len(host_cores)},
            "timing": {"steps": K_steps, "ms": dev_ms,
                       "note": "value / ms_per_step / e2e / pipelined / kernel_ms / graph_replay: exactly `steps` timed steps each"},
            "pairs_per_sec": world * K_steps / (dev_ms * 1e-3),
            "status1_fraction": st_mean,
            "kernel_ms": {"pyramid_build_both_images": pyr_ms, "lk": lk_ms},
            "e2e": {"value": e2e_value, "unit": "keypoints/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s / K_steps, "pairs_per_sec": world * K_steps / e2e_s,
                    "api": "visual_odom_pipeline_b200.calcOpticalFlowPyrLK(numpy arrays in PINNED host memory) -> numpy"},
            "e2e_pageable": {"value": world * n * K_steps / e2e_page_s, "unit": "keypoints/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                             "ms_per_step": 1e3 * e2e_page_s / K_steps, "pairs_per_sec": world * K_steps / e2e_page_s,
                             "api": "the same call with ordinary (pageable) numpy arrays, as the un-edited reference passes them; staged through "
                                    "pinned memory by the calling thread + 3 helper threads inside the C ABI"},
            "gpu_launches": launches_per_step * K_steps,
            "clocks": clocks,
            "roofline": roofline,
            "lk_roofline": lk_roofline,
            "pipelined": pipelined,
            "batched_lk": batched,
            "generic_lk": generic,
            "graph_replay": graph_replay,
            "sharded_batch": sharded,
            "parity": parity,
            "detection": detection,
            "prefilter": prefilter,
            "cpu_baseline": cpu,
            "device": ctx.name,
        }
        if last_outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in last_outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(line), flush=True)
    sharding.barrier()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


def run_sharded_batch(args, wl, rank, local_rank, world, dev):
    """BASELINE configs[3]: `--sequences` independent KITTI-shape sequences, block-partitioned over the ranks by
    sharding.shard_range; every rank uploads its shard, then per frame: ONE batched pyramid build and ONE batched LK launch
    for the whole shard, points carried from frame to frame on the device.  No collective on the data path; the final
    positions are gathered in sequence order afterwards and rank 0 bit-compares a sample of sequences with cv2."""
    import torch
    from visual_odom_pipeline_b200 import sharding, synth as S, tracker as T
    h, w, n = wl["h"], wl["w"], wl["n"]
    lk = dict(winSize=wl["win"], maxLevel=wl["max_level"], criteria=wl["criteria"])
    n_seq, n_frames = args.sequences, 4
    lo, hi = sharding.shard_range(n_seq, world, rank)
    B = hi - lo
    base = S.sequence(h, 2 * w, n_frames, seed=91)

    def host_frames(seq):     # deterministic per sequence id, on any rank: a crop of the wide base sequence (no seam)
        sh = (seq * 17) % w
        return [np.ascontiguousarray(f[:, sh:sh + w]) for f in base]

    def host_points(seq):
        return S.uniform_points(n, h, w, seed=7000 + seq).reshape(n, 2)

    frames = [T.alloc_image_batch(max(B, 1), h, w, device=dev) for _ in range(n_frames)]
    pts0 = torch.empty((max(B, 1), n, 2), dtype=torch.float32, device=dev)
    for j in range(B):
        fr = host_frames(lo + j)
        for t in range(n_frames):
            frames[t][j].copy_(torch.from_numpy(fr[t]))
        pts0[j].copy_(torch.from_numpy(host_points(lo + j)))
    stream = torch.cuda.current_stream(dev)

    def run_once():
        cur = pts0
        prev = T.DevicePyramid(frames[0][:B], lk["winSize"], lk["maxLevel"])
        st = None
        for t in range(1, n_frames):
            nxt = T.DevicePyramid(frames[t][:B], lk["winSize"], lk["maxLevel"], ctx=prev.ctx)
            cur, st, _er = T.lk_track(prev, nxt, cur[:B], None, lk["criteria"])
            prev = nxt
        return cur, st

    ms = []
    final = st = None
    for rep in range(4):          # first pass = warm-up
        torch.cuda.synchronize()
        sharding.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        if B > 0:
            final, st = run_once()
        e1.record(stream)
        torch.cuda.synchronize()
        sharding.barrier()
        if rep > 0:
            ms.append(sharding.max_over_ranks(e0.elapsed_time(e1)))
    t_ms = statistics.median(ms)
    if B == 0:
        final = torch.zeros((0, n, 2), dtype=torch.float32, device=dev)
        st = torch.zeros((0, n), dtype=torch.uint8, device=dev)
    all_q = sharding.gather_shards(final.contiguous(), n_seq)
    all_s = sharding.gather_shards(st.contiguous(), n_seq)
    if rank != 0:
        return None
    import cv2
    sample = sorted(set([0, n_seq // 3, n_seq // 2, n_seq - 1]))
    ok = True
    for seq in sample:
        fr = host_frames(seq)
        cur = host_points(seq).reshape(-1, 1, 2)
        for t in range(1, n_frames):
            cur, cs, _ce = cv2.calcOpticalFlowPyrLK(np.ascontiguousarray(fr[t - 1]), np.ascontiguousarray(fr[t]), cur, None, **lk)
        ok = ok and np.array_equal(cur.reshape(-1, 2).view(np.uint32), all_q[seq].cpu().numpy().view(np.uint32)) \
            and np.array_equal(cs.ravel(), all_s[seq].cpu().numpy())
    pairs = n_seq * (n_frames - 1)
    return {"workload": "configs[3]: %d independent KITTI-shape sequences x %d frames, %d keypoints each, block-partitioned over %d rank(s)"
                        % (n_seq, n_frames, n, world),
            "sequences_per_rank": sharding.shard_sizes(n_seq, world), "frames_per_sequence": n_frames,
            "ms": t_ms, "pairs_per_sec": pairs / (t_ms * 1e-3), "keypoints_per_sec": pairs * n / (t_ms * 1e-3),
            "launches_per_rank": n_frames + (n_frames - 1), "scaling": "strong",
            "timed": "per rank: %d batched pyramid builds + %d batched LK launches, device resident (CUDA events, max over ranks, median of 3)"
                     % (n_frames, n_frames - 1),
            "gathered_sequences_bit_identical_to_cv2": {"sample": sample, "ok": bool(ok)}}


def run_prefilter(args, wl, K, hp, imgs, P, local_rank, world, stream):
    """Row f3 (SURVEY.md s8f rank 3): the loader's cv2.bilateralFilter(img, 5, 1.5, 1.5) (src/loader/loader.py:16-20,86), once per
    frame.  Reported next to the headline, not part of `value`."""
    import torch
    from visual_odom_pipeline_b200 import filters as F
    h, w = wl["h"], wl["w"]
    ref_kw = dict(d=5, sigmaColor=1.5, sigmaSpace=1.5)
    frames = [np.array(x[0]) for x in hp[:8]]
    for r_ in range(5):
        got = K.bilateralFilter(frames[r_ % len(frames)], device=local_rank, **ref_kw)
    reps = 200
    t0 = time.perf_counter()
    for r_ in range(reps):
        K.bilateralFilter(frames[r_ % len(frames)], device=local_rank, **ref_kw)
    host_ms = 1e3 * (time.perf_counter() - t0) / reps
    nb = min(64, 2 * P)
    src = imgs[:nb, :, :w]
    dst = torch.empty_like(imgs[:nb])[:, :, :w]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r_ in range(3):
        if r_ == 2:
            ev[0].record(stream)
        F.bilateral_filter(src, out=dst, **ref_kw)
    ev[1].record(stream)
    torch.cuda.synchronize()
    bms = ev[0].elapsed_time(ev[1])
    out = {"api": "visual_odom_pipeline_b200.bilateralFilter(numpy image, d=5, sigmaColor=1.5, sigmaSpace=1.5) -> numpy",
           "e2e_ms_per_frame": host_ms, "h2d_bytes_per_frame": w * h, "d2h_bytes_per_frame": w * h,
           "batched": {"frames": nb, "ms": bms, "us_per_frame": 1e3 * bms / nb, "gbs": 2.0 * nb * w * h / (bms * 1e-3) / 1e9,
                       "algorithmic_bytes_per_frame": 2 * w * h, "note": "device resident, one launch for the batch (u8 in, u8 out)"}}
    try:
        import cv2
        was = cv2.ipp.useIPP()
        cv2.ipp.setUseIPP(False)
        gen = cv2.bilateralFilter(frames[0], **ref_kw)
        cv2.ipp.setUseIPP(True)
        ipp = cv2.bilateralFilter(frames[0], **ref_kw)
        got = K.bilateralFilter(frames[0], device=local_rank, **ref_kw)
        out["parity"] = {"pixels": int(got.size), "differ_from_opencv_generic_path": int((got != gen).sum()),
                         "max_abs_diff_vs_generic": int(np.abs(got.astype(int) - gen.astype(int)).max()),
                         "max_abs_diff_vs_ipp_wheel": int(np.abs(got.astype(int) - ipp.astype(int)).max()),
                         "ipp_vs_generic_differ_fraction": float((ipp != gen).mean())}
        if world == 1 and not args.no_cpu_baseline:
            for name, flag in (("cv2_ipp_ms_per_frame", True), ("cv2_generic_ms_per_frame", False)):
                cv2.ipp.setUseIPP(flag)
                for r_ in range(3):
                    cv2.bilateralFilter(frames[r_ % len(frames)], **ref_kw)
                t0 = time.perf_counter()
                for r_ in range(40):
                    cv2.bilateralFilter(frames[r_ % len(frames)], **ref_kw)
                out[name] = 1e3 * (time.perf_counter() - t0) / 40
            out["cv2_threads"] = cv2.getNumThreads()
        cv2.ipp.setUseIPP(was)
    except Exception as ex:   # pragma: no cover
        out["parity"] = {"error": repr(ex)}
    return out


def run_detection(args, wl, K, L, hp, hpin, imgs, P, n_host, local_rank, world, dev, stream):
    """Next row of the scope table (SURVEY.md s8f rank 2): Shi-Tomasi detection with the reference's parameters
    (src/extractor/extractor.py:21-24), once per frame.  Reported next to the headline, not part of `value`."""
    import torch
    from visual_odom_pipeline_b200 import detector as D
    h, w, n = wl["h"], wl["w"], wl["n"]
    det_kw = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)
    dimgs = [x[0] for x in hpin]
    dmask = K.pinned_empty(dimgs[0].shape, np.uint8)
    dmask[...] = 255
    for k_ in range(0, 400):   # discs around "tracked" keypoints, as extractor.py:102-107 builds the mask
        cy, cx = int(hp[0][2].reshape(-1, 2)[k_ % n][1]), int(hp[0][2].reshape(-1, 2)[k_ % n][0])
        dmask[max(cy - 7, 0):cy + 8, max(cx - 7, 0):cx + 8] = 0
    for r_ in range(5):
        got = K.goodFeaturesToTrack(dimgs[r_ % n_host], mask=dmask, device=local_rank, **det_kw)
    dreps = 200
    t0 = time.perf_counter()
    for r_ in range(dreps):
        K.goodFeaturesToTrack(dimgs[r_ % n_host], mask=dmask, device=local_rank, **det_kw)
    det_ms = 1e3 * (time.perf_counter() - t0) / dreps
    # the same step with the mask rasterised on the device from the tracked keypoints (opt-in fused call)
    tracked = K.pinned_empty((n, 2), np.float32)
    tracked[...] = hp[0][2].reshape(-1, 2)
    for r_ in range(5):
        K.detectNewFeatures(dimgs[r_ % n_host], tracked, 10, device=local_rank, **det_kw)
    t0 = time.perf_counter()
    for r_ in range(dreps):
        K.detectNewFeatures(dimgs[r_ % n_host], tracked, 10, device=local_rank, **det_kw)
    det_pts_ms = 1e3 * (time.perf_counter() - t0) / dreps
    # the whole data-parallel part of a frame chained on the device (KLTTracker.step: forward + second LK pass with
    # the reference's parameters, filter, mask, detection) against the same sequence of cv2 calls
    frame_step = None
    try:
        import cv2
        from visual_odom_pipeline_b200 import synth as S2, tracker as T2
        lkp = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))      # extractor.py:16-19
        seq = S2.sequence(h, w, 6, seed=11)
        dseq = [torch.from_numpy(f).to(dev) for f in seq]
        p_init = hp[0][2].reshape(-1, 2).copy()

        def run_b200(reps):
            trk = T2.KLTTracker(**lkp).reset(dseq[0])
            pts_d = torch.from_numpy(p_init).to(dev)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for r_ in range(reps):
                surv, keep_, new_ = trk.step(dseq[1 + r_ % 5], pts_d)
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / reps, int(surv.shape[0]), 0 if new_ is None else len(new_)
        run_b200(5)
        fs_ms, n_surv, n_new = run_b200(50)

        def run_cv2(reps):
            t0 = time.perf_counter()
            for r_ in range(reps):
                im0, im1 = seq[0], seq[1 + r_ % 5]
                p0 = p_init.reshape(-1, 1, 2)
                p1, _a, _b = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **lkp)
                p0r, _a, _b = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **lkp)
                good = abs(p0 - p0r).reshape(-1, 2).max(-1) < 30
                q = p1.reshape(-1, 2)
                kp_ = q[good & (0 <= q[:, 0]) & (q[:, 0] <= w) & (0 <= q[:, 1]) & (q[:, 1] <= h)]
                m_ = np.zeros_like(im1)
                m_[:] = 255
                for x_, y_ in [np.int32(p_) for p_ in kp_]:
                    cv2.circle(m_, (int(x_), int(y_)), 10, 0, -1)
                cv2.goodFeaturesToTrack(im1, mask=m_, **det_kw)
            return (time.perf_counter() - t0) / reps
        frame_step = {"api": "KLTTracker.step(frame, points): 2 LK passes (win 31, eps 0.03), filter, mask, goodFeaturesToTrack; frames and points device-resident",
                      "ms_per_frame": 1e3 * fs_ms, "tracked": int(len(p_init)), "survivors": n_surv, "new_corners": n_new}
        if world == 1 and not args.no_cpu_baseline:
            run_cv2(2)
            frame_step["cv2_ms_per_frame"] = 1e3 * run_cv2(10)
            frame_step["cv2_note"] = "same steps with cv2 on the host (%d threads), incl. the reference's Python loop over cv2.circle" % cv2.getNumThreads()
    except Exception as ex:   # pragma: no cover
        frame_step = {"error": repr(ex)}
    # device-resident, batched eigenvalue maps (the kernels only): 64 frames per launch sequence
    nbd = min(64, 2 * P)
    de = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r_ in range(3):
        if r_ == 2:
            de[0].record(stream)
        D.corner_min_eigen_val(imgs[:nbd, :, :w], 31)
    de[1].record(stream)
    torch.cuda.synchronize()
    eig_ms = de[0].elapsed_time(de[1])
    detection = {"api": "visual_odom_pipeline_b200.goodFeaturesToTrack(numpy pinned image, mask, %s) -> numpy" % det_kw,
                 "e2e_ms_per_frame": det_ms, "frames_per_sec": 1e3 / det_ms, "corners": 0 if got is None else int(len(got)),
                 "h2d_bytes_per_frame": 2 * w * h,
                 "frame_step": frame_step,
                 "fused_from_tracked_points": {"api": "visual_odom_pipeline_b200.detectNewFeatures(image, %d tracked keypoints, mask_radius=10)" % n,
                                               "e2e_ms_per_frame": det_pts_ms, "h2d_bytes_per_frame": w * h + 8 * n,
                                               "note": "mask of extractor.py:102-107 rasterised on the device; the reference additionally spends "
                                                       "a Python loop over cv2.circle per tracked keypoint building it on the host"},
                 "batched_min_eig": {"frames": nbd, "ms": eig_ms, "us_per_frame": 1e3 * eig_ms / nbd,
                                     "mpixels_per_sec": nbd * w * h / (eig_ms * 1e-3) / 1e6,
                                     "algorithmic_bytes_per_frame": 5 * w * h,
                                     "note": "u8 frame in, float32 eigenvalue map out; 4 launches per batch (products, running row sums, "
                                             "running column sums + eigenvalue, all in OpenCV's summation order)"}}
    try:
        import cv2
        got = K.goodFeaturesToTrack(dimgs[0], mask=dmask, device=local_rank, **det_kw)
        ref = cv2.goodFeaturesToTrack(np.array(dimgs[0]), mask=np.array(dmask), **det_kw)
        detection["parity"] = {"corners_identical_to_cv2": bool((got is None and ref is None) or (got is not None and ref is not None
                                                                                              and got.shape == ref.shape and np.array_equal(got, ref)))}
        if world == 1 and not args.no_cpu_baseline:
            ci, cm = np.array(dimgs[0]), np.array(dmask)
            for r_ in range(3):
                cv2.goodFeaturesToTrack(ci, mask=cm, **det_kw)
            t0 = time.perf_counter()
            for r_ in range(40):
                cv2.goodFeaturesToTrack(ci, mask=cm, **det_kw)
            detection["cv2_ms_per_frame"] = 1e3 * (time.perf_counter() - t0) / 40
            detection["cv2_threads"] = cv2.getNumThreads()
    except Exception as ex:   # pragma: no cover
        detection["parity"] = {"error": repr(ex)}
    return detection


if __name__ == "__main__":
    sys.exit(main())
