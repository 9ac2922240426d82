"""Time of the per-frame step for B sequences three ways over the same frames: (a) KLTTracker.step_batch per frame (one
host synchronisation each), (b) KLTSequenceBatch.step enqueued for T frames, then one synchronisation, (c) the same
replayed from CUDA graphs.  --history R adds (h): (c) with history=R, the per-track records of every step.  --control
adds (k): (h) built with control=True (the steered step's kernels, with no drop or restart requested), which must give the
same outputs as (h).

    python scripts/frame_step_async_time.py [--batches 1,4,16,64] [--frames 50] [--reps 5] [--points 2000]
                                            [--capacity 4096] [--arms abc] [--history R] [--control] [--extra]
                                            [--tree DIR] [--out LOG]

KITTI shape (376 x 1241), reference parameters (LK win 31, maxLevel 3, criteria (3, 30, 0.03); detection 1000 / 0.03 / 10 /
31, mask radius 10), `--points` initial corners per sequence.  Each rep starts every arm from the same state and times
frames 2 .. T + 1 (frame 1 is the eager step the graphs need before capture) with a host clock around work that ends in
a device synchronisation; the line reports the median over the reps of ms per frame.  The capacity is chosen so that it
never binds (checked: no sequence ever has more than capacity - maxCorners survivors), so all arms must end in the same
points, counts and keep flags, which is checked in the same run.  --extra adds two inputs: two 3840 x 2160 sequences and
a batch of noise frames with more than 8192 candidates (blockSize 3, qualityLevel 0.001), each with a capacity of
points + (frames + 3) * maxCorners.  --arms a with --tree DIR times step_batch of the package in another checkout (an A/B against an earlier tree).  Prints the card's name, power
limit and maximum SM clock first.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LK = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
DET = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)
H, W = 376, 1241


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,4,16,64")
    ap.add_argument("--frames", type=int, default=50, help="timed frames per rep")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--points", type=int, default=2000)
    ap.add_argument("--capacity", type=int, default=4096)
    ap.add_argument("--pool", type=int, default=8, help="distinct synthetic sequences (sequence b replays pool[b %% pool])")
    ap.add_argument("--arms", default="abc")
    ap.add_argument("--history", type=int, default=0, help="R >= 1: add arm h, graph replay with history=R")
    ap.add_argument("--control", action="store_true", help="add arm k, arm h with control=True")
    ap.add_argument("--extra", action="store_true", help="also the 4K and the noise inputs")
    ap.add_argument("--tree", default=ROOT, help="checkout whose package is imported")
    ap.add_argument("--out", help="also append the lines to this file")
    args = ap.parse_args()
    if args.history > 0:
        args.arms += "h"
    if args.control:
        args.arms += "k"
    sys.path.insert(0, os.path.abspath(args.tree))
    import torch
    import visual_odom_pipeline_b200 as K
    from visual_odom_pipeline_b200 import synth as S
    from visual_odom_pipeline_b200 import tracker as T
    if not torch.cuda.is_available():
        sys.exit("frame_step_async_time.py needs a CUDA device")

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(s + "\n")

    C, n_frames = args.capacity, args.frames + 2
    emit({"card": card(), "tree": os.path.relpath(os.path.abspath(args.tree), ROOT), "points": args.points, "capacity": C, "frames": args.frames,
          "reps": args.reps, "arms": args.arms, "history": args.history, "control": args.control})

    def run(name, frames, init, det, B, C=C):
        """frames: (B, n_frames, H, W) CUDA; init: list of (n_b, 2) CUDA point sets."""
        n = max(int(p.shape[0]) for p in init)
        pts0 = torch.zeros((B, n, 2), dtype=torch.float32, device="cuda")
        cnt0 = torch.zeros((B,), dtype=torch.int32, device="cuda")
        for b, p in enumerate(init):
            pts0[b, :p.shape[0]] = p
            cnt0[b] = p.shape[0]
        imgs = [frames[:, t].contiguous() for t in range(n_frames)]
        times = {a: [] for a in args.arms}
        finals = {}
        most = 0
        for rep in range(args.reps + 1):            # rep 0: warm-up of every arm
            if "a" in args.arms:
                trk = T.KLTTracker(**LK).reset(imgs[0])
                pts, cnt = pts0, cnt0
                for t in range(1, n_frames):
                    if t == 2:
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                    pts, cnt, keep, _n_new = trk.step_batch(imgs[t], pts, cnt, **det)
                    most = max(most, pts.shape[1])
                torch.cuda.synchronize()
                times["a"].append((time.perf_counter() - t0) / args.frames)
                finals["a"] = (pts, cnt, keep)
            for arm in "bchk":            # the arms alternate within each rep
                if arm not in args.arms:
                    continue
                sb = T.KLTSequenceBatch(imgs[0], pts0, cnt0, C, history=args.history if arm in "hk" else 0, control=arm == "k", **LK,
                                        **det)
                sb.step(imgs[1])
                if arm in "chk":
                    sb.capture()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for t in range(2, n_frames):
                    sb.step(imgs[t])
                torch.cuda.synchronize()
                times[arm].append((time.perf_counter() - t0) / args.frames)
                sb.check()
                finals[arm] = (sb.points, sb.counts, sb.keep)
                if "a" not in args.arms:
                    most = max(most, int(sb.counts.max()))
        if most > C - det["maxCorners"]:
            sys.exit("%s: %d points in a sequence: the capacity %d could bind" % (name, most, C))
        identical = True
        if "a" in finals:
            pa, ca, ka = finals["a"]
            for arm in "bchk":
                if arm in finals:
                    p, c, k = finals[arm]
                    identical &= bool(torch.equal(c, ca)) and bool(torch.equal(k[:, :ka.shape[1]], ka)) and not bool(k[:, ka.shape[1]:].any())
                    for b in range(B):
                        identical &= bool(torch.equal(p[b, :int(ca[b])].view(torch.int32), pa[b, :int(ca[b])].view(torch.int32)))
        else:
            arms = [a for a in "bchk" if a in finals]
            identical = all(bool(torch.equal(x.view(torch.uint8), y.view(torch.uint8))) for a in arms[1:]
                            for x, y in zip(finals[arms[0]], finals[a]))
        if not identical:
            sys.exit("%s B=%d: the arms differ" % (name, B))
        d = {"input": name, "batch": B, "capacity": C, "identical": identical, "max_points_per_seq": most}
        for a, label in (("a", "step_batch_ms"), ("b", "async_ms"), ("c", "graph_ms"), ("h", "graph_history_ms"), ("k", "graph_control_ms")):
            if a in times:
                v = times[a][1:]
                d[label] = round(float(np.median(v)) * 1e3, 4)
                d[label + "_min_max"] = [round(min(v) * 1e3, 4), round(max(v) * 1e3, 4)]
        emit(d)

    pool = [S.sequence(H, W, n_frames, seed=100 + i) for i in range(args.pool)]
    frames = torch.from_numpy(np.stack([np.stack(s) for s in pool])).cuda()          # (pool, T, H, W)
    init = []
    for s in pool:
        c = K.goodFeaturesToTrack(s[0], args.points, DET["qualityLevel"], DET["minDistance"], blockSize=DET["blockSize"])
        init.append(torch.from_numpy(c.reshape(-1, 2)).cuda())
    for B in [int(x) for x in args.batches.split(",")]:
        idx = (torch.arange(B) % args.pool).tolist()
        run("kitti", frames[idx], [init[i] for i in idx], DET, B)
    del frames
    if args.extra:
        seqs = [S.sequence(2160, 3840, n_frames, seed=80 + b) for b in range(2)]
        f4k = torch.from_numpy(np.stack([np.stack(s) for s in seqs])).cuda()
        i4k = [torch.from_numpy(K.goodFeaturesToTrack(s[0], args.points, 0.03, 10, blockSize=31).reshape(-1, 2)).cuda() for s in seqs]
        # points pile up on 4K frames (a new maxCorners every frame, few lost): a capacity that cannot bind
        run("4k", f4k, i4k, DET, 2, C=args.points + (n_frames + 1) * DET["maxCorners"])
        del f4k
        det = dict(maxCorners=500, qualityLevel=0.001, minDistance=10, blockSize=3)
        rng = np.random.default_rng(5)
        noise = torch.from_numpy(rng.integers(0, 256, (4, n_frames, H, W), dtype=np.uint8)).cuda()
        inoise = [torch.from_numpy(K.goodFeaturesToTrack(noise[b, 0].cpu().numpy(), 500, 0.001, 10, blockSize=3).reshape(-1, 2)).cuda()
                  for b in range(4)]
        run("noise", noise, inoise, det, 4, C=args.points + (n_frames + 1) * det["maxCorners"])


if __name__ == "__main__":
    main()
