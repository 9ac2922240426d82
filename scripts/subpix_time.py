"""What sub-pixel refinement of the new corners costs in KLTSequenceBatch: graph replay, two arms alternated in every rep over
the same frames: off, and subpix=((5, 5), (-1, -1), (3, 40, 0.001)).  Then the refinement kernel alone.

    python scripts/subpix_time.py [--batches 1,16,64] [--frames 40] [--warmup 5] [--reps 5] [--points 2000]
                                  [--capacity 4096] [--kernel-iters 50] [--out LOG]

KITTI shape (376 x 1241), reference parameters (LK win 31, maxLevel 3, criteria (3, 30, 0.03); detection 1000 / 0.03 / 10 /
31, mask radius 10, max_bidir_error 30), synthetic sequences with the default warp.  Each rep builds both arms from the
same initial corners, steps frame 1 eagerly, captures, replays the warm-up frames untimed and times the next `frames`
frames with a host clock around work that ends in a device synchronisation; the line reports ms per frame (median over
the reps, and [min, max]) and the mean new corners per sequence and step.

The kernel line times detector.corner_sub_pix with CUDA events on a full row, as at frame 0 or a restart: the first
1000 corners cv2.goodFeaturesToTrack finds on each sequence's first frame (B rows), refined from their integer positions
again at every launch (a copy of the corners is restored first, outside the events).  The oracle's mean iteration count on
the same corners is computed on the host, off the timed path.  Prints the card's name, power limit and maximum SM clock
first.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LK = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
DET = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)
H, W = 376, 1241
SUBPIX = ((5, 5), (-1, -1), (3, 40, 0.001))
ARMS = {"off": None, "subpix": SUBPIX}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,16,64")
    ap.add_argument("--frames", type=int, default=40, help="timed frames per rep")
    ap.add_argument("--warmup", type=int, default=5, help="untimed replayed frames before the timed ones")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--points", type=int, default=2000)
    ap.add_argument("--capacity", type=int, default=4096)
    ap.add_argument("--pool", type=int, default=8, help="distinct synthetic sequences (sequence b replays pool[b %% pool])")
    ap.add_argument("--kernel-iters", type=int, default=50, help="timed launches of the kernel line")
    ap.add_argument("--out", help="also append the lines to this file")
    args = ap.parse_args()
    import torch
    import visual_odom_pipeline_b200 as K
    from visual_odom_pipeline_b200 import detector as D
    from visual_odom_pipeline_b200 import synth as S
    from visual_odom_pipeline_b200 import tracker as T
    from oracle import subpix_oracle as O
    if not torch.cuda.is_available():
        sys.exit("subpix_time.py needs a CUDA device")

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(s + "\n")

    C = args.capacity
    t0_timed = 2 + args.warmup
    n_frames = t0_timed + args.frames
    emit({"card": card(), "points": args.points, "capacity": C, "frames": args.frames, "warmup": args.warmup,
          "reps": args.reps, "subpix": SUBPIX, "arms": list(ARMS)})

    def make(imgs, pts0, cnt0, arm):
        return T.KLTSequenceBatch(imgs[0], pts0, cnt0, C, subpix=ARMS[arm], **LK, **DET)

    pool = [S.sequence(H, W, n_frames, seed=100 + i) for i in range(args.pool)]
    frames = torch.from_numpy(np.stack([np.stack(s) for s in pool])).cuda()
    init, first = [], []
    for s in pool:
        c = K.goodFeaturesToTrack(s[0], args.points, DET["qualityLevel"], DET["minDistance"], blockSize=DET["blockSize"])
        init.append(torch.from_numpy(c.reshape(-1, 2)).cuda())
        first.append(c.reshape(-1, 2)[:DET["maxCorners"]])
    batches = [int(x) for x in args.batches.split(",")]
    for B in batches:
        idx = (torch.arange(B) % args.pool).tolist()
        imgs = [frames[idx, t].contiguous() for t in range(n_frames)]
        n = max(int(init[i].shape[0]) for i in idx)
        pts0 = torch.zeros((B, n, 2), dtype=torch.float32, device="cuda")
        cnt0 = torch.zeros((B,), dtype=torch.int32, device="cuda")
        for b, i in enumerate(idx):
            pts0[b, :init[i].shape[0]] = init[i]
            cnt0[b] = init[i].shape[0]
        times = {a: [] for a in ARMS}
        new_total = 0
        for rep in range(args.reps + 1):            # rep 0: warm-up of both arms
            for a in ARMS:
                sb = make(imgs, pts0, cnt0, a)
                sb.step(imgs[1])
                sb.capture()
                for t in range(2, t0_timed):
                    sb.step(imgs[t])
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for t in range(t0_timed, n_frames):
                    sb.step(imgs[t])
                    if rep == 0 and a == "subpix":
                        new_total += int(sb.n_new.sum())   # warm-up rep only: synchronises
                torch.cuda.synchronize()
                times[a].append((time.perf_counter() - t0) / args.frames)
                sb.check()
        d = {"batch": B, "new_corners_per_seq_step": round(new_total / args.frames / B, 1)}
        for a in ARMS:
            v = times[a][1:]
            d[a + "_ms"] = round(float(np.median(v)) * 1e3, 4)
            d[a + "_ms_min_max"] = [round(min(v) * 1e3, 4), round(max(v) * 1e3, 4)]
        d["added_ms"] = round(d["subpix_ms"] - d["off_ms"], 4)
        emit(d)

    # the kernel alone on full rows of new corners (frame 0 / restart)
    for B in batches:
        idx = [b % args.pool for b in range(B)]
        N = max(len(first[i]) for i in idx)
        rows = np.full((B, N, 2), np.nan, np.float32)
        counts = np.zeros(B, np.int32)
        for b, i in enumerate(idx):
            rows[b, :len(first[i])] = first[i]
            counts[b] = len(first[i])
        img0 = frames[idx, 0].contiguous()
        src = torch.from_numpy(rows).cuda()
        pts = src.clone()
        cnt = torch.from_numpy(counts).cuda()
        for _ in range(3):
            pts.copy_(src)
            D.corner_sub_pix(img0, pts, *SUBPIX, counts=cnt)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.kernel_iters)]
        for e0, e1 in ev:
            pts.copy_(src)
            e0.record()
            D.corner_sub_pix(img0, pts, *SUBPIX, counts=cnt)
            e1.record()
        torch.cuda.synchronize()
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev)
        iters = np.concatenate([O.corner_sub_pix(pool[i][0], first[i], *SUBPIX, return_iters=True)[1] for i in sorted(set(idx))])
        emit({"kernel": "subpix_kernel", "batch": B, "corners": int(counts.sum()), "ms_median": round(ms[len(ms) // 2], 4),
              "ms_min_max": [round(ms[0], 4), round(ms[-1], 4)], "us_per_corner": round(ms[len(ms) // 2] * 1e3 / int(counts.sum()), 4),
              "oracle_mean_iterations": round(float(iters.mean()), 2)})


if __name__ == "__main__":
    main()
