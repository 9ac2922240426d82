"""What grid detection in KLTSequenceBatch costs and gives: graph replay, two arms alternated in every rep over the same
frames: the global rule (detect_grid off), and detect_grid=(8, 4) with tracks_per_cell=64.

    python scripts/grid_detect_time.py [--batches 1,16,64] [--frames 40] [--warmup 5] [--reps 5] [--points 2000]
                                       [--capacity 4096] [--out LOG]

KITTI shape (376 x 1241), reference parameters (LK win 31, maxLevel 3, criteria (3, 30, 0.03); detection 1000 / 0.03 / 10 /
31, mask radius 10, max_bidir_error 30).  Two kinds of synthetic sequence with the default warp: "default" (uniform
contrast) and "uneven" (synth.uneven_sequence: the left third at a tenth of the contrast, like a shadow).  Each rep builds both arms
from the same initial corners, steps frame 1 eagerly, captures, replays the warm-up frames untimed and times the next
`frames` frames with a host clock around work that ends in a device synchronisation; the line reports ms per frame
(median over the reps, and [min, max]).  Off the timed path, one more pass per arm over the same frames reports the mean
points per sequence in the timed window and the fraction of (sequence, cell) pairs of the 8 x 4 grid holding at least
q / 2 = 32 points, after every timed step.  Prints the card's name, power
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
sys.path.insert(0, ROOT)

LK = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
DET = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)
H, W = 376, 1241
KINDS = ("default", "uneven")
GRID, Q = (8, 4), 64
ARMS = {"off": None, "grid8x4": GRID}


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
    ap.add_argument("--out", help="also append the lines to this file")
    args = ap.parse_args()
    import torch
    import visual_odom_pipeline_b200 as K
    from visual_odom_pipeline_b200 import synth as S
    from visual_odom_pipeline_b200 import tracker as T
    if not torch.cuda.is_available():
        sys.exit("grid_detect_time.py needs a CUDA device")

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
          "reps": args.reps, "kinds": KINDS, "grid": GRID, "tracks_per_cell": Q, "arms": list(ARMS)})

    def make(imgs, pts0, cnt0, arm):
        g = ARMS[arm]
        return T.KLTSequenceBatch(imgs[0], pts0, cnt0, C, detect_grid=g, tracks_per_cell=None if g is None else Q, **LK, **DET)

    X = torch.tensor([i * W // GRID[0] for i in range(GRID[0])], dtype=torch.float64, device="cuda")
    Y = torch.tensor([j * H // GRID[1] for j in range(GRID[1])], dtype=torch.float64, device="cuda")

    def filled_cells(sb):
        """(sequence, cell) pairs of the grid with at least Q / 2 points."""
        B = sb.counts.shape[0]
        p = sb.points.double()
        valid = (torch.arange(C, device="cuda")[None, :] < sb.counts[:, None].long()) & ~p.isnan().any(-1)
        i = (torch.searchsorted(X, p[..., 0].contiguous(), right=True) - 1).clamp(0, GRID[0] - 1)
        j = (torch.searchsorted(Y, p[..., 1].contiguous(), right=True) - 1).clamp(0, GRID[1] - 1)
        k = torch.where(valid, j * GRID[0] + i + GRID[0] * GRID[1] * torch.arange(B, device="cuda")[:, None], -1)
        n = torch.bincount(k[k >= 0], minlength=B * GRID[0] * GRID[1])
        return int((n >= Q // 2).sum())

    for kind in KINDS:
        pool = [S.sequence(H, W, n_frames, seed=100 + i) if kind == "default" else S.uneven_sequence(H, W, n_frames, seed=100 + i)
                for i in range(args.pool)]
        frames = torch.from_numpy(np.stack([np.stack(s) for s in pool])).cuda()
        init = []
        for s in pool:
            c = K.goodFeaturesToTrack(s[0], args.points, DET["qualityLevel"], DET["minDistance"], blockSize=DET["blockSize"])
            init.append(torch.from_numpy(c.reshape(-1, 2)).cuda())
        for B in [int(x) for x in args.batches.split(",")]:
            idx = (torch.arange(B) % args.pool).tolist()
            imgs = [frames[idx, t].contiguous() for t in range(n_frames)]
            n = max(int(init[i].shape[0]) for i in idx)
            pts0 = torch.zeros((B, n, 2), dtype=torch.float32, device="cuda")
            cnt0 = torch.zeros((B,), dtype=torch.int32, device="cuda")
            for b, i in enumerate(idx):
                pts0[b, :init[i].shape[0]] = init[i]
                cnt0[b] = init[i].shape[0]
            times = {a: [] for a in ARMS}
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
                    torch.cuda.synchronize()
                    times[a].append((time.perf_counter() - t0) / args.frames)
                    sb.check()
            d = {"sequence": kind, "batch": B}
            for a in ARMS:
                # untimed: points per sequence going into each timed step, cells holding at least Q / 2 after it
                sb = make(imgs, pts0, cnt0, a)
                pts_total, filled = 0, 0
                for t in range(1, n_frames):
                    if t >= t0_timed:
                        pts_total += int(sb.counts.sum())
                    sb.step(imgs[t])
                    if t >= t0_timed:
                        filled += filled_cells(sb)
                sb.check()
                v = times[a][1:]
                d[a + "_ms"] = round(float(np.median(v)) * 1e3, 4)
                d[a + "_ms_min_max"] = [round(min(v) * 1e3, 4), round(max(v) * 1e3, 4)]
                d[a + "_points_per_seq"] = round(pts_total / args.frames / B, 1)
                d[a + "_cells_at_half_q"] = round(filled / args.frames / B / (GRID[0] * GRID[1]), 3)
            emit(d)
        del frames


if __name__ == "__main__":
    main()
