"""What the minimum track distance of KLTSequenceBatch costs and saves: graph replay, two arms alternated in every rep over
the same frames: min_track_distance off, and min_track_distance=10.

    python scripts/thin_time.py [--batches 1,16,64] [--frames 40] [--warmup 5] [--reps 5] [--points 2000] [--capacity 4096]
                                [--out LOG]

KITTI shape (376 x 1241), reference parameters (LK win 31, maxLevel 3, criteria (3, 30, 0.03); detection 1000 / 0.03 / 10 /
31, mask radius 10, max_bidir_error 30).  Two motions of the synthetic sequences: the default warp (scale 1.003 per
frame, zoom in) and the same warp at scale 0.99 per frame (contracting: tracks converge).  Each rep builds both arms
from the same initial corners, steps frame 1 eagerly, captures, replays the warm-up frames untimed and times the next
`frames` frames with a host clock around work that ends in a device synchronisation; the line reports ms per frame
(median over the reps, and [min, max]).  Off the timed path, one more pass per arm over the same frames reports the mean
points per sequence in the timed window and the tracks thinned per frame and sequence.  Prints the card's name, power
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
MOTIONS = {"default": (1.1, -0.6, 0.15, 1.003), "scale0.99": (1.1, -0.6, 0.15, 0.99)}
ARMS = {"off": None, "thin10": 10.0}


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
        sys.exit("thin_time.py needs a CUDA device")

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
          "reps": args.reps, "motions": MOTIONS, "arms": ARMS})

    def make(imgs, pts0, cnt0, arm):
        return T.KLTSequenceBatch(imgs[0], pts0, cnt0, C, min_track_distance=ARMS[arm], **LK, **DET)

    for mname, motion in MOTIONS.items():
        pool = [S.sequence(H, W, n_frames, seed=100 + i, motion=motion) for i in range(args.pool)]
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
            d = {"motion": mname, "batch": B}
            for a in ARMS:
                # untimed: points per sequence going into each timed step, tracks thinned per frame
                sb = make(imgs, pts0, cnt0, a)
                pts_total, thinned = 0, 0
                for t in range(1, n_frames):
                    if t >= t0_timed:
                        pts_total += int(sb.counts.sum())
                    sb.step(imgs[t])
                    if t >= t0_timed and ARMS[a] is not None:
                        thinned += int(sb.thinned.sum())
                sb.check()
                v = times[a][1:]
                d[a + "_ms"] = round(float(np.median(v)) * 1e3, 4)
                d[a + "_ms_min_max"] = [round(min(v) * 1e3, 4), round(max(v) * 1e3, 4)]
                d[a + "_points_per_seq"] = round(pts_total / args.frames / B, 1)
                d[a + "_thinned_per_seq_frame"] = round(thinned / args.frames / B, 1)
            emit(d)
        del frames


if __name__ == "__main__":
    main()
