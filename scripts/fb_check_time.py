"""What the forward-backward check of KLTSequenceBatch costs: graph replay with history=2, three arms alternated in every
rep over the same frames: second_pass="reference" (the reference's same-direction pass, max_bidir_error 30),
second_pass="reverse" (max_bidir_error 1) and second_pass="reverse" with motion_prior="velocity" (the reverse pass from
the mirrored start).

    python scripts/fb_check_time.py [--batches 1,16,64] [--frames 40] [--reps 5] [--points 2000] [--capacity 4096]
                                    [--out LOG]

KITTI shape (376 x 1241), reference parameters (LK win 31, maxLevel 3, criteria (3, 30, 0.03); detection 1000 / 0.03 / 10 /
31, mask radius 10).  Two motions of the synthetic sequences: the default small warp (about 1.3 px per frame) and about
10 px per frame.  Each rep builds every arm from the same state, steps frame 1 eagerly, captures, and times frames
2 .. T + 1 with a host clock around work that ends in a device synchronisation; the line reports ms per frame (median
over the reps, and [min, max]).  Off the timed path, one more pass per arm reports the mean survivors per frame, and on
every fifth frame it re-runs the arm's passes with tracker.lk_track(..., return_iters=True) from the arm's own points:
the forward pass (from the velocity starts in the velocity arm), then the second pass in both directions from its
result, the same-direction pass started at p1 and the reverse pass started at p1 (at the mirrored start, with the flag,
in the velocity arm): mean LK iterations per point over all pyramid levels.  Prints the card's name, power limit and
maximum SM clock first.
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
MOTIONS = {"default": (1.1, -0.6, 0.15, 1.003), "10px": (10.0, 1.5, 0.2, 1.0)}
# arm -> (second_pass, motion_prior, max_bidir_error)
ARMS = {"reference": ("reference", None, 30.0), "reverse": ("reverse", None, 1.0), "reverse_velocity": ("reverse", "velocity", 1.0)}


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
    from visual_odom_pipeline_b200._lib import OPTFLOW_USE_INITIAL_FLOW
    if not torch.cuda.is_available():
        sys.exit("fb_check_time.py needs a CUDA device")

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(s + "\n")

    C, n_frames = args.capacity, args.frames + 2
    emit({"card": card(), "points": args.points, "capacity": C, "frames": args.frames, "reps": args.reps, "history": 2,
          "motions": MOTIONS, "arms": ARMS})

    def make(imgs, pts0, cnt0, arm):
        second_pass, prior, max_err = ARMS[arm]
        return T.KLTSequenceBatch(imgs[0], pts0, cnt0, C, history=2, motion_prior=prior, second_pass=second_pass,
                                  max_bidir_error=max_err, **LK, **DET)

    def iterations(imgs, recorded, mirrored):
        """Mean LK iterations per point of the forward pass and of both second passes, over the recorded frames."""
        its = {"forward": [], "same_direction": [], "reverse": []}
        for t, pts, cnt, starts in recorded:
            prev = T.DevicePyramid(imgs[t - 1], LK["winSize"], LK["maxLevel"], copy=True).build()
            nxt = T.DevicePyramid(imgs[t], LK["winSize"], LK["maxLevel"], copy=True).build()
            valid = torch.arange(pts.shape[1], device="cuda")[None, :] < cnt[:, None].long()
            fw = dict(nextPts=starts, flags=OPTFLOW_USE_INITIAL_FLOW) if mirrored else {}
            p1, _st, _er, it = T.lk_track(prev, nxt, pts, criteria=LK["criteria"], return_iters=True, **fw)
            its["forward"].append(it[valid].double())
            it = T.lk_track(prev, nxt, p1, criteria=LK["criteria"], return_iters=True)[3]
            its["same_direction"].append(it[valid].double())
            bw = dict(nextPts=p1 - (starts - pts), flags=OPTFLOW_USE_INITIAL_FLOW) if mirrored else {}
            it = T.lk_track(nxt, prev, p1, criteria=LK["criteria"], return_iters=True, **bw)[3]
            its["reverse"].append(it[valid].double())
        return {k: round(float(torch.cat(v).mean()), 3) for k, v in its.items()}

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
            for rep in range(args.reps + 1):            # rep 0: warm-up of every arm
                for a in ARMS:
                    sb = make(imgs, pts0, cnt0, a)
                    sb.step(imgs[1])
                    sb.capture()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for t in range(2, n_frames):
                        sb.step(imgs[t])
                    torch.cuda.synchronize()
                    times[a].append((time.perf_counter() - t0) / args.frames)
                    sb.check()
            d = {"motion": mname, "batch": B}
            most = 0
            for a in ARMS:
                # untimed: survivors per frame, and the arm's own points on every fifth frame
                sb = make(imgs, pts0, cnt0, a)
                total, recorded = 0, []
                for t in range(1, n_frames):
                    if t % 5 == 0:
                        p = sb.points.clone()
                        q = sb.window(2)[:, :, 0]
                        starts = torch.where(torch.isnan(q), p, p + (p - q))
                        recorded.append((t, p, sb.counts.clone(), starts))
                    sb.step(imgs[t])
                    total += int(sb.keep.sum())
                    most = max(most, int(sb.counts.max()))
                sb.check()
                v = times[a][1:]
                d[a + "_ms"] = round(float(np.median(v)) * 1e3, 4)
                d[a + "_ms_min_max"] = [round(min(v) * 1e3, 4), round(max(v) * 1e3, 4)]
                d[a + "_survivors_per_seq_frame"] = round(total / (n_frames - 1) / B, 1)
                d[a + "_lk_iters_per_point"] = iterations(imgs, recorded, ARMS[a][1] == "velocity")
            if most > C - DET["maxCorners"]:
                sys.exit("%s B=%d: %d points in a sequence: the capacity %d could bind" % (mname, B, most, C))
            emit(d)
        del frames


if __name__ == "__main__":
    main()
