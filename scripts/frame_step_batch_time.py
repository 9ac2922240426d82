"""Time of KLTTracker.step_batch (one call for B sequences) against B calls of KLTTracker.step over the same frames.

    python scripts/frame_step_batch_time.py [--batches 1,4,16,64] [--steps 50] [--warmup 5] [--points 2000] [--out LOG]

KITTI shape (376 x 1241), reference parameters (LK win 31, maxLevel 3, criteria (3, 30, 0.03); detection 1000 / 0.03 / 10 /
31, mask radius 10), `--points` initial corners per sequence.  Each step runs both arms on the same frames, each arm timed
with a host clock around work that ends in a device synchronisation, and checks in the same run that both return the
same survivors, keep flags and new corners.  Prints one JSON line per batch size (median ms per step over --steps steps
after --warmup) plus the card's name and power limit.
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
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--points", type=int, default=2000)
    ap.add_argument("--pool", type=int, default=8, help="distinct synthetic sequences (sequence b replays pool[b %% pool])")
    ap.add_argument("--out", help="also append the lines to this file")
    args = ap.parse_args()
    import torch
    import visual_odom_pipeline_b200 as K
    from visual_odom_pipeline_b200 import synth as S
    from visual_odom_pipeline_b200 import tracker as T
    if not torch.cuda.is_available():
        sys.exit("frame_step_batch_time.py needs a CUDA device")
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    emit({"card": card(), "shape": [H, W], "points": args.points, "steps": args.steps, "warmup": args.warmup})
    n_frames = args.warmup + args.steps + 1
    pool = [S.sequence(H, W, n_frames, seed=100 + i) for i in range(args.pool)]
    frames = torch.from_numpy(np.stack([np.stack(s) for s in pool])).cuda()          # (pool, T, H, W)
    init = []
    for s in pool:
        c = K.goodFeaturesToTrack(s[0], args.points, DET["qualityLevel"], DET["minDistance"], blockSize=DET["blockSize"])
        init.append(torch.from_numpy(c.reshape(-1, 2)).cuda())
    for B in [int(x) for x in args.batches.split(",")]:
        idx = torch.arange(B, device="cuda") % args.pool
        batch = T.KLTTracker(**LK).reset(frames[idx, 0])
        single = [T.KLTTracker(**LK).reset(frames[i, 0]) for i in idx.tolist()]
        n = max(int(init[i].shape[0]) for i in idx.tolist())
        pts = torch.zeros((B, n, 2), dtype=torch.float32, device="cuda")
        cnt = torch.zeros((B,), dtype=torch.int32, device="cuda")
        for b, i in enumerate(idx.tolist()):
            pts[b, :init[i].shape[0]] = init[i]
            cnt[b] = init[i].shape[0]
        spts = [init[i].clone() for i in idx.tolist()]
        t_batch, t_single, pts_total = [], [], 0
        for t in range(1, n_frames):
            imgs = frames[idx, t].contiguous()
            singles_in = [imgs[b] for b in range(B)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            nxt, ncnt, keep, n_new = batch.step_batch(imgs, pts, cnt, **DET)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            outs = [single[b].step(singles_in[b], spts[b], **DET) for b in range(B)]
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            if t > args.warmup:
                t_batch.append(t1 - t0)
                t_single.append(t2 - t1)
                pts_total += int(cnt.sum())
            # same outputs, and the next inputs of both arms
            hc, hn, hk = ncnt.cpu().numpy(), nxt.cpu().numpy(), keep.cpu().numpy()
            c_in = cnt.cpu().numpy()
            for b, (surv, k1, new) in enumerate(outs):
                s = int(hk[b].sum())
                new = np.zeros((0, 2), np.float32) if new is None else new.reshape(-1, 2)
                ok = (np.array_equal(hk[b, :c_in[b]], k1.cpu().numpy()) and not hk[b, c_in[b]:].any()
                      and np.array_equal(hn[b, :s].view(np.uint32), surv.cpu().numpy().view(np.uint32))
                      and np.array_equal(hn[b, s:hc[b]], new))
                if not ok:
                    sys.exit("B=%d step %d sequence %d: step_batch and step differ" % (B, t, b))
                spts[b] = torch.cat([surv, torch.from_numpy(new).cuda()])
            pts, cnt = nxt, ncnt
        mb, ms = float(np.median(t_batch)) * 1e3, float(np.median(t_single)) * 1e3
        emit({"batch": B, "step_batch_ms": round(mb, 4), "step_x_B_ms": round(ms, 4), "speedup": round(ms / mb, 3),
              "step_batch_ms_per_seq": round(mb / B, 4), "step_ms_per_seq": round(ms / B, 4),
              "step_batch_ms_min_max": [round(min(t_batch) * 1e3, 4), round(max(t_batch) * 1e3, 4)],
              "step_x_B_ms_min_max": [round(min(t_single) * 1e3, 4), round(max(t_single) * 1e3, 4)],
              "mean_points_per_seq": round(pts_total / (B * len(t_batch)), 1), "identical": True})
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
