"""What contrast-limited equalisation costs: the createCLAHE drop-in against cv2 on the host, the batched kernels alone, and
KLTSequenceBatch with equalize off and on.

    python scripts/clahe_time.py [--batches 1,16,64] [--frames 40] [--warmup 5] [--reps 5] [--points 2000]
                                 [--capacity 4096] [--kernel-iters 50] [--out LOG]

KITTI shape (376 x 1241), createCLAHE(3.0, (8, 8)) (VINS-Mono's setting), frames of synth.exposure_sequence with the gains
1, 1, .7, .7, 1, .5, .5, 1, 1.4, 1 repeated.  Prints the card's name, power limit, maximum and current SM clock first.

- drop-in: createCLAHE(3.0, (8, 8)).apply(numpy frame) end to end (upload, two kernels, download), and cv2's apply on all
  of the host's threads and on one thread; median of 200 calls after 20 warm-up calls.
- kernel: filters.clahe's two launches on B frames, `kernel-iters` pairs in a row captured in one CUDA graph, timed with
  CUDA events around a replay (median of 5 replays), so the host's enqueue is not in the time.  The launches rotate through copies of the batch that together take at least 256 MB, so no launch finds its frames in the
  126 MB L2.  GB/s uses the algorithmic bytes: the padded frame read once (the histograms), the frame read once and
  written once (the blend) and the LUTs written once; the copy peak is a device-to-device copy of 1 GB (read + write).
- step: graph replay of KLTSequenceBatch (reference parameters, second_pass="reverse", max_bidir_error=1, capacity 4096),
  the arms off and equalize=(3.0, (8, 8)) alternated in every rep over the same frames, as scripts/subpix_time.py does:
  ms per frame (median over the reps, and [min, max]) with a host clock around work that ends in a device
  synchronisation, and the tracks kept per sequence and step.  Two workloads: "exposure" (the gains above) and "steady"
  (every gain 1, the same scenes), where the arms differ by the equalisation alone and not by what it does to the tracks.
"""
import argparse
import ctypes
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
EQ = (3.0, (8, 8))
GAINS = [1.0, 1.0, 0.7, 0.7, 1.0, 0.5, 0.5, 1.0, 1.4, 1.0]
ARMS = {"off": None, "equalize": EQ}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def host_ms(fn, warm=20, n=200):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return round(float(np.median(ts)) * 1e3, 4)


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
    import cv2
    import torch
    import visual_odom_pipeline_b200 as K
    from visual_odom_pipeline_b200 import _lib
    from visual_odom_pipeline_b200 import filters as F
    from visual_odom_pipeline_b200 import synth as S
    from visual_odom_pipeline_b200 import tracker as T
    if not torch.cuda.is_available():
        sys.exit("clahe_time.py needs a CUDA device")

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(s + "\n")

    C = args.capacity
    t0_timed = 2 + args.warmup
    n_frames = t0_timed + args.frames
    emit({"card": card(), "equalize": EQ, "points": args.points, "capacity": C, "frames": args.frames, "warmup": args.warmup,
          "reps": args.reps, "arms": list(ARMS), "host_threads": os.cpu_count()})

    gains = (GAINS * (n_frames // len(GAINS) + 1))[:n_frames]
    pool = [S.exposure_sequence(H, W, n_frames, gains, seed=100 + i) for i in range(args.pool)]

    # ---- the drop-in against cv2 on the host
    img = pool[0][5]
    mine, ref = K.createCLAHE(*EQ), cv2.createCLAHE(*EQ)
    assert np.array_equal(mine.apply(img), ref.apply(img))
    d = {"line": "drop-in", "shape": [H, W], "klt_ms": host_ms(lambda: mine.apply(img))}
    threads = cv2.getNumThreads()
    for nt in (os.cpu_count(), 1):
        cv2.setNumThreads(nt)
        d["cv2_%d_threads_ms" % nt] = host_ms(lambda: ref.apply(img))
    cv2.setNumThreads(threads)
    emit(d)

    # ---- the kernels alone
    frames = torch.from_numpy(np.stack([np.stack(s) for s in pool])).cuda()
    big = torch.empty((1 << 30,), dtype=torch.uint8, device="cuda")
    big2 = torch.empty_like(big)
    for _ in range(3):
        big2.copy_(big)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        big2.copy_(big)
    e1.record()
    torch.cuda.synchronize()
    copy_gbs = 2 * big.numel() * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del big, big2
    tx, ty = EQ[1]
    wext, hext = W + tx - W % tx, H + ty - H % ty           # KITTI divides neither axis by 8
    ctx = _lib.default_context(0)
    for B in [int(x) for x in args.batches.split(",")]:
        idx = [b % args.pool for b in range(B)]
        src = frames[idx, 5].contiguous()
        n_buf = max(1, -(-(256 << 20) // (2 * src.numel())))
        ins = [T.alloc_image_batch(B, H, W) for _ in range(n_buf)]
        outs = [T.alloc_image_batch(B, H, W) for _ in range(n_buf)]
        for x in ins:
            x.copy_(src)
        ws = torch.empty((int(_lib.load().klt_clahe_ws_bytes(B, tx, ty)),), dtype=torch.uint8, device="cuda")
        ctypes_stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        want = np.stack([ref.apply(x) for x in src.cpu().numpy()])
        F.clahe_launch(ins[0], outs[0], EQ[0], EQ[1], ws, ctx, ctypes_stream)
        torch.cuda.synchronize()
        assert np.array_equal(outs[0].cpu().numpy(), want)
        for i in range(n_buf):
            F.clahe_launch(ins[i], outs[i], EQ[0], EQ[1], ws, ctx, ctypes_stream)
        torch.cuda.synchronize()
        # the launches replayed from a CUDA graph, so that the host's enqueue of each launch is not in the timed window
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            gs = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            for i in range(args.kernel_iters):
                F.clahe_launch(ins[i % n_buf], outs[i % n_buf], EQ[0], EQ[1], ws, ctx, gs)
        g.replay()
        torch.cuda.synchronize()
        per = []
        for _ in range(5):
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            per.append(e0.elapsed_time(e1) / args.kernel_iters)
        ms = float(np.median(per))
        nbytes = B * (wext * hext + 2 * W * H + tx * ty * 256)
        emit({"line": "kernels", "batch": B, "ms": round(ms, 4), "algorithmic_MB": round(nbytes / 1e6, 3),
              "GB_s": round(nbytes / (ms * 1e-3) / 1e9, 1), "copy_peak_GB_s": round(copy_gbs, 1),
              "share_of_copy_peak": round(nbytes / (ms * 1e-3) / 1e9 / copy_gbs, 3), "buffers": n_buf})
        del ins, outs, g

    # ---- the frame step, off and on, alternated
    init = []
    for s in pool:
        c = K.goodFeaturesToTrack(ref.apply(s[0]), args.points, DET["qualityLevel"], DET["minDistance"], blockSize=DET["blockSize"])
        init.append(torch.from_numpy(c.reshape(-1, 2)).cuda())
    steady = torch.from_numpy(np.stack([np.stack(S.exposure_sequence(H, W, n_frames, [1.0] * n_frames, seed=100 + i))
                                        for i in range(args.pool)])).cuda()
    for (workload, src_frames), B in [(w, b) for w in (("exposure", frames), ("steady", steady))
                                      for b in [int(x) for x in args.batches.split(",")]]:
        idx = (torch.arange(B) % args.pool).tolist()
        imgs = [src_frames[idx, t].contiguous() for t in range(n_frames)]
        n = max(int(init[i].shape[0]) for i in idx)
        pts0 = torch.zeros((B, n, 2), dtype=torch.float32, device="cuda")
        cnt0 = torch.zeros((B,), dtype=torch.int32, device="cuda")
        for b, i in enumerate(idx):
            pts0[b, :init[i].shape[0]] = init[i]
            cnt0[b] = init[i].shape[0]
        times = {a: [] for a in ARMS}
        alive = {a: 0 for a in ARMS}
        for rep in range(args.reps + 1):            # rep 0: warm-up of both arms
            for a in ARMS:
                sb = T.KLTSequenceBatch(imgs[0], pts0, cnt0, C, equalize=ARMS[a], second_pass="reverse", max_bidir_error=1.0,
                                        **LK, **DET)
                sb.step(imgs[1])
                sb.capture()
                for t in range(2, t0_timed):
                    sb.step(imgs[t])
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for t in range(t0_timed, n_frames):
                    sb.step(imgs[t])
                    if rep == 0:
                        alive[a] += int(sb.keep.sum())      # warm-up rep only: synchronises
                torch.cuda.synchronize()
                times[a].append((time.perf_counter() - t0) / args.frames)
                sb.check()
        d = {"line": "step", "workload": workload, "batch": B}
        for a in ARMS:
            v = times[a][1:]
            d[a + "_ms"] = round(float(np.median(v)) * 1e3, 4)
            d[a + "_ms_min_max"] = [round(min(v) * 1e3, 4), round(max(v) * 1e3, 4)]
            d[a + "_kept_per_seq_step"] = round(alive[a] / args.frames / B, 1)
        d["added_ms"] = round(d["equalize_ms"] - d["off_ms"], 4)
        emit(d)


if __name__ == "__main__":
    main()
