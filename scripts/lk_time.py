"""Times the LK kernel alone (CUDA events) on the KITTI config for quick A/B runs; checks vs cv2."""
import ctypes, os, sys, statistics
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, cv2
import visual_odom_pipeline_b200 as K
from visual_odom_pipeline_b200 import synth as S, tracker as T

def run(win, crit, n=2000, B=1, hw=(376, 1241), reps=30, maxLevel=3):
    h, w = hw
    prs = [S.frame_pair(h, w, seed=7 + i) for i in range(min(B, 4))]
    a = T.alloc_image_batch(B, h, w); b = T.alloc_image_batch(B, h, w)
    for i in range(B):
        a[i].copy_(torch.from_numpy(prs[i % len(prs)][0])); b[i].copy_(torch.from_numpy(prs[i % len(prs)][1]))
    pts_h = np.stack([S.uniform_points(n, h, w, seed=3 + (i % 8)).reshape(n, 2) for i in range(B)])
    pts = torch.from_numpy(pts_h).cuda()
    P0 = T.DevicePyramid(a, win, maxLevel); P1 = T.DevicePyramid(b, win, maxLevel)
    for _ in range(3): out = T.lk_track(P0, P1, pts, criteria=crit, return_iters=True)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); T.lk_track(P0, P1, pts, criteria=crit); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    q, st, er, it = out
    rq, rs, re_ = cv2.calcOpticalFlowPyrLK(prs[0][0], prs[0][1], pts_h[0].reshape(-1, 1, 2), None, winSize=win, maxLevel=maxLevel, criteria=crit)
    ok = np.array_equal(rq.reshape(-1, 2).view(np.uint32), q[0].cpu().numpy().view(np.uint32)) and np.array_equal(rs.ravel(), st[0].cpu().numpy())
    m = (rs.ravel() == 1)
    ok = ok and np.array_equal(re_.ravel()[m].view(np.uint32), er[0].cpu().numpy()[m].view(np.uint32))
    print(f"win{win[0]} B={B} n={n}: LK median {statistics.median(ts)*1e3:.1f} us min {min(ts)*1e3:.1f} us  ({B*n/statistics.median(ts)/1e3:.2f} Mpts/s) iters/pt {it.float().mean().item():.2f} max {it.max().item()} bit-exact-vs-cv2={ok}", flush=True)

run((21, 21), (3, 30, 0.01))
run((31, 31), (3, 30, 0.03))
run((21, 21), (3, 30, 0.01), B=64)
run((31, 31), (3, 30, 0.03), B=64)
