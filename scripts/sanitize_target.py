"""Small workload that drives every kernel family once, for compute-sanitizer (scripts/gpu_sanitize.sh): the specialised LK
kernel at win 21 (both team sizes) / 31 on inputs that reach the class-sum tier and the serial replay (large displacement, noise, border
points), the generic LK kernel, the pyramid ring kernel, its one-launch build, the shuffle fallback, the re-pitch kernel, the
Shi-Tomasi kernels (products, running sums, candidates, sort, scatter), the circle mask, the track filter and the per-track
records of the chained step.  Results are checked against cv2 (the records: against the step's own outputs) so that a
sanitizer run is also a parity run."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, cv2, torch
import visual_odom_pipeline_b200 as K
from visual_odom_pipeline_b200 import synth as S, tracker as T, detector as D

bad = 0
def check(name, ok):
    global bad
    print("%-60s %s" % (name, "ok" if ok else "MISMATCH"), flush=True)
    bad += 0 if ok else 1

def lk_equal(got, ref):
    m = ref[1].ravel() == 1
    return (np.array_equal(got[0].view(np.uint32), ref[0].view(np.uint32)) and np.array_equal(got[1], ref[1])
            and np.array_equal(got[2].ravel()[m].view(np.uint32), ref[2].ravel()[m].view(np.uint32)))

h, w = 200, 336
for win, crit, motion, kw, margin in [((21, 21), (3, 30, 0.01), S.BENIGN, {}, 15), ((31, 31), (3, 30, 0.03), S.HARD, dict(noise_sigma=3.0), 40),
                                       ((21, 21), (3, 30, 0.01), S.HARD, dict(noise_sigma=4.0), 30), ((15, 9), (3, 20, 0.01), S.BENIGN, {}, 10)]:
    a, b = S.frame_pair(h, w, seed=5, motion=motion, **kw)
    p = S.uniform_points(260, h, w, seed=6, margin=margin)
    lk = dict(winSize=win, maxLevel=3, criteria=crit)
    check("calcOpticalFlowPyrLK win %s motion %s" % (win, motion[:2]), lk_equal(K.calcOpticalFlowPyrLK(a, b, p, None, **lk), cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk)))
# 2 warps per point: a 21x21 launch of more than 32 points per SM (klt_lk_fast.cu: lk_launch_fast)
n2 = 33 * K.default_context(0).sm_count
a, b = S.frame_pair(h, w, seed=5, motion=S.HARD, noise_sigma=4.0)
p = S.uniform_points(n2, h, w, seed=7, margin=30)
lk = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
check("calcOpticalFlowPyrLK win 21, %d points (2 warps per point)" % n2, lk_equal(K.calcOpticalFlowPyrLK(a, b, p, None, **lk), cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk)))
# batched device API: ring kernel + one-launch build on pitched storage, fallback on a plain contiguous odd-width tensor
imgs = T.alloc_image_batch(3, h, w)
base = [S.texture(h, w, seed=s).astype(np.uint8) for s in range(3)]
for i in range(3):
    imgs[i].copy_(torch.from_numpy(base[i]))
pyr = T.DevicePyramid(imgs, (21, 21), 3)
ok = True
for i in range(3):
    ref = base[i]
    for l in range(1, pyr.top + 1):
        ref = cv2.pyrDown(ref)
        ok = ok and np.array_equal(pyr.level(l)[i].cpu().numpy(), ref)
check("DevicePyramid (ring kernel, one-launch build) vs cv2.pyrDown", ok)
odd = torch.from_numpy(np.ascontiguousarray(base[0][:, :333])).cuda()
pyr2 = T.DevicePyramid(odd, (21, 21), 2)
check("DevicePyramid (unaligned rows: fallback kernel) vs cv2.pyrDown", np.array_equal(pyr2.level(1)[0].cpu().numpy(), cv2.pyrDown(base[0][:, :333])))
top, levels = K.buildOpticalFlowPyramid(base[1], (21, 21), 3)
ok, ref = True, base[1]
for l in range(1, top + 1):
    ref = cv2.pyrDown(ref)
    ok = ok and np.array_equal(levels[l], ref)
check("buildOpticalFlowPyramid (host entry point)", ok and top >= 1)
# tracker: two passes + filter on the device
trk = T.KLTTracker(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03)).reset(torch.from_numpy(base[0]).cuda())
a, b = S.frame_pair(h, w, seed=9)
trk.reset(torch.from_numpy(a).cuda())
p = S.uniform_points(200, h, w, seed=2)
p1, keep, bid, st, er = trk.track_filtered(torch.from_numpy(b).cuda(), torch.from_numpy(p.reshape(1, -1, 2)).cuda())
r1 = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
check("KLTTracker.track_filtered forward pass", np.array_equal(p1.cpu().numpy().reshape(-1, 2).view(np.uint32), r1[0].reshape(-1, 2).view(np.uint32)))
# detection
det = dict(maxCorners=300, qualityLevel=0.03, minDistance=10, blockSize=31)
mask = np.full((h, w), 255, np.uint8); mask[40:80, 100:180] = 0
got, ref = K.goodFeaturesToTrack(a, mask=mask, **det), cv2.goodFeaturesToTrack(a, mask=mask, **det)
check("goodFeaturesToTrack with mask", got is not None and ref is not None and got.shape == ref.shape and np.array_equal(got, ref))
check("cornerMinEigenVal", np.array_equal(K.cornerMinEigenVal(a, 31).view(np.uint32), cv2.cornerMinEigenVal(a, 31).view(np.uint32)))
pts = p.reshape(-1, 2)[:100].copy()
m_ref = np.full((h, w), 255, np.uint8)
for x_, y_ in [np.int32(q) for q in pts]:
    cv2.circle(m_ref, (int(x_), int(y_)), 10, 0, -1)
got = K.detectNewFeatures(a, pts, 10, **det)
ref = cv2.goodFeaturesToTrack(a, mask=m_ref, **det)
check("detectNewFeatures (mask rasterised on the device)", (got is None and ref is None) or (got is not None and ref is not None and got.shape == ref.shape and np.array_equal(got, ref)))
# per-track records of the chained step (track_records_kernel, track_window_kernel): ragged counts, one sequence empty, a
# ring of depth 3 that wraps; the last window column is the current points, survivors keep their first frame
seq = [S.sequence(h, w, 6, seed=40 + b) for b in range(3)]
init = [cv2.goodFeaturesToTrack(s[0], maxCorners=[0, 60, 200][b], qualityLevel=0.03, minDistance=10, blockSize=31) if b else None
        for b, s in enumerate(seq)]
padded = np.zeros((3, 200, 2), np.float32)
cnt = np.zeros(3, np.int32)
for b, c in enumerate(init):
    if c is not None:
        padded[b, :len(c)] = c.reshape(-1, 2)
        cnt[b] = len(c)
sb = T.KLTSequenceBatch(torch.from_numpy(np.stack([s[0] for s in seq])).cuda(), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(),
                        400, winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03), maxCorners=150, history=3)
ok = True
for t in range(1, 6):
    n0, ids0, ff0 = sb.counts.cpu().numpy(), sb.ids.cpu().numpy(), sb.first_frames.cpu().numpy()
    prev_ff = [dict(zip(ids0[b, :n0[b]].tolist(), ff0[b, :n0[b]].tolist())) for b in range(3)]
    sb.step(torch.from_numpy(np.stack([s[t] for s in seq])).cuda())
    win, pts, n = sb.window(3).cpu().numpy(), sb.points.cpu().numpy(), sb.counts.cpu().numpy()
    ids, ff = sb.ids.cpu().numpy(), sb.first_frames.cpu().numpy()
    for b in range(3):
        ok = ok and np.array_equal(win[b, :n[b], 2].view(np.uint32), pts[b, :n[b]].view(np.uint32)) and bool(np.isnan(win[b, n[b]:]).all())
        s_b = int(sb.keep[b].sum())
        ok = ok and all(ff[b, j] == prev_ff[b][int(ids[b, j])] for j in range(s_b)) and bool((ff[b, s_b:n[b]] == t).all())
check("KLTSequenceBatch history=3: first frames, window(3)", ok and sb.history().counts.shape == (3, 3))
torch.cuda.synchronize()
print("sanitize_target: %d mismatches" % bad)
sys.exit(1 if bad else 0)
