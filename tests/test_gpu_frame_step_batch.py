"""GPU tier (pytest -m gpu, B200) of KLTTracker.step_batch / klt_frame_step_batch: the per-frame step (forward LK, the
reference's second pass, bidirectional / bounds filter, detection mask, goodFeaturesToTrack) for a batch of sequences
with a different point count each.

Bar: per sequence and frame, keep, the survivors (float32 compared as uint32) and the new corners (value and order) equal
the cv2 loop of the reference (src/extractor/extractor.py:38-59,102-111) and KLTTracker.step on that sequence alone."""
import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S

pytestmark = pytest.mark.gpu

LK = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
DET = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)
KITTI = (376, 1241)


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def cv2_step(cv2, im0, im1, pts, det, radius=10, max_bidir=30):
    """The reference's step with cv2 -> keep (n,) bool, survivors (s, 2), new corners (k, 2), candidate count."""
    h, w = im1.shape
    if len(pts):
        p0 = pts.reshape(-1, 1, 2)
        p1, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **LK)
        p0r, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **LK)
        good = abs(p0 - p0r).reshape(-1, 2).max(-1) < max_bidir
        p1 = p1.reshape(-1, 2)
        keep = good & (0 <= p1[:, 0]) & (p1[:, 0] <= w) & (0 <= p1[:, 1]) & (p1[:, 1] <= h)
        surv = p1[keep]
    else:
        keep, surv = np.zeros(0, bool), np.zeros((0, 2), np.float32)
    mask = np.full_like(im1, 255)
    for x, y in [np.int32(p) for p in surv]:
        cv2.circle(mask, (int(x), int(y)), radius, 0, -1)
    new = cv2.goodFeaturesToTrack(im1, mask=mask, **det)
    new = np.zeros((0, 2), np.float32) if new is None else new.reshape(-1, 2)
    return keep, surv, new, candidate_count(cv2, im1, mask, det)


def candidate_count(cv2, img, mask, det):
    """Corners goodFeaturesToTrack sorts before its greedy selection: thresholded local maxima of the eigenvalue map."""
    eig = cv2.cornerMinEigenVal(img, det["blockSize"], ksize=3)
    mx = eig[mask != 0].max() if (mask != 0).any() else 0.0
    e = np.where(eig > np.float32(mx * det["qualityLevel"]), eig, 0).astype(np.float32)
    loc = (e == cv2.dilate(e, None)) & (e > 0) & (mask != 0)
    loc[0, :] = loc[-1, :] = False
    loc[:, 0] = loc[:, -1] = False
    return int(loc.sum())


def pad(pts_list, fill=np.nan):
    """(B, N, 2) float32 with N = the longest set; the slots behind each count hold `fill` (never read)."""
    n = max([len(p) for p in pts_list] + [0])
    out = np.full((len(pts_list), n, 2), fill, np.float32)
    for b, p in enumerate(pts_list):
        out[b, :len(p)] = p.reshape(-1, 2)
    return out, np.array([len(p) for p in pts_list], np.int32)


def unpack(out, counts_in, b):
    nxt, ncnt, keep, n_new = [t.cpu().numpy() for t in out]
    s = int(keep[b].sum())
    assert not keep[b, counts_in[b]:].any()
    assert int(ncnt[b]) == s + int(n_new[b])
    assert nxt.shape[1] == int(ncnt.max())
    return keep[b, :counts_in[b]], nxt[b, :s], nxt[b, s:int(ncnt[b])]


def check_against_cv2(cv2, seqs, init, det=DET, radius=10, expect_candidates=None):
    """Runs step_batch over the sequences (list of frame lists) and compares every sequence and frame with the cv2 loop.
    expect_candidates(b, t, count) asserts the candidate count of the cv2 frame (the path the frame takes)."""
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    trk = T.KLTTracker(**LK).reset(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda())
    pts = [p.reshape(-1, 2) for p in init]
    B = len(seqs)
    for t in range(1, len(seqs[0])):
        padded, cnt = pad(pts)
        out = trk.step_batch(torch.from_numpy(np.stack([s[t] for s in seqs])).cuda(), torch.from_numpy(padded).cuda(),
                             torch.from_numpy(cnt).cuda(), mask_radius=radius, **det)
        nxt = []
        for b in range(B):
            keep_ref, surv_ref, new_ref, n_cand = cv2_step(cv2, seqs[b][t - 1], seqs[b][t], pts[b], det, radius)
            if expect_candidates:
                expect_candidates(b, t, n_cand)
            keep, surv, new = unpack(out, cnt, b)
            assert np.array_equal(keep, keep_ref), "sequence %d frame %d: keep" % (b, t)
            assert np.array_equal(surv.view(np.uint32), surv_ref.view(np.uint32)), "sequence %d frame %d: survivors" % (b, t)
            assert np.array_equal(new, new_ref), "sequence %d frame %d: new corners (%d vs %d)" % (b, t, len(new), len(new_ref))
            nxt.append(np.concatenate([surv_ref, new_ref]))
        pts = nxt


def test_batch_with_ragged_counts_equals_cv2_loop(klt, cv2):
    """B = 6 KITTI-shape sequences over 4 frames: one without points, one whose points all lie outside the image, four
    seeded from cv2.goodFeaturesToTrack; every sequence and frame against the cv2 loop."""
    h, w = KITTI
    seqs = [S.sequence(h, w, 4, seed=30 + b) for b in range(6)]
    init = [np.zeros((0, 2), np.float32),
            np.array([[-40.0, 12.0], [w + 25.5, 100.0], [300.0, h + 60.0], [-5.0, -7.0]], np.float32)]
    for b in range(2, 6):
        p = cv2.goodFeaturesToTrack(seqs[b][0], **DET).reshape(-1, 2)
        init.append(p[: 200 + 150 * b])   # a different count per sequence
    check_against_cv2(cv2, seqs, init)


@pytest.mark.parametrize("prefilter", [None, (5, 1.5, 1.5)])
def test_batch_equals_single_sequence_step(klt, cv2, prefilter):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    h, w = KITTI
    B = 5
    seqs = [S.sequence(h, w, 4, seed=50 + b) for b in range(B)]
    pts = [np.zeros((0, 2), np.float32)] + [cv2.goodFeaturesToTrack(seqs[b][0], **DET).reshape(-1, 2)[: 100 + 300 * b] for b in range(1, B)]
    batch = T.KLTTracker(prefilter=prefilter, **LK).reset(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda())
    single = [T.KLTTracker(prefilter=prefilter, **LK).reset(torch.from_numpy(s[0]).cuda()) for s in seqs]
    for t in range(1, 4):
        padded, cnt = pad(pts)
        out = batch.step_batch(torch.from_numpy(np.stack([s[t] for s in seqs])).cuda(), torch.from_numpy(padded).cuda(),
                               torch.from_numpy(cnt).cuda(), **DET)
        nxt = []
        for b in range(B):
            surv1, keep1, new1 = single[b].step(torch.from_numpy(seqs[b][t]).cuda(), torch.from_numpy(pts[b]).cuda(), **DET)
            keep, surv, new = unpack(out, cnt, b)
            new1 = np.zeros((0, 2), np.float32) if new1 is None else new1.reshape(-1, 2)
            assert np.array_equal(keep, keep1.cpu().numpy()), "sequence %d frame %d" % (b, t)
            assert np.array_equal(surv.view(np.uint32), surv1.cpu().numpy().view(np.uint32)), "sequence %d frame %d" % (b, t)
            assert np.array_equal(new, new1), "sequence %d frame %d" % (b, t)
            nxt.append(np.concatenate([surv, new]))
        pts = nxt


def noise_sequence(h, w, n, seed):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (h, w), dtype=np.uint8) for _ in range(n)]


def blob_sequence(cv2, h, w, n, seed, motion=(1.1, -0.6, 0.15, 1.003)):
    """Sparse bright discs on black, moving: a few thousand candidates at blockSize 3, qualityLevel 0.001."""
    rng = np.random.default_rng(seed)
    f = np.zeros((h, w), np.float32)
    for _ in range(400):
        cv2.circle(f, (int(rng.integers(0, w)), int(rng.integers(0, h))), int(rng.integers(3, 12)), float(rng.integers(60, 255)), -1)
    f = cv2.GaussianBlur(f, (0, 0), 1.5)
    out = [np.clip(f, 0, 255).astype(np.uint8)]
    for _ in range(n - 1):
        f = S.warp(f, motion)
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return out


def test_more_candidates_than_the_device_sort_takes(klt, cv2):
    """Noise frames with blockSize 3 and qualityLevel 0.001 have more than 8192 candidates: unsorted keys, host selection.
    Alone, and in a batch with frames that stay under the limit and are selected on the device."""
    h, w = KITTI
    det = dict(maxCorners=500, qualityLevel=0.001, minDistance=10, blockSize=3)
    noise = noise_sequence(h, w, 3, seed=5)
    blobs = [blob_sequence(cv2, h, w, 3, seed=61 + b) for b in range(2)]

    def expect(kinds):
        def check(b, t, n):
            if kinds[b] == "noise":
                assert n > 8192, "noise frame has only %d candidates" % n
            else:
                assert 0 < n <= 8192, "blob frame has %d candidates" % n
        return check

    p_noise = cv2.goodFeaturesToTrack(noise[0], **det).reshape(-1, 2)[:300]
    check_against_cv2(cv2, [noise], [p_noise], det=det, expect_candidates=expect(["noise"]))
    p_blobs = [cv2.goodFeaturesToTrack(s[0], **det).reshape(-1, 2) for s in blobs]
    check_against_cv2(cv2, [blobs[0], noise, blobs[1]], [p_blobs[0], p_noise, p_blobs[1][:50]], det=det,
                      expect_candidates=expect(["blobs", "noise", "blobs"]))


@pytest.mark.parametrize("min_distance", [80, 0])
def test_min_distance_outside_the_device_selection(klt, cv2, min_distance):
    """minDistance 80 (selection radius over 63 pixels) and 0 (no grid in cv2): every frame is selected on the host."""
    h, w = KITTI
    det = dict(DET, minDistance=min_distance)
    seqs = [S.sequence(h, w, 3, seed=70 + b) for b in range(3)]
    init = [cv2.goodFeaturesToTrack(s[0], **det).reshape(-1, 2)[: 40 + 60 * b] for b, s in enumerate(seqs)]
    check_against_cv2(cv2, seqs[:1], init[:1], det=det)
    check_against_cv2(cv2, seqs, init, det=det)


def test_4k_frames_bitmap_over_shared_memory(klt, cv2):
    """3840 x 2160: the selection bitmap does not fit the kernel's 180 KB, so the host selects."""
    h, w = 2160, 3840
    seqs = [S.sequence(h, w, 3, seed=80 + b) for b in range(2)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 200 + 150 * b] for b, s in enumerate(seqs)]
    check_against_cv2(cv2, seqs, init)


def test_argument_errors(klt):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    from visual_odom_pipeline_b200.lk import error
    h, w = 64, 96
    frames = torch.from_numpy(np.stack([S.sequence(h, w, 2, seed=90 + b)[1] for b in range(3)])).cuda()
    trk = T.KLTTracker(**LK)
    pts = torch.full((3, 8, 2), 20.0, device="cuda")
    cnt = torch.tensor([8, 0, 3], dtype=torch.int32, device="cuda")
    with pytest.raises(error):
        trk.step_batch(frames, pts, cnt)                       # before reset
    trk.reset(frames)
    with pytest.raises(error):
        trk.step_batch(frames[:2], pts[:2], cnt[:2])           # batch differs from reset
    with pytest.raises(error):
        trk.step_batch(frames, pts[:2], cnt)                   # points of another batch
    with pytest.raises(error):
        trk.step_batch(frames, pts, cnt[:2])                   # counts of another batch
    with pytest.raises(error):
        trk.step_batch(frames, pts.double(), cnt)
    with pytest.raises(error):
        trk.step_batch(frames, pts, cnt.long())
    with pytest.raises(error):
        trk.step_batch(frames.float(), pts, cnt)
    with pytest.raises(error):
        trk.step_batch(frames, pts.cpu(), cnt)
    with pytest.raises(error):
        trk.step_batch(frames, pts, cnt, maxCorners=0)
    for bad in ([9, 0, 3], [8, -1, 3]):
        with pytest.raises(error):
            trk.step_batch(frames, pts, torch.tensor(bad, dtype=torch.int32, device="cuda"))
    # the tracker still works after the refusals
    nxt, ncnt, keep, n_new = trk.step_batch(frames, pts, cnt)
    assert nxt.shape[0] == 3 and int(ncnt.max()) == nxt.shape[1]
    assert not keep[1].any() and not keep[2, 3:].any()
