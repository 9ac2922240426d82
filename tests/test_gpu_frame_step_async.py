"""GPU tier (pytest -m gpu, B200) of KLTSequenceBatch / klt_frame_step_batch_async: the per-frame step for a batch of
sequences, chained on the device with no host synchronisation between frames, eagerly or replayed from CUDA graphs.

Bar: per sequence and frame, keep, the survivors (float32 compared as uint32), the new corners (value and order), the
counts and the track ids equal the cv2 loop of the reference (src/extractor/extractor.py:38-59,102-111) with the
capacity cap (cv2 gets maxCorners = min(maxCorners, C - survivors); no detection when that is 0) and ids kept on the host
alongside it.  Graph replay equals eager steps bit for bit."""
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


def candidate_count(cv2, img, mask, det):
    """Corners goodFeaturesToTrack sorts before its greedy selection: thresholded local maxima of the eigenvalue map."""
    eig = cv2.cornerMinEigenVal(img, det["blockSize"], ksize=3)
    mx = eig[mask != 0].max() if (mask != 0).any() else 0.0
    e = np.where(eig > np.float32(mx * det["qualityLevel"]), eig, 0).astype(np.float32)
    loc = (e == cv2.dilate(e, None)) & (e > 0) & (mask != 0)
    loc[0, :] = loc[-1, :] = False
    loc[:, 0] = loc[:, -1] = False
    return int(loc.sum())


def cv2_step(cv2, im0, im1, pts, det, cap, radius=10, max_bidir=30):
    """The reference's step with cv2 and the capacity cap -> keep (n,) bool, survivors (s, 2), new corners (k, 2),
    candidate count, whether the cap bound (fewer corners than cv2 returns with det's maxCorners)."""
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
    k = min(det["maxCorners"], cap - len(surv))
    new = np.zeros((0, 2), np.float32)
    if k > 0:
        c = cv2.goodFeaturesToTrack(im1, mask=mask, **dict(det, maxCorners=k))
        new = new if c is None else c.reshape(-1, 2)
    bound = False
    if k < det["maxCorners"]:
        full = cv2.goodFeaturesToTrack(im1, mask=mask, **det)
        bound = full is not None and len(full) > len(new)
    return keep, surv, new, candidate_count(cv2, im1, mask, det), bound


def pad(pts_list, n=None, fill=np.nan):
    """(B, N, 2) float32; the slots behind each count hold `fill` (never read)."""
    n = max([len(p) for p in pts_list] + [0]) if n is None else n
    out = np.full((len(pts_list), n, 2), fill, np.float32)
    for b, p in enumerate(pts_list):
        out[b, :len(p)] = p.reshape(-1, 2)
    return out, np.array([len(p) for p in pts_list], np.int32)


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


def make_batch(seqs, init, cap, det=DET, radius=10, prefilter=None):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init)
    return T.KLTSequenceBatch(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda(), torch.from_numpy(padded).cuda(),
                              torch.from_numpy(cnt).cuda(), cap, mask_radius=radius, prefilter=prefilter, **LK, **det)


def snapshot(sb):
    """Host copies of the object's current outputs (synchronises: test code only)."""
    return {k: getattr(sb, k).cpu().numpy() for k in ("points", "counts", "ids", "keep", "n_new")}


def check_against_cv2(cv2, seqs, init, cap, det=DET, radius=10, graph=False, expect_candidates=None, expect_bound=None):
    """Steps a KLTSequenceBatch over the sequences (graph: the first step eager, then captured and replayed) and compares
    every sequence and frame with the capped cv2 loop, ids kept on the host.  Returns the (frame, sequence) pairs where
    the cap bound and where it did not."""
    import torch
    sb = make_batch(seqs, init, cap, det, radius)
    pts = [p.reshape(-1, 2) for p in init]
    ids = [np.arange(len(p), dtype=np.int32) for p in pts]
    next_id = [len(p) for p in pts]
    B = len(seqs)
    bound, free = [], []
    for t in range(1, len(seqs[0])):
        cin = [len(p) for p in pts]
        sb.step(torch.from_numpy(np.stack([s[t] for s in seqs])).cuda())
        if graph and t == 1:
            sb.capture()
        out = snapshot(sb)
        sb.check()
        for b in range(B):
            keep_ref, surv_ref, new_ref, n_cand, was_bound = cv2_step(cv2, seqs[b][t - 1], seqs[b][t], pts[b], det, cap, radius)
            if expect_candidates:
                expect_candidates(b, t, n_cand)
            (bound if was_bound else free).append((t, b))
            s, k = len(surv_ref), len(new_ref)
            tag = "sequence %d frame %d" % (b, t)
            assert np.array_equal(out["keep"][b, :cin[b]], keep_ref), tag + ": keep"
            assert not out["keep"][b, cin[b]:].any(), tag + ": keep behind the count"
            assert int(out["counts"][b]) == s + k and int(out["n_new"][b]) == k, tag + ": counts (%d + %d expected, %d)" % (
                s, k, int(out["counts"][b]))
            assert np.array_equal(out["points"][b, :s].view(np.uint32), surv_ref.view(np.uint32)), tag + ": survivors"
            assert np.array_equal(out["points"][b, s:s + k], new_ref), tag + ": new corners"
            ids_ref = np.concatenate([ids[b][keep_ref], np.arange(next_id[b], next_id[b] + k, dtype=np.int32)])
            assert np.array_equal(out["ids"][b, :s + k], ids_ref), tag + ": ids"
            ids[b], next_id[b] = ids_ref, next_id[b] + k
            pts[b] = np.concatenate([surv_ref, new_ref])
    if expect_bound is not None:
        expect_bound(bound, free)
    return bound, free


def test_capacity_binds_on_some_frames(klt, cv2):
    """Five KITTI sequences over five frames with ragged counts (one empty, one with every point outside the image,
    three seeded from goodFeaturesToTrack); C = 1500 binds on some frames and not on others."""
    h, w = KITTI
    seqs = [S.sequence(h, w, 5, seed=130 + b) for b in range(5)]
    init = [np.zeros((0, 2), np.float32),
            np.array([[-40.0, 12.0], [w + 25.5, 100.0], [300.0, h + 60.0], [-5.0, -7.0]], np.float32)]
    for b in range(2, 5):
        init.append(cv2.goodFeaturesToTrack(seqs[b][0], **DET).reshape(-1, 2)[: 300 + 300 * b])

    def both(bound, free):
        assert bound, "the cap never bound"
        assert free, "the cap bound on every frame"
    check_against_cv2(cv2, seqs, init, 1500, expect_bound=both)


def test_capacity_never_binds_equals_step_batch(klt, cv2):
    """With a capacity that never binds, every frame equals KLTTracker.step_batch."""
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    h, w = KITTI
    B, C = 4, 4096
    seqs = [S.sequence(h, w, 4, seed=150 + b) for b in range(B)]
    init = [np.zeros((0, 2), np.float32)] + [cv2.goodFeaturesToTrack(seqs[b][0], **DET).reshape(-1, 2)[: 200 + 300 * b] for b in range(1, B)]
    sb = make_batch(seqs, init, C)
    trk = T.KLTTracker(**LK).reset(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda())
    padded, cnt = pad(init)
    pts, counts = torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda()
    for t in range(1, 4):
        frames = torch.from_numpy(np.stack([s[t] for s in seqs])).cuda()
        nxt, ncnt, keep, n_new = trk.step_batch(frames, pts, counts, **DET)
        sb.step(frames)
        out = snapshot(sb)
        sb.check()
        n_in = pts.shape[1]
        assert int(ncnt.max()) <= C
        assert np.array_equal(out["counts"], ncnt.cpu().numpy())
        assert np.array_equal(out["n_new"], n_new.cpu().numpy())
        assert np.array_equal(out["keep"][:, :n_in], keep.cpu().numpy()) and not out["keep"][:, n_in:].any()
        hn, hc = nxt.cpu().numpy(), ncnt.cpu().numpy()
        for b in range(B):
            assert np.array_equal(out["points"][b, :hc[b]].view(np.uint32), hn[b, :hc[b]].view(np.uint32)), "sequence %d frame %d" % (b, t)
        pts, counts = nxt.contiguous(), ncnt


@pytest.mark.parametrize("B", [4, 6])
@pytest.mark.parametrize("prefilter", [None, (5, 1.5, 1.5)])
def test_graph_replay_equals_eager(klt, cv2, B, prefilter):
    """Six frames, both parities of the ping-pong slots replayed from the graphs, against an eager twin, bit for bit.
    B = 4 builds pyramids in thread-block clusters, B = 6 with the grid build.  Capture fails if anything in the step
    synchronises."""
    import torch
    h, w = KITTI
    seqs = [S.sequence(h, w, 7, seed=170 + b) for b in range(B)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 100 + 200 * b] for b, s in enumerate(seqs)]
    init[0] = init[0][:0]
    eager = make_batch(seqs, init, 1800, prefilter=prefilter)
    graph = make_batch(seqs, init, 1800, prefilter=prefilter)
    for t in range(1, 7):
        frames = torch.from_numpy(np.stack([s[t] for s in seqs])).cuda()
        eager.step(frames)
        graph.step(frames)
        if t == 1:
            graph.capture()
        a, b = snapshot(eager), snapshot(graph)
        for k in a:
            assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), "frame %d: %s" % (t, k)
        eager.check()
        graph.check()
    assert graph._graphs is not None


@pytest.mark.parametrize("graph", [False, True])
def test_more_than_8192_candidates_on_the_device(klt, cv2, graph):
    """Noise frames (blockSize 3, qualityLevel 0.001: more than 8192 candidates, radix sort) in one batch with blob
    frames that stay under 8192 (rank sort)."""
    h, w = KITTI
    det = dict(maxCorners=500, qualityLevel=0.001, minDistance=10, blockSize=3)
    noise = noise_sequence(h, w, 3, seed=5)
    blobs = [blob_sequence(cv2, h, w, 3, seed=61 + b) for b in range(2)]
    kinds = ["blobs", "noise", "blobs"]

    def check(b, t, n):
        if kinds[b] == "noise":
            assert n > 8192, "noise frame has only %d candidates" % n
        else:
            assert 0 < n <= 8192, "blob frame has %d candidates" % n
    init = [cv2.goodFeaturesToTrack(blobs[0][0], **det).reshape(-1, 2), cv2.goodFeaturesToTrack(noise[0], **det).reshape(-1, 2)[:300],
            cv2.goodFeaturesToTrack(blobs[1][0], **det).reshape(-1, 2)[:50]]
    check_against_cv2(cv2, [blobs[0], noise, blobs[1]], init, 1200, det=det, graph=graph, expect_candidates=check)


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("min_distance", [80, 0])
def test_min_distance_80_and_0(klt, cv2, min_distance, graph):
    """minDistance 80 (selection radius over 63 pixels) and 0 (no grid in cv2: the first candidates)."""
    h, w = KITTI
    det = dict(DET, minDistance=min_distance)
    seqs = [S.sequence(h, w, 3, seed=70 + b) for b in range(3)]
    init = [cv2.goodFeaturesToTrack(s[0], **det).reshape(-1, 2)[: 40 + 60 * b] for b, s in enumerate(seqs)]
    check_against_cv2(cv2, seqs, init, 2000, det=det, graph=graph)


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("min_distance", [10, 80])
def test_4k_frames_bitmap_in_global_memory(klt, cv2, graph, min_distance):
    """3840 x 2160: the selection bitmap exceeds 180 KB of shared memory and lives in global memory; minDistance 80
    adds a selection radius over 63 pixels (half widths per row, 64-bit distances) to it."""
    h, w = 2160, 3840
    det = dict(DET, minDistance=min_distance)
    seqs = [S.sequence(h, w, 3, seed=80 + b) for b in range(2)]
    init = [cv2.goodFeaturesToTrack(s[0], **det).reshape(-1, 2)[: 200 + 150 * b] for b, s in enumerate(seqs)]
    check_against_cv2(cv2, seqs, init, 2000, det=det, graph=graph)


def dots(n, seed=0, shape=KITTI):
    """n isolated one-pixel dots on a 4-pixel grid: exactly n candidates at blockSize 3, many of equal strength."""
    h, w = shape
    img = np.zeros((h, w), np.uint8)
    ys, xs = np.mgrid[4:h - 4:4, 4:w - 4:4]
    rng = np.random.default_rng(seed)
    img[ys.ravel()[:n], xs.ravel()[:n]] = rng.integers(100, 256, n).astype(np.uint8)
    return img


@pytest.mark.parametrize("min_distance", [3, 0])
def test_sort_boundary_and_ties(klt, cv2, min_distance):
    """Frames with exactly 8192 (rank sort) and 8193 (radix sort) candidates, and a periodic texture (np.tile of a small
    random patch: thousands of equal eigenvalues, so the tie order of the radix sort decides), every candidate selected
    (maxCorners above the candidate counts)."""
    h, w = KITTI
    det = dict(maxCorners=40000, qualityLevel=0.01, minDistance=min_distance, blockSize=3)
    rng = np.random.default_rng(3)
    tile = np.tile(rng.integers(0, 256, (8, 8), dtype=np.uint8), (h // 8 + 1, w // 8 + 1))[:h, :w]
    frames = [dots(8192, seed=1), dots(8193, seed=2), tile]
    full = np.full((h, w), 255, np.uint8)
    counts = [candidate_count(cv2, f, full, det) for f in frames]
    assert counts[0] == 8192 and counts[1] == 8193 and counts[2] > 8192, counts
    seqs = [[f, f] for f in frames]
    check_against_cv2(cv2, seqs, [np.zeros((0, 2), np.float32)] * 3, 40000, det=det)


def test_track_ids(klt, cv2):
    """Ids given at construction: survivors keep theirs in input order, new ids are consecutive from the largest given id
    + 1, strongest first; after several frames they match bookkeeping on the host (check_against_cv2 covers the default
    ids 0 .. n - 1)."""
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    h, w = KITTI
    seqs = [S.sequence(h, w, 4, seed=190 + b) for b in range(3)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 100 + 200 * b] for b, s in enumerate(seqs)]
    padded, cnt = pad(init)
    given = np.zeros(cnt.shape + (padded.shape[1],), np.int32)
    for b in range(3):
        given[b, :cnt[b]] = 1000 * (b + 1) + 7 * np.arange(cnt[b])
    sb = T.KLTSequenceBatch(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda(), torch.from_numpy(padded).cuda(),
                            torch.from_numpy(cnt).cuda(), 1500, ids=torch.from_numpy(given).cuda(), **LK, **DET)
    ids = [given[b, :cnt[b]] for b in range(3)]
    next_id = [int(given[b, :cnt[b]].max()) + 1 for b in range(3)]
    for t in range(1, 4):
        n_in = [len(i) for i in ids]
        sb.step(torch.from_numpy(np.stack([s[t] for s in seqs])).cuda())
        out = snapshot(sb)
        for b in range(3):
            keep = out["keep"][b, :n_in[b]]
            k = int(out["n_new"][b])
            ref = np.concatenate([ids[b][keep], np.arange(next_id[b], next_id[b] + k, dtype=np.int32)])
            assert np.array_equal(out["ids"][b, :int(out["counts"][b])], ref), "sequence %d frame %d" % (b, t)
            ids[b], next_id[b] = ref, next_id[b] + k
    sb.check()


def test_errors(klt):
    import torch
    from visual_odom_pipeline_b200 import _lib
    from visual_odom_pipeline_b200 import tracker as T
    from visual_odom_pipeline_b200.lk import error
    h, w = 64, 96
    frames = torch.from_numpy(np.stack([S.sequence(h, w, 2, seed=90 + b)[1] for b in range(3)])).cuda()
    pts = torch.full((3, 8, 2), 20.0, device="cuda")
    cnt = torch.tensor([8, 0, 3], dtype=torch.int32, device="cuda")
    for bad in ([9, 0, 3], [8, -1, 3]):
        with pytest.raises(error):
            T.KLTSequenceBatch(frames, pts, torch.tensor(bad, dtype=torch.int32, device="cuda"), 16)
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts, cnt, 4)                       # more points than the capacity
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts[:2], cnt, 16)                  # points of another batch
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts, cnt[:2], 16)                  # counts of another batch
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts.double(), cnt, 16)
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts, cnt.long(), 16)
    with pytest.raises(error):
        T.KLTSequenceBatch(frames.float(), pts, cnt, 16)
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts.cpu(), cnt, 16)
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts, cnt.cpu(), 16)
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts, cnt, 16, ids=torch.zeros((3, 8), dtype=torch.int64, device="cuda"))
    with pytest.raises(error):
        T.KLTSequenceBatch(frames, pts, cnt, 16, maxCorners=0)
    sb = T.KLTSequenceBatch(frames, pts, cnt, 16)
    with pytest.raises(error):
        sb.capture()                                                   # before an eager step
    with pytest.raises(error):
        sb.step(frames[:2])
    # a direct ABI call whose counts lie outside [0, n_per_seq]: the kernels clamp, the flag is set, nothing faults
    L = _lib.load()
    C = sb.capacity
    for bad in (C + 1, -1):
        cur, nxt = sb._cur, 1 - sb._cur
        sb._counts[cur, 1] = bad
        prev, new = sb._slots[cur], sb._slots[nxt]
        new.images.copy_(frames)
        new.build()
        rc = L.klt_frame_step_batch_async(
            sb.ctx.handle, prev.images.data_ptr(), prev.buffer.data_ptr(), new.images.data_ptr(), new.buffer.data_ptr(),
            prev.layout, 0, 0, 1, 3, sb._pts[cur].data_ptr(), sb._counts[cur].data_ptr(), C, sb.params, 30.0, 10, 1000, 0.03, 10.0, 31,
            sb._pts[nxt].data_ptr(), C, sb._keep.data_ptr(), sb._counts[nxt].data_ptr(), sb._n_new.data_ptr(), sb._ids[cur].data_ptr(),
            sb._ids[nxt].data_ptr(), sb._next_id.data_ptr(), sb._flags.data_ptr(), sb._ws_ptr, sb._ws_bytes,
            torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        sb._cur = nxt
        torch.cuda.synchronize()
        assert int(sb._flags.item()) == 1
        assert 0 <= int(sb.counts.min()) and int(sb.counts.max()) <= C
        with pytest.raises(error):
            sb.check()
        # the next call works, and reports nothing
        sb.step(frames)
        sb.check()
        assert 0 <= int(sb.counts.min()) and int(sb.counts.max()) <= C
    # argument checks of the entry point itself
    assert L.klt_frame_step_batch_async(
        sb.ctx.handle, prev.images.data_ptr(), prev.buffer.data_ptr(), new.images.data_ptr(), new.buffer.data_ptr(), prev.layout,
        0, 0, 1, 3, sb._pts[0].data_ptr(), sb._counts[0].data_ptr(), C, sb.params, 30.0, 10, 1000, 0.03, 10.0, 31,
        sb._pts[1].data_ptr(), C - 1, sb._keep.data_ptr(), sb._counts[1].data_ptr(), sb._n_new.data_ptr(), None, None, None,
        sb._flags.data_ptr(), sb._ws_ptr, sb._ws_bytes, None) == _lib.KLT_ERR_INVALID_ARG          # out_stride < n_per_seq
    assert L.klt_frame_step_batch_async(
        sb.ctx.handle, prev.images.data_ptr(), prev.buffer.data_ptr(), new.images.data_ptr(), new.buffer.data_ptr(), prev.layout,
        0, 0, 1, 3, sb._pts[0].data_ptr(), sb._counts[0].data_ptr(), C, sb.params, 30.0, 10, 1000, 0.03, 10.0, 31,
        sb._pts[1].data_ptr(), C, sb._keep.data_ptr(), sb._counts[1].data_ptr(), sb._n_new.data_ptr(), None, None, None,
        None, sb._ws_ptr, sb._ws_bytes, None) == _lib.KLT_ERR_INVALID_ARG                          # no flag word
