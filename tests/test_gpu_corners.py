"""GPU tier (pytest -m gpu, B200) of the detection step (SURVEY.md s8f rank 2): the CUDA path, called through
the C ABI, against the committed golden vectors, the C oracle and live cv2.goodFeaturesToTrack /
cv2.cornerMinEigenVal (the reference's implementation, src/extractor/extractor.py:110-111) on the same inputs.

Bar: the eigenvalue map is bit-exact (float32 compared as uint32) and the returned corners are identical in
value AND order (integer pixel coordinates, strongest first)."""
import numpy as np
import pytest

from conftest import load_golden
from visual_odom_pipeline_b200 import synth as S

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def discs_mask(cv2, shape, n, seed, radius=10):
    rng = np.random.default_rng(seed)
    m = np.full(shape, 255, np.uint8)
    for _ in range(n):
        cv2.circle(m, (int(rng.integers(0, shape[1])), int(rng.integers(0, shape[0]))), radius, 0, -1)
    return m


def same(a, b):
    if a is None or b is None:
        return a is None and b is None
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b)


def assert_eig_equal(got, want):
    bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
    assert bad.size == 0, "%d / %d eigenvalues differ; first at %s: %r vs %r" % (len(bad), got.size, bad[0], got[tuple(bad[0])], want[tuple(bad[0])])


@pytest.mark.parametrize("name", ["gftt_reference", "gftt_default", "gftt_even_block", "gftt_block5"])
def test_detection_matches_golden(klt, name):
    g = load_golden(name)
    img, bs = g["img"], int(g["blockSize"])
    mask = g["mask"] if g["mask"].size else None
    assert_eig_equal(klt.cornerMinEigenVal(img, bs), g["eig"])
    c = klt.goodFeaturesToTrack(img, int(g["maxCorners"]), float(g["qualityLevel"]), float(g["minDistance"]), mask=mask, blockSize=bs)
    assert same(c, g["corners"] if len(g["corners"]) else None)


@pytest.mark.parametrize("hw", [(376, 1241), (480, 640), (768, 1024), (120, 161), (100, 101), (57, 43), (64, 96), (33, 200)])
@pytest.mark.parametrize("bs", [31, 3, 5, 7, 4])
def test_detection_bit_exact_vs_oracle_and_cv2(klt, oracle, cv2, hw, bs):
    if bs // 2 >= min(hw):
        pytest.skip("block larger than the image")
    img = S.frame_pair(hw[0], hw[1], seed=hw[1] + bs)[0]
    got = klt.cornerMinEigenVal(img, bs)
    assert_eig_equal(got, cv2.cornerMinEigenVal(img, bs, ksize=3))
    if hw[0] * hw[1] <= 640 * 480:
        assert_eig_equal(got, oracle.corner_min_eigen_val(img, bs))
    mask = discs_mask(cv2, img.shape, 30, bs)
    for (mc, ql, md, m) in [(1000, 0.03, 10, mask), (1000, 0.03, 7, None), (0, 0.01, 3.5, mask), (50, 0.2, 0, None), (200, 0.001, 25, mask),
                            (0, 0.01, 3.5, None), (300, 0.02, 25.5, mask), (0, 0.05, 1.0, None), (50, 0.01, 80, None)]:
        c = klt.goodFeaturesToTrack(img, mc, ql, md, mask=m, blockSize=bs)
        k = cv2.goodFeaturesToTrack(img, mc, ql, md, mask=m, blockSize=bs)
        assert same(c, k), "corners differ for maxCorners=%d quality=%g minDistance=%g mask=%s" % (mc, ql, md, m is not None)


def test_reference_call_pattern_extract(klt, cv2):
    """src/extractor/extractor.py:102-111: mask = 255 with a filled circle of radius mask_radius around every tracked
    keypoint, then goodFeaturesToTrack(img, mask=mask, maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)."""
    params = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)   # extractor.py:21-24, min_kp_dist=10
    img = S.frame_pair(376, 1241, seed=9)[0]
    tracked = S.uniform_points(400, 376, 1241, seed=10).reshape(-1, 2)
    mask = np.zeros_like(img)
    mask[:] = 255
    for x, y in [np.int32(p) for p in tracked]:
        cv2.circle(mask, (int(x), int(y)), 10, 0, -1)
    kp = klt.goodFeaturesToTrack(img.copy(), mask=mask, **params)
    ref = cv2.goodFeaturesToTrack(img.copy(), mask=mask, **params)
    assert same(kp, ref) and kp.shape[1:] == (1, 2) and kp.dtype == np.float32
    # every corner respects the mask and the minimum distance
    xy = kp.reshape(-1, 2).astype(int)
    assert (mask[xy[:, 1], xy[:, 0]] != 0).all()
    d = np.linalg.norm(kp.reshape(-1, 1, 2) - kp.reshape(1, -1, 2), axis=-1) + np.eye(len(kp)) * 1e9
    assert d.min() >= 10


def test_detection_edge_cases(klt, cv2):
    flat = np.full((60, 80), 77, np.uint8)
    assert klt.goodFeaturesToTrack(flat, 100, 0.01, 5, blockSize=7) is None
    img = S.frame_pair(60, 80, seed=4)[0]
    assert klt.goodFeaturesToTrack(img, 100, 0.01, 5, mask=np.zeros(img.shape, np.uint8), blockSize=7) is None
    # non-contiguous views (cv2 accepts any strides)
    big = S.frame_pair(120, 200, seed=5)[0]
    view, mview = big[::2, 10:170], discs_mask(cv2, big.shape, 10, 1)[::2, 10:170]
    assert same(klt.goodFeaturesToTrack(view, 200, 0.02, 6, mask=mview, blockSize=9), cv2.goodFeaturesToTrack(view, 200, 0.02, 6, mask=mview, blockSize=9))
    # (h, w, 1) image, inputs not mutated
    keep = img.copy()
    assert same(klt.goodFeaturesToTrack(img[:, :, None], 50, 0.01, 3, blockSize=5), cv2.goodFeaturesToTrack(img, 50, 0.01, 3, blockSize=5))
    assert np.array_equal(img, keep)


def test_plateaus_and_many_candidates(klt, cv2):
    """Periodic pattern: thousands of candidates with exactly equal eigenvalues -> tie order (later pixel first), the
    unsorted pass-through of the device sort (> 8192 keys) and the host radix sort."""
    per = np.tile(np.array([[0, 255], [255, 0]], np.uint8).repeat(8, 0).repeat(8, 1), (40, 60))
    assert per.shape == (640, 960)
    for md in (0, 4, 9.5):
        c = klt.goodFeaturesToTrack(per, 0, 0.01, md, blockSize=3)
        k = cv2.goodFeaturesToTrack(per, 0, 0.01, md, blockSize=3)
        assert same(c, k) and len(c) > (8192 if md == 0 else 100)
    assert_eig_equal(klt.cornerMinEigenVal(per, 3), cv2.cornerMinEigenVal(per, 3, ksize=3))


def test_full_size_stress_frame(klt, cv2):
    """BASELINE configs[4] frame shape (3840 x 2160): more candidates than the mapped staging buffer holds."""
    img = S.frame_pair(2160, 3840, seed=3)[0]
    assert_eig_equal(klt.cornerMinEigenVal(img, 31), cv2.cornerMinEigenVal(img, 31, ksize=3))
    mask = discs_mask(cv2, img.shape, 40, 5)
    for (mc, ql, md, m) in [(1000, 0.03, 10, None), (0, 0.01, 3.5, None), (300, 0.02, 25.5, mask), (50, 0.01, 80, None)]:
        assert same(klt.goodFeaturesToTrack(img, mc, ql, md, mask=m, blockSize=31), cv2.goodFeaturesToTrack(img, mc, ql, md, mask=m, blockSize=31))


def test_batched_device_api_equals_per_frame_host_calls(klt, cv2):
    import torch
    from visual_odom_pipeline_b200 import detector as D, tracker as T
    B, H, W = 5, 188, 621
    frames = [S.frame_pair(H, W, seed=80 + i)[0] for i in range(B)]
    masks = [discs_mask(cv2, (H, W), 20, i) for i in range(B)]
    dev = T.alloc_image_batch(B, H, W); dev.copy_(torch.from_numpy(np.stack(frames)))
    dmask = torch.from_numpy(np.stack(masks)).cuda()
    eig = D.corner_min_eigen_val(dev, 31)
    res = D.good_features_to_track(dev, 500, 0.03, 10, mask=dmask, blockSize=31)
    torch.cuda.synchronize()
    for b in range(B):
        assert_eig_equal(eig[b].cpu().numpy(), cv2.cornerMinEigenVal(frames[b], 31, ksize=3))
        assert same(res[b], cv2.goodFeaturesToTrack(frames[b], 500, 0.03, 10, mask=masks[b], blockSize=31)), "frame %d" % b


def _frame_loop(lk, gftt, cv2, frames, n_init):
    """The data-parallel part of the reference's per-frame step (src/pipeline/pipeline.py:92-103,159-163 with
    src/extractor/extractor.py:38-59, 61-88, 95-112): track candidate and landmark keypoints with two LK calls each, drop
    points by bidirectional error and the inclusive bounds test, mask discs around the survivors, detect new candidates."""
    lk_params = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))                    # extractor.py:16-19
    st_params = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)        # extractor.py:21-24
    h, w = frames[0].shape
    first = gftt(frames[0], mask=None, **st_params).reshape(-1, 2)
    landmarks, candidates = first[:n_init], first[n_init:]
    trace = []
    for t in range(1, len(frames)):
        im0, im1 = frames[t - 1], frames[t]
        groups = []
        for p0 in (candidates, landmarks):
            if len(p0) == 0:
                groups.append(p0)
                continue
            p0 = np.float32(p0).reshape(-1, 1, 2)
            p1, _st, _err = lk(im0, im1, p0, None, **lk_params)
            p0r, _st, _err = lk(im0, im1, p1, None, **lk_params)
            d = abs(p0 - p0r).reshape(-1, 2).max(-1)
            good = d < 30
            p1 = p1.reshape(-1, 2)
            keep = good & (0 <= p1[:, 0]) & (p1[:, 0] <= w) & (0 <= p1[:, 1]) & (p1[:, 1] <= h)
            groups.append(p1[keep])
        candidates, landmarks = groups
        mask = np.zeros_like(im1)
        mask[:] = 255
        for x, y in [np.int32(p) for p in np.concatenate([landmarks, candidates])]:
            cv2.circle(mask, (int(x), int(y)), 10, 0, -1)
        new = gftt(im1.copy(), mask=mask, **st_params)
        if new is not None:
            candidates = np.concatenate([candidates, new.reshape(-1, 2)])
        trace.append((landmarks.copy(), candidates.copy()))
    return trace


def test_reference_frame_loop_malaga_shape(klt, cv2):
    """BASELINE configs[2] shape (1024 x 768, ~3000 keypoints tracked frame to frame): the tracking + detection calls of
    the reference's step, chained over a sequence, give identical keypoint sets with this library and with cv2."""
    frames = S.sequence(768, 1024, 6, seed=12)
    got = _frame_loop(klt.calcOpticalFlowPyrLK, klt.goodFeaturesToTrack, cv2, frames, 600)
    want = _frame_loop(cv2.calcOpticalFlowPyrLK, cv2.goodFeaturesToTrack, cv2, frames, 600)
    assert len(got) == len(want) == 5
    for t, ((l1, c1), (l2, c2)) in enumerate(zip(got, want)):
        assert l1.shape == l2.shape and np.array_equal(l1.view(np.uint32), l2.view(np.uint32)), "landmarks differ at frame %d" % (t + 1)
        assert c1.shape == c2.shape and np.array_equal(c1.view(np.uint32), c2.view(np.uint32)), "candidates differ at frame %d" % (t + 1)
    assert len(got[-1][0]) + len(got[-1][1]) > 2000


def test_detection_is_deterministic_and_independent_of_candidate_order(klt, cv2):
    """The candidate list is appended with atomics (arbitrary order); the device sort makes the result a function of the
    image alone: repeated calls give identical corner lists, and so does a call on a context that ran other work."""
    img = S.frame_pair(376, 1241, seed=21)[0]
    mask = discs_mask(cv2, img.shape, 50, 3)
    ref = cv2.goodFeaturesToTrack(img, 1000, 0.03, 10, mask=mask, blockSize=31)
    runs = [klt.goodFeaturesToTrack(img, 1000, 0.03, 10, mask=mask, blockSize=31) for _ in range(5)]
    other = S.frame_pair(480, 640, seed=2)[0]
    klt.goodFeaturesToTrack(other, 300, 0.01, 5, blockSize=7)          # grows / reuses the context workspace differently
    runs.append(klt.goodFeaturesToTrack(img, 1000, 0.03, 10, mask=mask, blockSize=31))
    for r in runs:
        assert same(r, ref)


def test_eigenvalue_map_properties_at_full_size(klt):
    """Size-independent properties at the stress shape (3840 x 2160): flipping the frame flips the map (the running sums
    follow the flipped order, so this is a tolerance check, not bit-exact), a constant frame gives an all-zero map, and
    the map is non-negative up to rounding."""
    img = S.frame_pair(2160, 3840, seed=4)[0]
    e = klt.cornerMinEigenVal(img, 31)
    ef = klt.cornerMinEigenVal(np.ascontiguousarray(img[::-1, ::-1]), 31)[::-1, ::-1]
    scale = float(e.max())
    assert scale > 0 and np.abs(e - ef).max() <= 1e-5 * scale          # tolerance: float32 sums in a different order
    assert e.min() >= -1e-6 * scale
    assert not klt.cornerMinEigenVal(np.full((2160, 3840), 200, np.uint8), 31).any()


@pytest.mark.parametrize("radius", [0, 1, 5, 10, 31, 100])
def test_device_mask_from_points_equals_cv2_circle(klt, cv2, oracle, radius):
    import torch
    from visual_odom_pipeline_b200 import detector as D
    rng = np.random.default_rng(radius + 1)
    for shape in [(376, 1241), (61, 47)]:
        h, w = shape
        pts = np.stack([rng.uniform(-radius - 5, w + radius + 5, 300), rng.uniform(-radius - 5, h + radius + 5, 300)], -1).astype(np.float32)
        want = np.zeros(shape, np.uint8)
        want[:] = 255
        for x, y in [np.int32(p) for p in pts.astype(np.float64)]:
            cv2.circle(want, (int(x), int(y)), radius, 0, -1)
        got = D.mask_from_points(torch.from_numpy(pts).cuda(), radius, shape).cpu().numpy()
        assert np.array_equal(got, want) and np.array_equal(got, oracle.mask_from_points(pts, radius, shape))
    assert np.array_equal(D.mask_from_points(torch.zeros((0, 2), dtype=torch.float32, device="cuda"), 5, (20, 30)).cpu().numpy(),
                          np.full((20, 30), 255, np.uint8))


def test_fused_detection_from_tracked_points_equals_reference_step(klt, cv2):
    """detectNewFeatures(image, tracked, mask_radius) == the mask loop + cv2.goodFeaturesToTrack of extractor.py:102-111."""
    for hw, n_tracked, seed in [((376, 1241), 1500, 3), ((768, 1024), 3000, 4), ((120, 160), 0, 5)]:
        img = S.frame_pair(hw[0], hw[1], seed=seed)[0]
        tracked = S.uniform_points(max(n_tracked, 1), hw[0], hw[1], seed=seed + 1, margin=15).reshape(-1, 2)[:n_tracked]
        mask = np.zeros_like(img)
        mask[:] = 255
        for x, y in [np.int32(p) for p in tracked.astype(np.float64)]:
            cv2.circle(mask, (int(x), int(y)), 10, 0, -1)
        want = cv2.goodFeaturesToTrack(img, mask=mask, maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)
        got = klt.detectNewFeatures(img, tracked, 10)
        assert same(got, want), hw


def test_device_resident_frame_step_equals_cv2_loop(klt, cv2):
    """KLTTracker.step(): tracking + filtering + mask + detection of one frame on the device == the same steps with cv2
    (the reference's extend_tracks / extract sequence, src/extractor/extractor.py:38-59,102-111)."""
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    lk_params = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
    st_params = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)
    frames = S.sequence(376, 1241, 4, seed=14)
    h, w = frames[0].shape
    pts = cv2.goodFeaturesToTrack(frames[0], **st_params).reshape(-1, 2)
    trk = T.KLTTracker(**lk_params).reset(torch.from_numpy(frames[0]).cuda())
    dpts = torch.from_numpy(pts).cuda()
    for t in range(1, len(frames)):
        im0, im1 = frames[t - 1], frames[t]
        p0 = pts.reshape(-1, 1, 2)
        p1, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **lk_params)
        p0r, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **lk_params)
        good = abs(p0 - p0r).reshape(-1, 2).max(-1) < 30
        p1 = p1.reshape(-1, 2)
        keep_ref = good & (0 <= p1[:, 0]) & (p1[:, 0] <= w) & (0 <= p1[:, 1]) & (p1[:, 1] <= h)
        surv_ref = p1[keep_ref]
        mask = np.zeros_like(im1)
        mask[:] = 255
        for x, y in [np.int32(p) for p in surv_ref]:
            cv2.circle(mask, (int(x), int(y)), 10, 0, -1)
        new_ref = cv2.goodFeaturesToTrack(im1, mask=mask, **st_params)
        surv, keep, new = trk.step(torch.from_numpy(im1).cuda(), dpts)
        assert np.array_equal(keep.cpu().numpy(), keep_ref), "frame %d" % t
        assert np.array_equal(surv.cpu().numpy().view(np.uint32), surv_ref.view(np.uint32)), "frame %d" % t
        assert same(new, new_ref), "frame %d" % t
        pts = surv_ref if new_ref is None else np.concatenate([surv_ref, new_ref.reshape(-1, 2)])
        dpts = torch.from_numpy(np.ascontiguousarray(pts)).cuda()
