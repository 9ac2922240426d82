"""CPU tier of the motion prior of KLTSequenceBatch (motion_prior="given" / "velocity"): the host reference the GPU tier
compares against (the velocity rule in numpy float32 and the cv2 step with start positions), a property of that
reference (the velocity prior follows a motion that LK cannot capture from a zero start), and the argument checks of the
two entry points that run before any device work."""
import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S

DET = dict(maxCorners=1000, qualityLevel=0.03, minDistance=10, blockSize=31)
KITTI = (376, 1241)
# the property case: one pyramid level, a 21 x 21 window, fine texture, 6 px in the first step and 12 px in every later one
FAST_LK = dict(winSize=(21, 21), maxLevel=0, criteria=(3, 30, 0.03))
FAST_STEPS = [(6.0, -1.0)] + [(12.0, -2.0)] * 6


def velocity_starts(pts, prev):
    """pts (n, 2) float32, the current positions p; prev (n, 2) float32, each track's position q one frame ago, NaN where it
    has none -> start positions: p + (p - q) in float32 (each operation rounded once), p where q is NaN."""
    pts = np.asarray(pts, np.float32).reshape(-1, 2)
    prev = np.asarray(prev, np.float32).reshape(-1, 2)
    has = ~np.isnan(prev[:, 0])
    out = pts.copy()
    out[has] = pts[has] + (pts[has] - prev[has])
    return out


def lk_keep_from(cv2, lk, im0, im1, pts, starts, max_bidir=30):
    """The tracking half of the reference's step with the forward pass started at `starts`
    (cv2.OPTFLOW_USE_INITIAL_FLOW); the second pass starts from the forward result as always -> keep (n,) bool, p1 (n, 2)."""
    h, w = im1.shape
    if not len(pts):
        return np.zeros(0, bool), np.zeros((0, 2), np.float32)
    p0 = np.asarray(pts, np.float32).reshape(-1, 1, 2)
    s = np.array(starts, np.float32).reshape(-1, 1, 2)
    p1, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p0, s, flags=cv2.OPTFLOW_USE_INITIAL_FLOW, **lk)
    p0r, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **lk)
    good = abs(p0 - p0r).reshape(-1, 2).max(-1) < max_bidir
    p1 = p1.reshape(-1, 2)
    return good & (0 <= p1[:, 0]) & (p1[:, 0] <= w) & (0 <= p1[:, 1]) & (p1[:, 1] <= h), p1


def detect(cv2, im1, surv, cap, radius=10):
    """The detection half of the reference's step with the capacity cap: the corners cv2 finds around the survivors."""
    mask = np.full_like(im1, 255)
    for x, y in [np.int32(p) for p in surv]:
        cv2.circle(mask, (int(x), int(y)), radius, 0, -1)
    k = min(DET["maxCorners"], cap - len(surv))
    if k <= 0:
        return np.zeros((0, 2), np.float32)
    c = cv2.goodFeaturesToTrack(im1, mask=mask, **dict(DET, maxCorners=k))
    return np.zeros((0, 2), np.float32) if c is None else c.reshape(-1, 2)


def fine_sequence(cv2, h, w, steps, seed, sigma=1.5):
    """Frames of white noise blurred at sigma (little texture beyond a few pixels), each translated by steps[t] from the
    one before."""
    rng = np.random.default_rng(seed)
    f = cv2.GaussianBlur(rng.standard_normal((h, w)).astype(np.float32), (0, 0), sigma)
    f = (f - f.min()) / (f.max() - f.min()) * 255.0
    out = [np.clip(f, 0, 255).astype(np.uint8)]
    for tx, ty in steps:
        f = S.warp(f, (tx, ty, 0.0, 1.0))
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return out


def host_loop(cv2, seq, init, cap, lk, velocity):
    """One sequence through the reference's capped loop, the forward pass started by the velocity rule (or at p) ->
    per step: (survivors, survivors within 0.5 px of the true translation)."""
    pts = np.asarray(init, np.float32).reshape(-1, 2)
    prev = np.full_like(pts, np.nan)
    out = []
    for t in range(1, len(seq)):
        starts = velocity_starts(pts, prev) if velocity else pts
        keep, p1 = lk_keep_from(cv2, lk, seq[t - 1], seq[t], pts, starts)
        surv = p1[keep]
        err = abs(surv - pts[keep] - np.float32(FAST_STEPS[t - 1])).max(-1) if len(surv) else np.zeros(0)
        out.append((len(surv), int((err <= 0.5).sum())))
        new = detect(cv2, seq[t], surv, cap)
        prev = np.concatenate([pts[keep], np.full_like(new, np.nan)])
        pts = np.concatenate([surv, new]).astype(np.float32)
    return out


# survivors on the true motion per step, from host_loop on fine_sequence(cv2, 376, 1241, FAST_STEPS, seed=5), C = 1500
# (cv2 4.13): the first step has no velocity yet, so both loops agree there
FAST_ON_MOTION = {None: [595, 43, 96, 150, 197, 252, 299], "velocity": [595, 590, 608, 630, 649, 672, 675]}


def test_velocity_rule_rounds_like_numpy_float32():
    p = np.array([[1e8, 3.0], [0.1, 7.25], [5.0, 5.0]], np.float32)
    q = np.array([[1e8 - 8.0, 2.5], [np.nan, np.nan], [5.0, 6.0]], np.float32)
    s = velocity_starts(p, q)
    assert s.dtype == np.float32
    assert np.array_equal(s[0], np.float32([1e8 + 8.0, 3.5])) and np.array_equal(s[1], p[1]) and np.array_equal(s[2], [5.0, 4.0])
    # rounded twice in float32, not once in double: (0.1 + (0.1 - 0.3)) differs between the two
    a, b = np.float32(0.1), np.float32(0.3)
    assert velocity_starts([[a, a]], [[b, b]])[0, 0] == np.float32(a + np.float32(a - b))


def test_velocity_follows_a_motion_lk_cannot_capture_from_zero(cv2_mod):
    """maxLevel 0, a 21 x 21 window, fine texture: after a 6 px step, 12 px per frame is beyond what LK captures from the
    old position, so without a prior most survivors are tracks that LK lost but that stay in the image (the reference's
    filter keeps them); the velocity prior keeps more than twice as many tracks on the true motion in every later step.
    The raw survivor counts stay close."""
    cv2 = cv2_mod
    h, w = KITTI
    seq = fine_sequence(cv2, h, w, FAST_STEPS, seed=5)
    init = cv2.goodFeaturesToTrack(seq[0], **DET).reshape(-1, 2)
    got = {m: host_loop(cv2, seq, init, 1500, FAST_LK, m == "velocity") for m in (None, "velocity")}
    for m, want in FAST_ON_MOTION.items():
        assert [o for _n, o in got[m]] == want, (m, got[m])
    for t in range(1, len(FAST_STEPS)):
        assert got["velocity"][t][1] > 2 * got[None][t][1]
        assert abs(got["velocity"][t][0] - got[None][t][0]) < 0.05 * got[None][t][0]


@pytest.fixture(scope="module")
def cv2_mod():
    return pytest.importorskip("cv2")


def test_entry_points_reject_null_pointers(klt):
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    for name in ("klt_frame_step_batch_init_async", "klt_track_predict"):
        assert hasattr(L, name) and name in _lib.SYMBOLS
    inval = _lib.KLT_ERR_INVALID_ARG
    lay = _lib.klt_pyr_layout()
    prm = _lib.klt_lk_params()
    args = [None, None, None, None, None, lay, 0, 0, 1, 1, None, None, 0, prm, 30.0, 10, 100, 0.03, 10.0, 31, None, 100, None,
            None, None, None, None, None, None, None, 0]
    # a null context (with and without start positions and control), a null d_init_pts with points: rejected before
    # anything touches a device
    assert L.klt_frame_step_batch_init_async(*args, None, None, None) == inval
    assert L.klt_frame_step_batch_init_async(*args, 16, _lib.klt_step_control(), None) == inval
    args[12] = 8
    assert L.klt_frame_step_batch_init_async(*args, None, None, None) == inval
    # klt_track_predict(ctx, n_seqs, n_per_seq, pts, counts, guess_pts, guess_mask, depth, ring_pts, ring_src, ring_counts,
    # frame, init, stream)
    good = [None, 2, 8, 16, 16, 16, 16, 2, 16, 16, 16, 16, 16, None]
    for i, v in [(0, None), (1, 0), (2, -1), (7, -1), (7, 1)]:
        a = list(good)
        a[i] = v
        assert L.klt_track_predict(*a) == inval, (i, v)
    assert L.klt_track_predict(*good) == inval                       # the null context
