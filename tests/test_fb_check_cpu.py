"""CPU tier of the forward-backward check (second_pass="reverse"): the host reference the GPU tier compares against (the
mirrored start in numpy float32 and the cv2 step whose second pass runs from the new frame back into the old one), two
properties of that reference against the reference's same-direction pass, and the argument checks of the two new entry
points that run before any device work."""
import numpy as np
import pytest

from test_motion_prior_cpu import DET, FAST_LK, FAST_STEPS, KITTI, detect, fine_sequence, velocity_starts

# the library's own parameters (KLTTracker / KLTSequenceBatch defaults, the reference's _lk_params)
REF_LK = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
# fast translations of the blurred-noise sequence: above about 15 px per frame the same-direction pass moves a correct
# track by twice the motion, so d >= 30 for every track
FAST_MOTIONS = {16: [(16.0, -1.0)] * 5, 20: [(20.0, -1.0)] * 5}
FB_CAP = 1500
FB_MAX_ERR = 1.0


def mirror_start(p0, p1, starts):
    """Start of the reverse pass after a forward pass started at `starts`: p1 - (s - p0) in float32, each operation
    rounded once (the forward pass started s - p0 away from p0; the reverse pass starts as far from p1 the other way)."""
    p0 = np.asarray(p0, np.float32).reshape(-1, 2)
    p1 = np.asarray(p1, np.float32).reshape(-1, 2)
    s = np.asarray(starts, np.float32).reshape(-1, 2)
    return p1 - (s - p0)


def fb_keep_from(cv2, lk, im0, im1, pts, starts, max_bidir=FB_MAX_ERR, mirror=True):
    """The tracking half of the step with the forward-backward check.  starts None: both passes start without the flag
    (the reverse pass at p1); else the forward pass starts at `starts` (cv2.OPTFLOW_USE_INITIAL_FLOW) and the reverse pass
    at mirror_start with the flag (mirror=False: at p1 without it, for comparison) -> keep (n,) bool, p1 (n, 2), d (n,)."""
    h, w = im1.shape
    if not len(pts):
        return np.zeros(0, bool), np.zeros((0, 2), np.float32), np.zeros(0, np.float32)
    p0 = np.asarray(pts, np.float32).reshape(-1, 1, 2)
    if starts is None:
        p1, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **lk)
    else:
        s = np.array(starts, np.float32).reshape(-1, 1, 2)
        p1, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p0, s, flags=cv2.OPTFLOW_USE_INITIAL_FLOW, **lk)
    if starts is not None and mirror:
        b = mirror_start(p0, p1, starts).reshape(-1, 1, 2)
        p0r, _s, _e = cv2.calcOpticalFlowPyrLK(im1, im0, p1, b, flags=cv2.OPTFLOW_USE_INITIAL_FLOW, **lk)
    else:
        p0r, _s, _e = cv2.calcOpticalFlowPyrLK(im1, im0, p1, None, **lk)
    d = abs(p0 - p0r).reshape(-1, 2).max(-1)
    p1 = p1.reshape(-1, 2)
    keep = (d < max_bidir) & (0 <= p1[:, 0]) & (p1[:, 0] <= w) & (0 <= p1[:, 1]) & (p1[:, 1] <= h)
    return keep, p1, d


def same_direction_keep(cv2, lk, im0, im1, pts, max_bidir=30):
    """The reference's check (second pass im0 -> im1 from p1), as KLTTracker and the step run it by default."""
    h, w = im1.shape
    p0 = np.asarray(pts, np.float32).reshape(-1, 1, 2)
    p1, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **lk)
    p0r, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **lk)
    d = abs(p0 - p0r).reshape(-1, 2).max(-1)
    p1 = p1.reshape(-1, 2)
    return (d < max_bidir) & (0 <= p1[:, 0]) & (p1[:, 0] <= w) & (0 <= p1[:, 1]) & (p1[:, 1] <= h), p1


def fb_loop(cv2, seq, steps, init, cap, lk, mode, velocity=False):
    """One sequence through the capped loop -> per step (survivors, survivors within 0.5 px of the true translation,
    points LK tracked within 0.5 px of it).  mode: "reference" (same-direction pass, max error 30), "reverse" (the
    forward-backward check at FB_MAX_ERR; with velocity, the mirrored start) or "reverse-p1" (velocity starts, the reverse
    pass started at p1)."""
    pts = np.asarray(init, np.float32).reshape(-1, 2)
    prev = np.full_like(pts, np.nan)
    out = []
    for t in range(1, len(seq)):
        if mode == "reference":
            keep, p1 = same_direction_keep(cv2, lk, seq[t - 1], seq[t], pts)
        else:
            starts = velocity_starts(pts, prev) if velocity else None
            keep, p1, _d = fb_keep_from(cv2, lk, seq[t - 1], seq[t], pts, starts, mirror=mode == "reverse")
        on = abs(p1 - pts - np.float32(steps[t - 1])).max(-1) <= 0.5 if len(pts) else np.zeros(0, bool)
        out.append((int(keep.sum()), int((keep & on).sum()), int(on.sum())))
        surv = p1[keep]
        new = detect(cv2, seq[t], surv, cap)
        prev = np.concatenate([pts[keep], np.full_like(new, np.nan)])
        pts = np.concatenate([surv, new]).astype(np.float32)
    return out


def fast_case(cv2, px):
    h, w = KITTI
    seq = fine_sequence(cv2, h, w, FAST_MOTIONS[px], seed=5)
    return seq, cv2.goodFeaturesToTrack(seq[0], **DET).reshape(-1, 2)


# per step (survivors, survivors on the true motion, LK results on the true motion) of fb_loop on fast_case(cv2, px) with
# REF_LK and FB_CAP (cv2 4.13)
FAST_FB = {
    (16, "reference"): [(0, 0, 985), (0, 0, 991), (1, 1, 996), (0, 0, 994), (1, 1, 991)],
    (16, "reverse"): [(981, 980, 985), (1476, 1475, 1489), (1459, 1459, 1485), (1472, 1472, 1494), (1469, 1467, 1484)],
    (20, "reference"): [(0, 0, 984), (0, 0, 992), (1, 1, 988), (1, 0, 988), (1, 1, 988)],
    (20, "reverse"): [(977, 977, 984), (1463, 1463, 1485), (1457, 1456, 1476), (1464, 1461, 1481), (1464, 1463, 1478)],
}
# FAST_STEPS (test_motion_prior_cpu.py) with the velocity prior: survivors on the true motion per step, the reverse pass
# started at the mirrored start and at p1 (cv2 4.13); the first step has no velocity yet, so both agree there
FAST_FB_VELOCITY = {"reverse": [454, 442, 437, 430, 417, 408, 400], "reverse-p1": [454, 27, 26, 26, 24, 25, 25]}


@pytest.fixture(scope="module")
def cv2_mod():
    return pytest.importorskip("cv2")


def test_mirror_start_rounds_like_numpy_float32():
    p0 = np.array([[1e8, 3.0], [0.1, 7.25], [5.0, 5.0]], np.float32)
    p1 = np.array([[1e8 + 16.0, 2.0], [np.nan, 9.0], [-0.0, 4.0]], np.float32)
    s = np.array([[1e8 + 8.0, 3.5], [0.3, np.nan], [5.0, 6.0]], np.float32)
    b = mirror_start(p0, p1, s)
    assert b.dtype == np.float32
    assert np.array_equal(b[0], np.float32([1e8 + 8.0, 1.5])) and np.isnan(b[1]).all() and np.array_equal(b[2], [-0.0, 3.0])
    # rounded twice in float32, not once in double
    a, q, r = np.float32(0.1), np.float32(0.7), np.float32(0.3)
    assert mirror_start([[a, a]], [[q, q]], [[r, r]])[0, 0] == np.float32(q - np.float32(r - a))


def test_mirror_start_without_a_prior_is_p1_bit_for_bit():
    rng = np.random.default_rng(3)
    p0 = rng.uniform(-50, 1300, (64, 2)).astype(np.float32)
    p1 = (p0 + rng.uniform(-20, 20, (64, 2))).astype(np.float32)
    p1[3] = np.nan
    p1[5, 0] = -0.0
    p1[7, 1] = np.inf
    p1[9] = np.float32(np.frombuffer(np.uint32(0x7fc01234).tobytes(), np.float32)[0])   # a NaN with a payload
    b = mirror_start(p0, p1, p0)
    assert np.array_equal(b.view(np.uint32), p1.view(np.uint32))


@pytest.mark.parametrize("px", sorted(FAST_MOTIONS))
def test_reverse_check_keeps_fast_correct_tracks(cv2_mod, px):
    """16 and 20 px per frame, the library's parameters: the same-direction check keeps at most one track in the first step
    (a correct track has d = 2 x motion > 30), the reverse check at 1 px keeps at least 98 % of the tracks LK got right, in
    every step."""
    cv2 = cv2_mod
    seq, init = fast_case(cv2, px)
    got = {m: fb_loop(cv2, seq, FAST_MOTIONS[px], init, FB_CAP, REF_LK, m) for m in ("reference", "reverse")}
    for m in got:
        assert got[m] == FAST_FB[(px, m)], (px, m, got[m])
    assert got["reference"][0][0] <= 1
    for kept, kept_on, on in got["reverse"]:
        assert kept_on >= 0.98 * on, (px, got["reverse"])


def test_mirrored_start_follows_the_velocity_prior(cv2_mod):
    """FAST_STEPS with the velocity prior (maxLevel 0, 21 x 21 window, 12 px per frame): started at p1, the reverse pass
    cannot capture 12 px either and rejects correct tracks; from the mirrored start it keeps at least 15 times as many
    tracks on the true motion in every step after the first."""
    cv2 = cv2_mod
    h, w = KITTI
    seq = fine_sequence(cv2, h, w, FAST_STEPS, seed=5)
    init = cv2.goodFeaturesToTrack(seq[0], **DET).reshape(-1, 2)
    got = {m: [o for _n, o, _l in fb_loop(cv2, seq, FAST_STEPS, init, FB_CAP, FAST_LK, m, velocity=True)] for m in FAST_FB_VELOCITY}
    assert got == FAST_FB_VELOCITY, got
    for t in range(1, len(FAST_STEPS)):
        assert got["reverse"][t] >= 15 * got["reverse-p1"][t], got


def test_entry_points_reject_null_pointers(klt):
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    for name in ("klt_frame_step_batch_fb_async", "klt_track_fb_host"):
        assert hasattr(L, name) and name in _lib.SYMBOLS
    inval = _lib.KLT_ERR_INVALID_ARG
    lay = _lib.klt_pyr_layout()
    prm = _lib.klt_lk_params()
    args = [None, None, None, None, None, lay, 0, 0, 1, 1, None, None, 0, prm, 1.0, 10, 100, 0.03, 10.0, 31, None, 100, None,
            None, None, None, None, None, None, None, 0]
    # a null context (with and without start positions, control and the error output), a null flag word: rejected before
    # anything touches a device
    assert L.klt_frame_step_batch_fb_async(*args, None, None, None, None) == inval
    assert L.klt_frame_step_batch_fb_async(*args, 16, _lib.klt_step_control(), 16, None) == inval
    args[12] = 8
    args[28] = 16
    assert L.klt_frame_step_batch_fb_async(*args, None, None, None, None) == inval
    args[28] = None
    assert L.klt_frame_step_batch_fb_async(*args, 16, None, 16, None) == inval
    # klt_track_fb_host(ctx, prev, prev_pitch, next, next_pitch, w, h, pts, n, max_level, params, max_err, next_pts, status,
    # err, keep, bidir_err)
    img = np.zeros((8, 8), np.uint8)
    pts = np.zeros((4, 2), np.float32)
    outs = [np.zeros(n, t) for n, t in ((8, np.float32), (4, np.uint8), (4, np.float32), (4, np.uint8), (4, np.float32))]
    good = [None, img.ctypes.data, 8, img.ctypes.data, 8, 8, 8, pts.ctypes.data, 4, 0, prm, 1.0] + [o.ctypes.data for o in outs]
    for i, v in [(0, None), (15, None), (16, None), (5, 0), (6, -1), (8, -1), (9, -1)]:
        a = list(good)
        a[i] = v
        assert L.klt_track_fb_host(*a) == inval, (i, v)
    flagged = _lib.klt_lk_params(31, 31, 3, 30, 0.03, _lib.OPTFLOW_USE_INITIAL_FLOW, 1e-4)
    a = list(good)
    a[10] = flagged
    assert L.klt_track_fb_host(*a) == inval                          # no start positions in this entry point


@pytest.mark.parametrize("bad", ["forward", "REVERSE", None, 1])
def test_invalid_second_pass_raises_before_device_work(bad):
    from visual_odom_pipeline_b200 import lk as K
    from visual_odom_pipeline_b200 import tracker as T
    with pytest.raises(K.error):
        K.trackBidirectional(None, None, None, second_pass=bad)
    with pytest.raises(K.error):
        T.KLTSequenceBatch(None, None, None, 16, second_pass=bad)
    trk = T.KLTTracker()
    for call in (lambda: trk.track(None, None, True, second_pass=bad), lambda: trk.track_filtered(None, None, second_pass=bad),
                 lambda: trk.step(None, None, second_pass=bad), lambda: trk.step_batch(None, None, None, second_pass=bad)):
        with pytest.raises(K.error):
            call()
