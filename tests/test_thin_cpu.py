"""CPU tier of the minimum track distance of KLTSequenceBatch (min_track_distance=d): the host reference the GPU tier
compares against (a plain slot-order loop in numpy float64), its properties on random and crafted sets, the capped cv2
loop's counts on a contracting sequence with and without thinning, and the argument checks of the new entry point and
of the Python option that run before any device work."""
import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from test_fb_check_cpu import REF_LK, same_direction_keep
from test_motion_prior_cpu import DET, KITTI, detect

# the synthetic sequence's default warp with scale 0.99 per frame instead of 1.003: the image contracts, tracks converge
SHRINK = (1.1, -0.6, 0.15, 0.99)
THIN_D = 10.0
THIN_CAP = 4096


def thin(p1, keep, d):
    """Slots thinned at distance d: the candidates (keep) in slot order; slot j is thinned when an earlier candidate that
    was not thinned has dx * dx + dy * dy < d * d, dx = double(x_j) - double(x_i), in numpy float64 (each subtraction,
    product and sum rounded once) -> (n,) bool."""
    p = np.asarray(p1, np.float32).reshape(-1, 2).astype(np.float64)
    dd = np.float64(d) * np.float64(d)
    out = np.zeros(len(p), bool)
    kx, ky = [], []
    for j in np.flatnonzero(np.asarray(keep, bool)):
        if kx:
            dx = p[j, 0] - np.asarray(kx)
            dy = p[j, 1] - np.asarray(ky)
            if ((dx * dx + dy * dy) < dd).any():
                out[j] = True
                continue
        kx.append(p[j, 0])
        ky.append(p[j, 1])
    return out


def close(a, b, d):
    dx = np.float64(a[0]) - np.float64(b[0])
    dy = np.float64(a[1]) - np.float64(b[1])
    return dx * dx + dy * dy < np.float64(d) * np.float64(d)


def shrink_case(cv2, frames=13, seed=7, n=2000):
    seq = S.sequence(*KITTI, frames, seed=seed, motion=SHRINK)
    return seq, cv2.goodFeaturesToTrack(seq[0], **dict(DET, maxCorners=n)).reshape(-1, 2)


def thin_loop(cv2, seq, init, cap, d):
    """One sequence through the capped loop with the reference's check and thinning at d (None: off) -> per step
    (survivors, thinned, new corners)."""
    pts = np.asarray(init, np.float32).reshape(-1, 2)
    out = []
    for t in range(1, len(seq)):
        keep, p1 = same_direction_keep(cv2, REF_LK, seq[t - 1], seq[t], pts)
        th = thin(p1, keep, d) if d is not None else np.zeros(len(pts), bool)
        keep = keep & ~th
        surv = p1[keep]
        new = detect(cv2, seq[t], surv, cap)
        out.append((int(keep.sum()), int(th.sum()), len(new)))
        pts = np.concatenate([surv, new]).astype(np.float32)
    return out


# per step (survivors, thinned, new corners) of thin_loop on shrink_case(cv2), C = 4096 (cv2 4.13)
SHRINK_COUNTS = {
    None: [(2000, 0, 340), (2340, 0, 89), (2429, 0, 75), (2504, 0, 70), (2574, 0, 79), (2653, 0, 71), (2724, 0, 62),
           (2786, 0, 68), (2854, 0, 57), (2911, 0, 62), (2972, 0, 51), (3022, 0, 60)],
    THIN_D: [(1798, 202, 467), (2160, 105, 178), (2213, 125, 163), (2258, 118, 148), (2316, 90, 141), (2363, 94, 132),
             (2397, 98, 149), (2427, 119, 135), (2420, 142, 152), (2422, 150, 166), (2437, 150, 131), (2444, 123, 132)],
}


@pytest.fixture(scope="module")
def cv2_mod():
    return pytest.importorskip("cv2")


@pytest.mark.parametrize("seed", range(6))
def test_reference_spacing_on_random_sets(seed):
    """No two kept candidates closer than d; every thinned slot has an earlier kept slot closer than d; only candidates
    are thinned; and the result depends on the slot order."""
    rng = np.random.default_rng(seed)
    n = 400
    p = rng.uniform(0, 120, (n, 2)).astype(np.float32)
    p[rng.integers(0, n, 40)] = p[rng.integers(0, n, 40)]          # exact duplicates
    keep = rng.random(n) < 0.8
    d = [10.0, 3.5, 0.5, 25.0, 1e-3, 7.25][seed]
    th = thin(p, keep, d)
    assert not (th & ~keep).any()
    kept = np.flatnonzero(keep & ~th)
    for a in range(len(kept)):
        for b in range(a + 1, len(kept)):
            assert not close(p[kept[a]], p[kept[b]], d), (kept[a], kept[b])
    for j in np.flatnonzero(th):
        assert any(close(p[j], p[i], d) for i in kept if i < j), j
    if seed < 4:
        assert th.any()
        rev = thin(p[::-1], keep[::-1], d)[::-1]
        assert not np.array_equal(rev, th)


def test_distance_exactly_d_is_kept_one_ulp_below_is_thinned():
    below = np.nextafter(np.float32(10.0), np.float32(0.0))
    assert thin([[0.0, 0.0], [10.0, 0.0]], [True, True], 10.0).tolist() == [False, False]
    assert thin([[0.0, 0.0], [below, 0.0]], [True, True], 10.0).tolist() == [False, True]
    assert thin([[0.0, 0.0], [3.0, 4.0]], [True, True], 5.0).tolist() == [False, False]          # 9 + 16 == 25
    below4 = np.nextafter(np.float32(4.0), np.float32(0.0))
    assert thin([[0.0, 0.0], [3.0, below4]], [True, True], 5.0).tolist() == [False, True]
    # an exact duplicate at the smallest distance, a thinned slot does not thin a later one, a non-candidate does not count
    assert thin([[5.0, 5.0], [5.0, 5.0]], [True, True], 1e-30).tolist() == [False, True]
    assert thin([[0.0, 0.0], [6.0, 0.0], [12.0, 0.0]], [True, True, True], 10.0).tolist() == [False, True, False]
    assert thin([[0.0, 0.0], [6.0, 0.0]], [False, True], 10.0).tolist() == [False, False]
    # d * d is rounded once in float64: below that square the pair is thinned, at it not
    d = 0.1
    x = np.float32(0.1)
    want = np.float64(x) * np.float64(x) < d * d
    assert thin([[0.0, 0.0], [x, 0.0]], [True, True], d).tolist() == [False, bool(want)]


def test_capped_loop_counts_on_contracting_sequence(cv2_mod):
    """Scale 0.99 per frame, 2000 initial corners, C = 4096: without thinning nothing is thinned and the row grows by the
    new corners; at 10 px about a hundred survivors a step are thinned, the row stays smaller and detection finds more."""
    cv2 = cv2_mod
    seq, init = shrink_case(cv2)
    got = {d: thin_loop(cv2, seq, init, THIN_CAP, d) for d in SHRINK_COUNTS}
    for d, want in SHRINK_COUNTS.items():
        assert got[d] == want, (d, got[d])
    assert sum(t for _s, t, _n in got[THIN_D]) >= 1000
    assert got[THIN_D][-1][0] + got[THIN_D][-1][2] < got[None][-1][0] + got[None][-1][2]


def test_entry_point_rejects_null_pointers_and_bad_distances(klt):
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    name = "klt_frame_step_batch_thin_async"
    assert hasattr(L, name) and name in _lib.SYMBOLS
    inval, unsup = _lib.KLT_ERR_INVALID_ARG, _lib.KLT_ERR_UNSUPPORTED
    lay = _lib.klt_pyr_layout()
    prm = _lib.klt_lk_params()
    args = [None, None, None, None, None, lay, 0, 0, 1, 1, None, None, 0, prm, 30.0, 10, 100, 0.03, 10.0, 31, None, 100, None,
            None, None, None, None, None, None, None, 0]
    # a null context, with and without start positions, control, the error and the thinned outputs, either direction
    assert L.klt_frame_step_batch_thin_async(*args, None, None, None, 0, 10.0, None, None) == inval
    assert L.klt_frame_step_batch_thin_async(*args, 16, _lib.klt_step_control(), 16, 1, 10.0, 16, None) == inval
    assert L.klt_frame_step_batch_thin_async(*args, None, None, None, 0, 131072.0, None, None) == inval
    # the distance is checked first: NaN, infinite, zero or negative is invalid, above the header's limit unsupported
    for d in (float("nan"), float("inf"), -float("inf"), 0.0, -0.0, -1.0):
        assert L.klt_frame_step_batch_thin_async(*args, None, None, None, 0, d, None, None) == inval, d
    for d in (131072.5, 1e300):
        assert L.klt_frame_step_batch_thin_async(*args, None, None, None, 0, d, None, None) == unsup, d
    # a null flag word and a reverse flag outside {0, 1}
    assert L.klt_frame_step_batch_thin_async(*args, None, None, None, 2, 10.0, None, None) == inval
    args[28] = 16
    assert L.klt_frame_step_batch_thin_async(*args, None, None, None, -1, 10.0, None, None) == inval


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), -float("inf"), 0, 0.0, -3.0, 131073.0, "10", True, [10.0], object()])
def test_invalid_min_track_distance_raises_before_device_work(bad):
    from visual_odom_pipeline_b200 import lk as K
    from visual_odom_pipeline_b200 import tracker as T
    with pytest.raises(K.error):
        T.KLTSequenceBatch(None, None, None, 16, min_track_distance=bad)


def test_valid_min_track_distance_values():
    from visual_odom_pipeline_b200 import tracker as T
    assert T.check_min_track_distance(None) is None
    assert T.check_min_track_distance(10) == 10.0 and isinstance(T.check_min_track_distance(10), float)
    assert T.check_min_track_distance(np.float32(0.5)) == 0.5
    assert T.check_min_track_distance(131072) == 131072.0
    assert T.check_min_track_distance(5e-324) == 5e-324
