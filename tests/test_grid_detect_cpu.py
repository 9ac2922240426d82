"""CPU tier of grid detection in the batched frame step (KLTSequenceBatch(detect_grid=(cols, rows), tracks_per_cell=q)):
the host reference of the rule the GPU tier compares against (cells, tracks per cell, quotas, one cv2.goodFeaturesToTrack
call per cell, the interleave and the cap), the cv2 facts it rests on, the point-to-cell cases, pinned counts of the
capped cv2 loop on a sequence with a low-contrast left third, and the argument checks that run without a device."""
import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from test_fb_check_cpu import REF_LK, same_direction_keep
from test_motion_prior_cpu import DET, KITTI, detect


def edges(n, length):
    """X_i = floor(i * length / n), i = 0 .. n, in integer arithmetic."""
    return [i * length // n for i in range(n + 1)]


def cells_of(pts, shape, grid):
    """(n, 2) float32 points -> (n,) cell index j * cols + i, -1 for NaN: column max{i : X_i <= x} clamped to [0, cols - 1],
    rows alike."""
    h, w = shape
    cols, rows = grid
    p = np.asarray(pts, np.float32).reshape(-1, 2)
    xs = np.asarray(edges(cols, w)[:-1], np.float64)
    ys = np.asarray(edges(rows, h)[:-1], np.float64)
    i = np.clip(np.searchsorted(xs, p[:, 0].astype(np.float64), side="right") - 1, 0, cols - 1)
    j = np.clip(np.searchsorted(ys, p[:, 1].astype(np.float64), side="right") - 1, 0, rows - 1)
    return np.where(np.isnan(p).any(1), -1, j * cols + i)


def step_mask(im, surv, radius=10):
    """The step's detection mask: 255 with a filled disc around np.int32 of every finite point."""
    mask = np.full_like(im, 255)
    for x, y in np.asarray(surv, np.float32).reshape(-1, 2):
        if np.isfinite(x) and np.isfinite(y) and abs(x) < 1e9 and abs(y) < 1e9:
            import cv2
            cv2.circle(mask, (int(np.int32(x)), int(np.int32(y))), radius, 0, -1)
    return mask


def cell_lists(cv2, im, mask, grid, quotas, det=DET):
    """Per cell k: cv2.goodFeaturesToTrack(im, maxCorners=quotas[k], mask=mask & R_k) as (m, 2) float32, empty for 0."""
    h, w = im.shape
    cols, rows = grid
    X, Y = edges(cols, w), edges(rows, h)
    out = []
    for j in range(rows):
        for i in range(cols):
            n = int(quotas[j * cols + i])
            c = None
            if n > 0:
                mk = np.zeros_like(mask)
                mk[Y[j]:Y[j + 1], X[i]:X[i + 1]] = mask[Y[j]:Y[j + 1], X[i]:X[i + 1]]
                c = cv2.goodFeaturesToTrack(im, mask=mk, **dict(det, maxCorners=n))
            out.append(np.zeros((0, 2), np.float32) if c is None else c.reshape(-1, 2))
    return out


def interleave(lists, cut):
    """L_0[0], L_1[0], ..., L_0[1], ... (exhausted lists skipped), the first `cut` of them."""
    out = []
    for r in range(max([len(L) for L in lists] + [0])):
        out.extend(L[r] for L in lists if len(L) > r)
    return np.asarray(out[:max(cut, 0)], np.float32).reshape(-1, 2)


def grid_detect(cv2, im, surv, cap, grid, q, radius=10, det=DET, lists=False):
    """The detection half of the step with grid detection: the new corners in row order (and the per-cell lists)."""
    surv = np.asarray(surv, np.float32).reshape(-1, 2)
    cols, rows = grid
    cell = cells_of(surv, im.shape, grid)
    s = np.bincount(cell[cell >= 0], minlength=cols * rows)
    L = cell_lists(cv2, im, step_mask(im, surv, radius), grid, np.maximum(0, q - s), det)
    new = interleave(L, min(det["maxCorners"], cap - len(surv)))
    return (new, L) if lists else new


@pytest.fixture(scope="module")
def cv2_mod():
    return pytest.importorskip("cv2")


def test_cell_edges_and_point_to_cell():
    assert edges(3, 10) == [0, 3, 6, 10] and edges(7, 1241)[-1] == 1241
    h, w = 10, 10
    pts = np.float32([[0, 0], [2.99, 0], [3, 0], [5.999, 9.5], [6, 0], [9.99, 0], [10, 10], [-0.5, -3], [1e30, 5],
                      [-np.inf, np.inf], [np.nan, 1], [1, np.nan], [np.nextafter(np.float32(3), np.float32(0)), 0]])
    got = cells_of(pts, (h, w), (3, 2)).tolist()
    assert got == [0, 0, 1, 4, 2, 2, 5, 0, 5, 3, -1, -1, 0]
    # W % cols != 0: every pixel in exactly one cell, widths differ by at most 1
    X = edges(7, 1241)
    widths = np.diff(X)
    assert widths.sum() == 1241 and widths.max() - widths.min() <= 1
    xs = np.arange(1241, dtype=np.float32)
    cols = cells_of(np.stack([xs, np.zeros_like(xs)], 1), (1, 1241), (7, 1))
    assert all(X[c] <= x < X[c + 1] for x, c in zip(range(1241), cols))


def test_interleave_and_cut():
    L = [np.float32([[0, 0], [0, 1], [0, 2]]), np.zeros((0, 2), np.float32), np.float32([[2, 0]]), np.float32([[3, 0], [3, 1]])]
    assert interleave(L, 100).tolist() == [[0, 0], [2, 0], [3, 0], [0, 1], [3, 1], [0, 2]]
    assert interleave(L, 4).tolist() == [[0, 0], [2, 0], [3, 0], [0, 1]]
    assert interleave(L, 0).shape == (0, 2)


def test_cv2_facts(cv2_mod):
    """The masked maximum sets the threshold; maxCorners=0 means no limit; the result is prefix-stable in maxCorners."""
    cv2 = cv2_mod
    im = S.uneven_sequence(120, 200, 1, seed=5, left_gain=0.1)[0]
    kw = dict(qualityLevel=0.03, minDistance=10, blockSize=31)
    left = np.zeros_like(im)
    left[:, :60] = 255
    a = cv2.goodFeaturesToTrack(im, 0, mask=left, **kw)
    b = cv2.goodFeaturesToTrack(im, 0, **kw)
    assert a is not None and len(a) > 0                   # the masked maximum of the dim part: it keeps its corners
    assert b is None or (b.reshape(-1, 2)[:, 0] < 60).sum() < len(a)
    full = cv2.goodFeaturesToTrack(im, 0, **kw).reshape(-1, 2)
    assert len(full) > 40
    for n in (1, 5, 17, len(full) - 1, len(full), len(full) + 9):
        assert np.array_equal(cv2.goodFeaturesToTrack(im, n, **kw).reshape(-1, 2), full[:n]), n


def test_identity_grid_is_the_global_rule(cv2_mod):
    """detect_grid=(1, 1) with q = C gives detect() exactly, with survivors and with the capacity binding."""
    cv2 = cv2_mod
    seq = S.sequence(*KITTI, 2, seed=31)
    surv = cv2.goodFeaturesToTrack(seq[0], **dict(DET, maxCorners=600)).reshape(-1, 2)
    for cap in (4096, 1000, 650):
        got = grid_detect(cv2, seq[1], surv, cap, (1, 1), cap)
        assert np.array_equal(got, detect(cv2, seq[1], surv, cap)), cap


# per left-third gain: (corners of the global rule in the left third, fewest corners in a cell of the 8 x 4 grid at
# q = 32) on frame 0 of S.uneven_sequence(376, 1241, seed=100), no survivors (cv2 4.13)
UNEVEN_COUNTS = {1.0: (319, 32), 0.3: (0, 32), 0.1: (0, 18)}


@pytest.mark.parametrize("gain", sorted(UNEVEN_COUNTS))
def test_uneven_contrast_counts(cv2_mod, gain):
    cv2 = cv2_mod
    im = S.uneven_sequence(*KITTI, 1, seed=100, left_gain=gain)[0]
    glob = detect(cv2, im, np.zeros((0, 2), np.float32), 4096)
    new, L = grid_detect(cv2, im, np.zeros((0, 2), np.float32), 4096, (8, 4), 32, lists=True)
    got = (int((glob[:, 0] < KITTI[1] // 3).sum()), min(len(x) for x in L))
    assert got == UNEVEN_COUNTS[gain], got
    assert len(new) == min(1000, sum(len(x) for x in L))


def grid_loop(cv2, seq, init, cap, grid, q):
    """The capped loop with the reference's check and grid detection (grid None: the global rule) -> per step
    (survivors, new corners, cells of an 8 x 4 grid holding at least q / 2 points)."""
    pts = np.asarray(init, np.float32).reshape(-1, 2)
    out = []
    for t in range(1, len(seq)):
        keep, p1 = same_direction_keep(cv2, REF_LK, seq[t - 1], seq[t], pts)
        surv = p1[keep]
        new = detect(cv2, seq[t], surv, cap) if grid is None else grid_detect(cv2, seq[t], surv, cap, grid, q)
        pts = np.concatenate([surv, new]).astype(np.float32)
        c = cells_of(pts, seq[t].shape, (8, 4))
        out.append((int(keep.sum()), len(new), int((np.bincount(c[c >= 0], minlength=32) >= 32).sum())))
    return out


# per step (survivors, new corners, cells of 8 x 4 with >= 32 points) of grid_loop on S.uneven_sequence(376, 1241, 4,
# seed=100, left_gain=0.1) from 400 corners of its frame 0, C = 4096 (cv2 4.13)
UNEVEN_LOOP = {None: [(400, 1000, 20), (1394, 133, 20), (1506, 41, 20)],
               (8, 4): [(400, 1000, 28), (1397, 485, 28), (1862, 29, 28)]}


def test_capped_loop_counts_on_uneven_contrast(cv2_mod):
    """With the global rule a third of the cells stays below q / 2 = 32 points; with the grid (q = 64, so the 1000-corner cap
    binds at the first step) only the cells whose own cv2 call has fewer corners do."""
    cv2 = cv2_mod
    seq = S.uneven_sequence(*KITTI, 4, seed=100, left_gain=0.1)
    init = cv2.goodFeaturesToTrack(seq[0], **dict(DET, maxCorners=400)).reshape(-1, 2)
    got = {g: grid_loop(cv2, seq, init, 4096, g, 64) for g in UNEVEN_LOOP}
    for g, want in UNEVEN_LOOP.items():
        assert got[g] == want, (g, got[g])
    assert got[(8, 4)][-1][2] > got[None][-1][2]


def test_entry_points_reject_bad_arguments(klt):
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    for name in ("klt_frame_step_batch_grid_async", "klt_frame_step_grid_ws_bytes", "klt_good_features_to_track_grid",
                 "klt_good_features_to_track_grid_ws_bytes"):
        assert hasattr(L, name) and name in _lib.SYMBOLS
    inval, unsup = _lib.KLT_ERR_INVALID_ARG, _lib.KLT_ERR_UNSUPPORTED
    lay = _lib.klt_pyr_layout()
    prm = _lib.klt_lk_params()
    args = [None, None, None, None, None, lay, 0, 0, 1, 1, None, None, 0, prm, 30.0, 10, 100, 0.03, 10.0, 31, None, 100, None,
            None, None, None, None, None, 16, None, 0, None, None, None, 0]
    f = L.klt_frame_step_batch_grid_async
    assert f(*args, 0.0, None, 8, 4, 64, None) == inval                # null context
    for d in (float("nan"), float("inf"), -1.0):
        assert f(*args, d, None, 8, 4, 64, None) == inval, d
    assert f(*args, 1e300, None, 8, 4, 64, None) == unsup
    for c, r, q in ((0, 4, 64), (8, 0, 64), (8, 4, 0), (-1, 4, 64)):
        assert f(*args, 0.0, None, c, r, q, None) == inval, (c, r, q)
    assert f(*args, 0.0, None, 33, 32, 64, None) == unsup
    args[-1] = 2
    assert f(*args, 0.0, None, 8, 4, 64, None) == inval                # reverse outside {0, 1}
    assert L.klt_frame_step_grid_ws_bytes(1241, 376, 2, 100, 33, 32) == 0
    assert L.klt_frame_step_grid_ws_bytes(1241, 376, 2, 100, 8, 4) > L.klt_frame_step_ws_bytes(1241, 376, 2, 100)
    g = L.klt_good_features_to_track_grid
    assert g(None, None, 64, 48, 64, 0, 1, 2, 2, 8, 0.03, 10.0, 3, None, 0, 0, None, None, None, 0, None) == inval
    assert L.klt_good_features_to_track_grid_ws_bytes(64, 48, 1, 0, 2) == 0


@pytest.mark.parametrize("grid,q", [((8, 4), None), (None, 64), ((0, 4), 64), ((8, 0), 64), ((8, 4), 0), ((8, 4), -1),
                                    ((33, 32), 64), ((8.0, 4), 64), ((8, 4), 2.5), ((8, 4), True), ((True, 4), 64), (8, 64),
                                    ((8, 4, 1), 64), ("84", 64)])
def test_invalid_grid_raises_before_device_work(grid, q):
    from visual_odom_pipeline_b200 import lk as K
    from visual_odom_pipeline_b200 import tracker as T
    with pytest.raises(K.error):
        T.KLTSequenceBatch(None, None, None, 16, detect_grid=grid, tracks_per_cell=q)


def test_valid_grid_values():
    from visual_odom_pipeline_b200 import tracker as T
    assert T.check_detect_grid(None, None) is None
    assert T.check_detect_grid((8, 4), 64) == ((8, 4), 64)
    assert T.check_detect_grid([np.int64(32), 32], np.int32(1)) == ((32, 32), 1)
