"""CPU tier of the back-end control of KLTSequenceBatch (control=True): the per-sequence row choice of history() and
tracks_from_history on hand-built rings whose sequences are at different frames (after restarts), and the argument checks
of the two entry points that run before any device work."""
import numpy as np

from visual_odom_pipeline_b200.tracker import TrackHistory, history_from_ring, history_rows, tracks_from_history


def test_history_rows_equal_frames_is_the_plain_window():
    """With every sequence at the same frame (no restart), the rows are the last min(R, f + 1) frames, oldest first."""
    for R in (1, 3, 4):
        for f in range(0, 9):
            fr, rows = history_rows(np.full(3, f, np.int32), R)
            n = min(R, f + 1)
            want = np.arange(f - n + 1, f + 1)
            assert fr.dtype == np.int32 and fr.shape == (n, 3)
            assert np.array_equal(fr, np.tile(want[:, None], (1, 3)))
            assert np.array_equal(rows, np.tile((want % R)[:, None], (1, 3)))


def test_history_rows_per_sequence_frames():
    """T follows the sequence with the most frames; the others get their own last frames, negative before their frame 0."""
    fr, rows = history_rows(np.array([9, 1, 0, 2], np.int32), 4)
    assert np.array_equal(fr, [[6, -2, -3, -1], [7, -1, -2, 0], [8, 0, -1, 1], [9, 1, 0, 2]])
    assert np.array_equal(rows, [[2, 2, 1, 3], [3, 3, 2, 0], [0, 0, 3, 1], [1, 1, 0, 2]])
    fr, rows = history_rows(np.array([0, 1], np.int32), 5)
    assert np.array_equal(fr, [[-1, 0], [0, 1]]) and np.array_equal(rows, [[4, 0], [0, 1]])


def build_ring(R, width, per_seq):
    """per_seq: per sequence, {frame: [(id, x, y), ...]} of the frames its ring should hold now; every other row keeps
    stale entries of an older sequence (count 3, ids 900+), which history() must not hand over."""
    B = len(per_seq)
    counts = np.full((R, B), 3, np.int32)
    frames = np.full((R, B), 77, np.int32)
    pts = np.full((R, B, width, 2), 5.0, np.float32)
    ids = np.tile(900 + np.arange(width, dtype=np.int32), (R, B, 1))
    src = np.zeros((R, B, width), np.int32)
    for b, rows in enumerate(per_seq):
        for f in sorted(rows):
            r = f % R
            prev = [e[0] for e in rows.get(f - 1, [])]
            counts[r, b], frames[r, b] = len(rows[f]), f
            for j, (i, x, y) in enumerate(rows[f]):
                pts[r, b, j] = (x, y)
                ids[r, b, j] = i
                src[r, b, j] = prev.index(i) if i in prev else -1
    return TrackHistory(counts, frames, pts, ids, src)


def test_history_from_ring_after_restarts():
    """Ring of depth 4: sequence 0 at frame 9 (never restarted), sequence 1 restarted one frame ago, sequence 2 restarted
    at this frame, sequence 3 restarted five frames ago (its rows have wrapped since).  Each sequence's rows are
    its own; rows before a restart have count 0 and never reach tracks_from_history."""
    R, W = 4, 4
    per_seq = [
        {6: [(1, 1.0, 1.0)], 7: [(1, 1.5, 1.0), (2, 4.0, 4.0)], 8: [(2, 4.5, 4.0)], 9: [(2, 5.0, 4.0), (3, 0.5, 0.5)]},
        {0: [(40, 2.0, 2.0), (41, 3.0, 3.0)], 1: [(41, 3.5, 3.0)]},
        {0: [(7, 9.0, 9.0)]},
        {2: [(60, 1.0, 0.0)], 3: [(60, 1.25, 0.0)], 4: [(60, 1.5, 0.0), (61, 6.0, 6.0)], 5: [(61, 6.5, 6.0)]},
    ]
    ring = build_ring(R, W, per_seq)
    frames = np.array([9, 1, 0, 5], np.int32)
    hist = history_from_ring(ring, frames)
    assert hist.counts.shape == (4, 4) and hist.points.shape == (4, 4, W, 2) and hist.src.shape == (4, 4, W)
    assert np.array_equal(hist.frames, [[6, -2, -3, 2], [7, -1, -2, 3], [8, 0, -1, 4], [9, 1, 0, 5]])
    assert np.array_equal(hist.counts, [[1, 0, 0, 1], [2, 0, 0, 1], [1, 2, 0, 2], [2, 1, 1, 1]])
    assert np.array_equal(hist.src[3, 0, :2], [0, -1]) and np.array_equal(hist.src[2, 1, :2], [-1, -1])
    seqs = tracks_from_history(hist)
    for b, rows in enumerate(per_seq):
        want = {}
        for f in sorted(rows):
            for i, x, y in rows[f]:
                want.setdefault(i, ([], []))
                want[i][0].append(f)
                want[i][1].append((x, y))
        assert set(seqs[b]) == set(want), b
        for i, (fs, ps) in want.items():
            assert np.array_equal(seqs[b][i][0], np.asarray(fs, np.int32))
            assert np.array_equal(seqs[b][i][1], np.asarray(ps, np.float32))


def test_history_from_ring_without_restart_is_the_ring_window():
    """Every sequence at frame 5 of a ring of depth 3: the rows are frames 3, 4, 5 of the storage as they are."""
    rng = np.random.default_rng(1)
    R, B, W = 3, 2, 5
    ring = TrackHistory(rng.integers(0, W + 1, (R, B)).astype(np.int32), np.array([[3, 3], [4, 4], [5, 5]], np.int32),
                        rng.standard_normal((R, B, W, 2)).astype(np.float32), rng.integers(0, 99, (R, B, W)).astype(np.int32),
                        rng.integers(-1, W, (R, B, W)).astype(np.int32))
    hist = history_from_ring(ring, np.array([5, 5], np.int32))
    rows = [3 % R, 4 % R, 5 % R]
    for name, got, src in zip(hist._fields, hist, ring):
        assert np.array_equal(got, src[rows]), name


def test_entry_points_reject_null_pointers(klt):
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    for name in ("klt_frame_step_batch_control_async", "klt_track_records_step_control"):
        assert hasattr(L, name) and name in _lib.SYMBOLS
    ctl = _lib.klt_step_control()
    lay = _lib.klt_pyr_layout()
    prm = _lib.klt_lk_params()
    args = [None, None, None, None, None, lay, 0, 0, 1, 1, None, None, 0, prm, 30.0, 10, 100, 0.03, 10.0, 31, None, 100, None,
            None, None, None, None, None, None, None, 0]
    # a null control, and a null context with a control: rejected before anything touches a device
    assert L.klt_frame_step_batch_control_async(*args, None, None) == _lib.KLT_ERR_INVALID_ARG
    assert L.klt_frame_step_batch_control_async(*args, ctl, None) == _lib.KLT_ERR_INVALID_ARG
    assert L.klt_track_records_step_control(None, 1, 0, 4, None, None, None, None, None, None, None, None, None, 2, None, None, None,
                                            None, None, None, None, None, None, None) == _lib.KLT_ERR_INVALID_ARG
