"""CPU tier of the per-track records of KLTSequenceBatch: tracks_from_history on hand-built rings (no GPU), and the
symbols of the two entry points."""
import numpy as np

from visual_odom_pipeline_b200.tracker import TrackHistory, tracks_from_history


def ring(rows, frames, width=4):
    """rows: per frame (oldest first), per sequence, a list of (id, x, y) in slot order; src is derived from the ids."""
    T, B = len(rows), len(rows[0])
    counts = np.zeros((T, B), np.int32)
    fr = np.tile(np.asarray(frames, np.int32)[:, None], (1, B))
    pts = np.full((T, B, width, 2), 12345.0, np.float32)          # garbage behind the counts
    ids = np.full((T, B, width), -77, np.int32)
    src = np.full((T, B, width), -99, np.int32)
    for t in range(T):
        for b in range(B):
            counts[t, b] = len(rows[t][b])
            prev = [e[0] for e in rows[t - 1][b]] if t else []
            for j, (i, x, y) in enumerate(rows[t][b]):
                pts[t, b, j] = (x, y)
                ids[t, b, j] = i
                src[t, b, j] = prev.index(i) if i in prev else -1
    return TrackHistory(counts, fr, pts, ids, src)


def check(tracks, want):
    assert set(tracks) == set(want)
    for i, (f, p) in want.items():
        gf, gp = tracks[i]
        assert gf.dtype == np.int32 and gp.dtype == np.float32 and gp.shape == (len(f), 2)
        assert np.array_equal(gf, np.asarray(f, np.int32)), i
        assert np.array_equal(gp, np.asarray(p, np.float32).reshape(-1, 2)), i


def test_wrap_around_birth_death_and_empty_sequence():
    """Frames 5..8 of a ring of depth 4 whose storage has wrapped (history() hands them over oldest first): sequence 0
    has a track over the whole window, one that dies at frame 6, one born at frame 7 and a new id in a reused slot;
    sequence 1 is empty throughout; sequence 2 loses every track and gets new ones."""
    rows = [
        [[(3, 1.0, 2.0), (4, 5.0, 6.0)], [], [(10, 0.5, 0.5)]],                   # frame 5
        [[(3, 1.5, 2.5), (4, 5.5, 6.5)], [], [(10, 0.75, 0.5)]],                  # frame 6
        [[(3, 2.0, 3.0), (9, 7.0, 7.0)], [], []],                                 # frame 7: 4 died, 9 born; 10 died
        [[(3, 2.5, 3.5), (9, 7.5, 7.25), (11, 8.0, 1.0)], [], [(12, 4.0, 4.0)]],  # frame 8
    ]
    hist = ring(rows, [5, 6, 7, 8])
    seqs = tracks_from_history(hist)
    assert len(seqs) == 3
    check(seqs[0], {3: ([5, 6, 7, 8], [1.0, 2.0, 1.5, 2.5, 2.0, 3.0, 2.5, 3.5]), 4: ([5, 6], [5.0, 6.0, 5.5, 6.5]),
                    9: ([7, 8], [7.0, 7.0, 7.5, 7.25]), 11: ([8], [8.0, 1.0])})
    assert seqs[1] == {}
    check(seqs[2], {10: ([5, 6], [0.5, 0.5, 0.75, 0.5]), 12: ([8], [4.0, 4.0])})


def test_slots_move_and_bits_survive():
    """Survivors move to lower slots as tracks before them die; the positions come back bit for bit (a NaN payload and
    -0.0 included) and the ids need not be in slot order."""
    odd = np.array([0x7fc01234], np.uint32).view(np.float32)[0]
    rows = [
        [[(50, 1.0, 1.0), (7, odd, -0.0), (8, 3.0, 3.0)]],
        [[(7, -0.0, odd), (8, 3.25, 3.0)]],
        [[(8, 3.5, 3.0), (51, 9.0, 9.0)]],
    ]
    hist = ring(rows, [0, 1, 2])
    assert list(hist.src[1, 0, :2]) == [1, 2] and list(hist.src[2, 0, :2]) == [1, -1]
    tr = tracks_from_history(hist)[0]
    assert set(tr) == {50, 7, 8, 51}
    assert np.array_equal(tr[7][0], [0, 1])
    assert np.array_equal(tr[7][1].view(np.uint32), np.array([[odd, -0.0], [-0.0, odd]], np.float32).view(np.uint32))
    check({k: tr[k] for k in (50, 8, 51)}, {50: ([0], [1.0, 1.0]), 8: ([0, 1, 2], [3.0, 3.0, 3.25, 3.0, 3.5, 3.0]),
                                             51: ([2], [9.0, 9.0])})


def test_single_frame_and_negative_ids():
    """Right after construction history() holds frame 0 only; ids given by the caller may be negative."""
    hist = ring([[[(-5, 1.0, 2.0), (0, 3.0, 4.0)], []]], [0])
    seqs = tracks_from_history(hist)
    check(seqs[0], {-5: ([0], [1.0, 2.0]), 0: ([0], [3.0, 4.0])})
    assert seqs[1] == {}


def test_entry_points_exported(klt):
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    for name in ("klt_track_records_step", "klt_track_window"):
        assert hasattr(L, name) and name in _lib.SYMBOLS
    # a null context is rejected before anything touches a device
    assert L.klt_track_records_step(None, 1, 0, 4, None, None, None, None, None, None, None, None, None, 2, None, None, None, None,
                                    None, None) == _lib.KLT_ERR_INVALID_ARG
    assert L.klt_track_window(None, 1, 4, 2, None, None, None, None, 1, None, None) == _lib.KLT_ERR_INVALID_ARG
