"""GPU tier (pytest -m gpu, B200) of the per-track records of KLTSequenceBatch (history=R): first_points / first_frames /
lengths per slot, the observation ring, window(k) and history().

Bar: every frame and sequence, against records kept on the host per track id alongside the capped cv2 loop of
test_gpu_frame_step_async.py: first positions compared as uint32, first frames and lengths exactly, every window and
the ring's rows bit for bit (NaN where the track has no position).  The records change nothing of the step itself (a
history=0 twin gives the same points, ids, counts, keep and n_new), and graph replay equals eager steps bit for bit."""
import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from test_gpu_frame_step_async import DET, KITTI, LK, cv2_step, pad

pytestmark = pytest.mark.gpu

OUTSIDE = np.array([[-40.0, 12.0], [1241 + 25.5, 100.0], [300.0, 376 + 60.0], [-5.0, -7.0]], np.float32)


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def frames_at(seqs, t):
    import torch
    return torch.from_numpy(np.stack([s[t] for s in seqs])).cuda()


def make(seqs, init, cap, history, ids=None, first=None, prefilter=None):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init)
    kw = {}
    if ids is not None:
        kw["ids"] = torch.from_numpy(ids).cuda()
    if first is not None:
        kw["first_points"], kw["first_frames"] = (torch.from_numpy(a).cuda() for a in first)
    return T.KLTSequenceBatch(frames_at(seqs, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), cap,
                              history=history, prefilter=prefilter, **kw, **LK, **DET)


class Records:
    """Host-side per-id records of one sequence: position per frame, first frame and first position, plus the rows."""

    def __init__(self, pts, ids, first_pts=None, first_frames=None):
        self.pos = {int(i): {0: p} for i, p in zip(ids, pts)}
        self.first = {int(i): (0 if first_frames is None else int(first_frames[j]), pts[j] if first_pts is None else first_pts[j])
                      for j, i in enumerate(ids)}
        self.rows = {0: (np.asarray(ids, np.int32), pts.reshape(-1, 2), np.full(len(ids), -1, np.int32))}

    def step(self, t, ids, pts):
        prev = {int(i): j for j, i in enumerate(self.rows[t - 1][0])}
        src = np.array([prev.get(int(i), -1) for i in ids], np.int32)
        for i, p in zip(ids, pts):
            i = int(i)
            if i not in self.pos:
                self.pos[i], self.first[i] = {}, (t, p)
            self.pos[i][t] = p
        self.rows[t] = (np.asarray(ids, np.int32), pts.reshape(-1, 2), src)


def expected_window(recs, t, cap, k):
    out = np.full((len(recs), cap, k, 2), np.nan, np.float32)
    for b, r in enumerate(recs):
        for j, i in enumerate(r.rows[t][0]):
            for d in range(k):
                p = r.pos[int(i)].get(t - d)
                if p is not None:
                    out[b, j, k - 1 - d] = p
    return out


def check_records(sb, recs, t, cap, R):
    import torch
    tag = "frame %d" % t
    assert sb.frame == t
    fp, ff, ln = sb.first_points.cpu().numpy(), sb.first_frames.cpu().numpy(), sb.lengths.cpu().numpy()
    counts = sb.counts.cpu().numpy()
    for b, r in enumerate(recs):
        ids = r.rows[t][0]
        n = len(ids)
        assert int(counts[b]) == n, tag
        want_ff = np.array([r.first[int(i)][0] for i in ids], np.int32)
        want_fp = np.array([r.first[int(i)][1] for i in ids], np.float32).reshape(-1, 2)
        assert np.array_equal(ff[b, :n], want_ff), "%s sequence %d: first_frames" % (tag, b)
        assert np.array_equal(fp[b, :n].view(np.uint32), want_fp.view(np.uint32)), "%s sequence %d: first_points" % (tag, b)
        assert np.array_equal(ln[b, :n], t - want_ff + 1), "%s sequence %d: lengths" % (tag, b)
    for k in sorted({1, max(1, R // 2), R}):
        w = sb.window(k)
        assert w.shape == (len(recs), cap, k, 2) and w.dtype == torch.float32 and w.is_cuda
        assert np.array_equal(w.cpu().numpy().view(np.uint32), expected_window(recs, t, cap, k).view(np.uint32)), "%s: window(%d)" % (tag, k)
    hist = sb.history()
    n = min(R, t + 1)
    assert hist.counts.shape == (n, len(recs)) and np.array_equal(hist.frames, np.tile(np.arange(t - n + 1, t + 1)[:, None], (1, len(recs))))
    for row, f in enumerate(range(t - n + 1, t + 1)):
        for b, r in enumerate(recs):
            ids, pts, src = r.rows[f]
            c = len(ids)
            assert int(hist.counts[row, b]) == c, "%s: ring row of frame %d, sequence %d" % (tag, f, b)
            assert np.array_equal(hist.ids[row, b, :c], ids) and np.array_equal(hist.src[row, b, :c], src), "%s: ring frame %d" % (tag, f)
            assert np.array_equal(hist.points[row, b, :c].view(np.uint32), pts.view(np.uint32)), "%s: ring frame %d" % (tag, f)
    from visual_odom_pipeline_b200.tracker import tracks_from_history
    lo = t - n + 1
    for b, (got, r) in enumerate(zip(tracks_from_history(hist), recs)):
        want = {i: sorted(f for f in r.pos[i] if f >= lo) for i in r.pos}
        want = {i: fs for i, fs in want.items() if fs}
        assert set(got) == set(want), "%s sequence %d: tracks" % (tag, b)
        for i, fs in want.items():
            assert np.array_equal(got[i][0], fs)
            assert np.array_equal(got[i][1].view(np.uint32), np.array([r.pos[i][f] for f in fs], np.float32).view(np.uint32))


def snapshot(sb):
    return {k: getattr(sb, k).cpu().numpy() for k in ("points", "counts", "ids", "keep", "n_new")}


def test_records_against_cv2_loop(klt, cv2):
    """Five KITTI sequences (one empty, one with every point outside the image, three from goodFeaturesToTrack), C = 1500
    (binds on some frames), R = 4, eleven steps: the ring wraps twice.  Each step against the capped cv2 loop and
    host records; a history=0 twin steps alongside with the same outputs."""
    h, w = KITTI
    R, C, T = 4, 1500, 12
    seqs = [S.sequence(h, w, T, seed=130 + b) for b in range(5)]
    init = [np.zeros((0, 2), np.float32), OUTSIDE.copy()]
    for b in range(2, 5):
        init.append(cv2.goodFeaturesToTrack(seqs[b][0], **DET).reshape(-1, 2)[: 300 + 300 * b])
    sb = make(seqs, init, C, R)
    twin = make(seqs, init, C, 0)
    pts = [p.reshape(-1, 2) for p in init]
    ids = [np.arange(len(p), dtype=np.int32) for p in pts]
    next_id = [len(p) for p in pts]
    recs = [Records(p, i) for p, i in zip(pts, ids)]
    check_records(sb, recs, 0, C, R)
    bound = False
    for t in range(1, T):
        frames = frames_at(seqs, t)
        sb.step(frames)
        twin.step(frames)
        a, b_ = snapshot(sb), snapshot(twin)
        for key in a:
            assert np.array_equal(a[key].view(np.uint8), b_[key].view(np.uint8)), "frame %d: %s differs from history=0" % (t, key)
        sb.check()
        for b in range(len(seqs)):
            keep_ref, surv_ref, new_ref, _n, was_bound = cv2_step(cv2, seqs[b][t - 1], seqs[b][t], pts[b], DET, C)
            bound |= was_bound
            s, k = len(surv_ref), len(new_ref)
            assert int(a["counts"][b]) == s + k and np.array_equal(a["points"][b, :s].view(np.uint32), surv_ref.view(np.uint32))
            assert np.array_equal(a["points"][b, s:s + k], new_ref)
            ids[b] = np.concatenate([ids[b][keep_ref], np.arange(next_id[b], next_id[b] + k, dtype=np.int32)])
            next_id[b] += k
            pts[b] = np.concatenate([surv_ref, new_ref])
            recs[b].step(t, ids[b], pts[b])
        check_records(sb, recs, t, C, R)
    assert bound, "the cap never bound"


def test_first_points_given_at_construction(klt, cv2):
    """first_points / first_frames passed at construction, negative frames included (tracks older than the batch); R = 3
    and odd given ids.  The window never reaches before frame 0."""
    h, w = KITTI
    R, C, T = 3, 2500, 5
    seqs = [S.sequence(h, w, T, seed=200 + b) for b in range(3)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 150 + 200 * b] for b, s in enumerate(seqs)]
    padded, cnt = pad(init)
    rng = np.random.default_rng(4)
    given_ids = np.zeros(padded.shape[:2], np.int32)
    first_pts = rng.uniform(-50, 1300, padded.shape).astype(np.float32)
    first_frames = rng.integers(-40, 1, padded.shape[:2]).astype(np.int32)
    for b in range(3):
        given_ids[b, :cnt[b]] = 500 * (b + 1) + 3 * np.arange(cnt[b])
    sb = make(seqs, init, C, R, ids=given_ids, first=(first_pts, first_frames))
    pts = [p.reshape(-1, 2) for p in init]
    ids = [given_ids[b, :cnt[b]] for b in range(3)]
    next_id = [int(i.max()) + 1 for i in ids]
    recs = [Records(pts[b], ids[b], first_pts[b, :cnt[b]], first_frames[b, :cnt[b]]) for b in range(3)]
    check_records(sb, recs, 0, C, R)
    assert int(sb.lengths[0, :cnt[0]].min()) >= 1 and int(sb.first_frames.min()) < 0
    for t in range(1, T):
        sb.step(frames_at(seqs, t))
        out = snapshot(sb)
        for b in range(3):
            keep = out["keep"][b, :len(ids[b])]
            k = int(out["n_new"][b])
            ids[b] = np.concatenate([ids[b][keep], np.arange(next_id[b], next_id[b] + k, dtype=np.int32)])
            next_id[b] += k
            pts[b] = out["points"][b, :int(out["counts"][b])].copy()
            assert np.array_equal(out["ids"][b, :len(ids[b])], ids[b])
            recs[b].step(t, ids[b], pts[b])
        check_records(sb, recs, t, C, R)
    sb.check()


@pytest.mark.parametrize("B", [4, 6])
@pytest.mark.parametrize("prefilter", [None, (5, 1.5, 1.5)])
def test_graph_replay_equals_eager(klt, cv2, B, prefilter):
    """Nine frames with R = 4, both parities replayed from the graphs (which hold the records launch), against an eager
    twin, bit for bit: the step's outputs, first_points, first_frames, lengths, every window and history()."""
    h, w = KITTI
    R = 4
    seqs = [S.sequence(h, w, 10, seed=170 + b) for b in range(B)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 100 + 200 * b] for b, s in enumerate(seqs)]
    init[0] = init[0][:0]
    eager = make(seqs, init, 1800, R, prefilter=prefilter)
    graph = make(seqs, init, 1800, R, prefilter=prefilter)
    for t in range(1, 10):
        frames = frames_at(seqs, t)
        eager.step(frames)
        graph.step(frames)
        if t == 1:
            graph.capture()
        assert eager.frame == graph.frame == t
        for name in ("points", "counts", "ids", "keep", "n_new", "first_points", "first_frames", "lengths"):
            x, y = getattr(eager, name).cpu().numpy(), getattr(graph, name).cpu().numpy()
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "frame %d: %s" % (t, name)
        for k in (1, 2, 4):
            assert np.array_equal(eager.window(k).cpu().numpy().view(np.uint32), graph.window(k).cpu().numpy().view(np.uint32))
        for name, x, y in zip(eager.history()._fields, eager.history(), graph.history()):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "frame %d: history().%s" % (t, name)
        eager.check()
        graph.check()
    assert graph._graphs is not None


def test_errors(klt):
    import torch
    from visual_odom_pipeline_b200 import _lib
    from visual_odom_pipeline_b200 import tracker as T
    from visual_odom_pipeline_b200.lk import error
    h, w = 64, 96
    frames = torch.from_numpy(np.stack([S.sequence(h, w, 2, seed=90 + b)[1] for b in range(3)])).cuda()
    pts = torch.full((3, 8, 2), 20.0, device="cuda")
    cnt = torch.tensor([8, 0, 3], dtype=torch.int32, device="cuda")
    fp = pts.clone()
    ff = torch.zeros((3, 8), dtype=torch.int32, device="cuda")
    bad = [dict(history=-1), dict(history=2, first_points=fp), dict(history=2, first_frames=ff),
           dict(history=0, first_points=fp, first_frames=ff), dict(history=2, first_points=fp[:, :4], first_frames=ff),
           dict(history=2, first_points=fp.double(), first_frames=ff), dict(history=2, first_points=fp, first_frames=ff.long()),
           dict(history=2, first_points=fp.cpu(), first_frames=ff), dict(history=2, first_points=fp, first_frames=ff[:2])]
    for kw in bad:
        with pytest.raises(error):
            T.KLTSequenceBatch(frames, pts, cnt, 16, **kw)
    plain = T.KLTSequenceBatch(frames, pts, cnt, 16)
    for name in ("first_points", "first_frames", "lengths"):
        with pytest.raises(error):
            getattr(plain, name)
    with pytest.raises(error):
        plain.window(1)
    with pytest.raises(error):
        plain.history()
    sb = T.KLTSequenceBatch(frames, pts, cnt, 16, history=3, first_points=fp, first_frames=ff)
    for k in (0, 4, -1):
        with pytest.raises(error):
            sb.window(k)
    sb.step(frames)
    sb.check()
    assert sb.frame == 1 and sb.window(3).shape == (3, 16, 3, 2)

    # the entry points' own argument checks
    L = _lib.load()
    C, st = sb.capacity, torch.cuda.current_stream().cuda_stream
    cur, nxt = sb._cur, 1 - sb._cur
    good = [sb.ctx.handle, 3, C, C, sb._keep.data_ptr(), sb._pts[nxt].data_ptr(), sb._ids[nxt].data_ptr(), sb._counts[nxt].data_ptr(),
            sb._first_pts[cur].data_ptr(), sb._first_frames[cur].data_ptr(), sb._first_pts[nxt].data_ptr(),
            sb._first_frames[nxt].data_ptr(), sb._frame.data_ptr(), 3, sb._ring_pts.data_ptr(), sb._ring_ids.data_ptr(),
            sb._ring_src.data_ptr(), sb._ring_counts.data_ptr(), sb._ring_frames.data_ptr(), st]
    for i in [0, 4, 5, 6, 7, 8, 9, 10, 11, 12, 14, 15, 16, 17, 18]:
        args = list(good)
        args[i] = None
        assert L.klt_track_records_step(*args) == _lib.KLT_ERR_INVALID_ARG, "null argument %d" % i
    for i, v in [(13, 0), (13, -2), (3, C - 1), (2, -1), (1, 0)]:                # R < 1, out_stride < n_per_seq, n_per_seq < 0, n_seqs
        args = list(good)
        args[i] = v
        assert L.klt_track_records_step(*args) == _lib.KLT_ERR_INVALID_ARG, (i, v)
    out = torch.empty((3, C, 3, 2), dtype=torch.float32, device="cuda")
    wgood = [sb.ctx.handle, 3, C, 3, sb._ring_pts.data_ptr(), sb._ring_src.data_ptr(), sb._ring_counts.data_ptr(),
             sb._frame.data_ptr(), 3, out.data_ptr(), st]
    for i in [0, 4, 5, 6, 7, 9]:
        args = list(wgood)
        args[i] = None
        assert L.klt_track_window(*args) == _lib.KLT_ERR_INVALID_ARG, "null argument %d" % i
    for i, v in [(8, 0), (8, 4), (3, 0), (2, -1), (1, 0)]:                     # k outside [1, R], R < 1, width, n_seqs
        args = list(wgood)
        args[i] = v
        assert L.klt_track_window(*args) == _lib.KLT_ERR_INVALID_ARG, (i, v)
    # nothing was launched by the rejected calls: the state is that of one step
    torch.cuda.synchronize()
    assert sb.frame == 1 and bool((sb._frame == 1).all())
    sb.step(frames)
    sb.check()
    assert bool((sb._frame == 2).all())
