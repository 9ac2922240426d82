"""GPU tier (pytest -m gpu, B200) of the back-end control of KLTSequenceBatch (control=True): drop(mask) ends chosen tracks
at the next step, restart(seqs, ...) starts chosen sequences over at the next step, on the device and in the graphs.

Bar: every sequence and frame against the capped cv2 loop of test_gpu_frame_step_async.py, with keep_ref & ~drop for the
drops and the staged points as the survivors of a restart, ids kept on the host, and the per-track records of
test_gpu_track_history.py (first positions, first frames, lengths, windows, history rows and tracks) bit for bit, each
sequence at its own frame.  An idle control=True object equals control=False, and graph replay equals eager steps."""
import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from test_gpu_frame_step_async import DET, KITTI, LK, cv2_step, pad
from test_gpu_track_history import OUTSIDE, Records, frames_at

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def make(seqs, init, cap, history, control=True, prefilter=None):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init)
    return T.KLTSequenceBatch(frames_at(seqs, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), cap,
                              history=history, prefilter=prefilter, control=control, **LK, **DET)


def lk_keep(cv2, im0, im1, pts, max_bidir=30):
    """The first half of cv2_step: keep (n,) bool and the tracked points (n, 2)."""
    h, w = im1.shape
    if not len(pts):
        return np.zeros(0, bool), np.zeros((0, 2), np.float32)
    p0 = pts.reshape(-1, 1, 2)
    p1, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **LK)
    p0r, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **LK)
    good = abs(p0 - p0r).reshape(-1, 2).max(-1) < max_bidir
    p1 = p1.reshape(-1, 2)
    return good & (0 <= p1[:, 0]) & (p1[:, 0] <= w) & (0 <= p1[:, 1]) & (p1[:, 1] <= h), p1


def detect(cv2, im1, surv, cap, radius=10):
    """The second half of cv2_step: the capped corners cv2 finds around the survivors (k, 2)."""
    mask = np.full_like(im1, 255)
    for x, y in [np.int32(p) for p in surv]:
        cv2.circle(mask, (int(x), int(y)), radius, 0, -1)
    k = min(DET["maxCorners"], cap - len(surv))
    if k <= 0:
        return np.zeros((0, 2), np.float32)
    c = cv2.goodFeaturesToTrack(im1, mask=mask, **dict(DET, maxCorners=k))
    return np.zeros((0, 2), np.float32) if c is None else c.reshape(-1, 2)


class Model:
    """Host state of one sequence: points, ids, id counter, own frame index and Records (keyed by that frame)."""

    def __init__(self, pts):
        self.pts = pts.reshape(-1, 2)
        self.ids = np.arange(len(self.pts), dtype=np.int32)
        self.next_id = len(self.pts)
        self.f = 0
        self.recs = Records(self.pts, self.ids)


def expected_window(models, cap, k):
    out = np.full((len(models), cap, k, 2), np.nan, np.float32)
    for b, m in enumerate(models):
        for j, i in enumerate(m.recs.rows[m.f][0]):
            for d in range(k):
                p = m.recs.pos[int(i)].get(m.f - d)
                if p is not None:
                    out[b, j, k - 1 - d] = p
    return out


def check_state(sb, models, cap, R, tag):
    """Counts, points, ids and every record of every sequence at its own frame."""
    import torch
    from visual_odom_pipeline_b200.tracker import tracks_from_history
    B = len(models)
    got = {k: getattr(sb, k).cpu().numpy() for k in ("points", "counts", "ids", "first_points", "first_frames", "lengths", "frames")}
    for b, m in enumerate(models):
        n = len(m.ids)
        assert int(got["counts"][b]) == n, "%s sequence %d: count" % (tag, b)
        assert np.array_equal(got["points"][b, :n].view(np.uint32), m.pts.view(np.uint32)), "%s sequence %d: points" % (tag, b)
        assert np.array_equal(got["ids"][b, :n], m.ids), "%s sequence %d: ids" % (tag, b)
        assert int(got["frames"][b]) == m.f, "%s sequence %d: frame" % (tag, b)
        ids = m.recs.rows[m.f][0]
        want_ff = np.array([m.recs.first[int(i)][0] for i in ids], np.int32)
        want_fp = np.array([m.recs.first[int(i)][1] for i in ids], np.float32).reshape(-1, 2)
        assert np.array_equal(got["first_frames"][b, :n], want_ff), "%s sequence %d: first_frames" % (tag, b)
        assert np.array_equal(got["first_points"][b, :n].view(np.uint32), want_fp.view(np.uint32)), "%s sequence %d: first_points" % (tag, b)
        assert np.array_equal(got["lengths"][b, :n], m.f - want_ff + 1), "%s sequence %d: lengths" % (tag, b)
    for k in sorted({1, max(1, R // 2), R}):
        w = sb.window(k)
        assert w.shape == (B, cap, k, 2) and w.dtype == torch.float32
        assert np.array_equal(w.cpu().numpy().view(np.uint32), expected_window(models, cap, k).view(np.uint32)), "%s: window(%d)" % (tag, k)
    hist = sb.history()
    T_ = min(R, max(m.f for m in models) + 1)
    assert hist.counts.shape == (T_, B)
    for b, m in enumerate(models):
        for row in range(T_):
            f = m.f - T_ + 1 + row
            assert int(hist.frames[row, b]) == f, "%s: history frames" % tag
            if f < 0:
                assert int(hist.counts[row, b]) == 0, "%s: history row of frame %d, sequence %d" % (tag, f, b)
                continue
            ids, pts, src = m.recs.rows[f]
            c = len(ids)
            assert int(hist.counts[row, b]) == c, "%s: history row of frame %d, sequence %d" % (tag, f, b)
            assert np.array_equal(hist.ids[row, b, :c], ids) and np.array_equal(hist.src[row, b, :c], src), "%s: ring frame %d" % (tag, f)
            assert np.array_equal(hist.points[row, b, :c].view(np.uint32), pts.view(np.uint32)), "%s: ring frame %d" % (tag, f)
    for b, (tracks, m) in enumerate(zip(tracks_from_history(hist), models)):
        lo = m.f - T_ + 1
        want = {i: sorted(f for f in m.recs.pos[i] if f >= lo) for i in m.recs.pos}
        want = {i: fs for i, fs in want.items() if fs}
        assert set(tracks) == set(want), "%s sequence %d: tracks" % (tag, b)
        for i, fs in want.items():
            assert np.array_equal(tracks[i][0], fs)
            assert np.array_equal(tracks[i][1].view(np.uint32), np.array([m.recs.pos[i][f] for f in fs], np.float32).view(np.uint32))


def test_drops_and_restarts_against_cv2_loop(klt, cv2):
    """Five KITTI sequences (one empty, one with every point outside the image, three from goodFeaturesToTrack), C = 1500,
    R = 4, fourteen steps.  Random drop masks every frame (a random subset, the whole sequence, nothing, or only slots
    behind the count); restarts with no points, with goodFeaturesToTrack points of the restart frame, with given ids,
    first points and negative first frames, with counts below the points given, and of a sequence that is dropped in the
    same step; two sequences restart at different frames, so their frames differ and their rings wrap after it.  Several
    restart calls before one step: the last one that marks a sequence wins.  Sequence 1 is never dropped or restarted and
    equals a twin without control."""
    import torch
    h, w = KITTI
    R, C, T = 4, 1500, 15
    B = 5
    seqs = [S.sequence(h, w, T, seed=330 + b) for b in range(B)]
    init = [np.zeros((0, 2), np.float32), OUTSIDE.copy()]
    for b in range(2, B):
        init.append(cv2.goodFeaturesToTrack(seqs[b][0], **DET).reshape(-1, 2)[: 300 + 300 * b])
    sb = make(seqs, init, C, R)
    twin = make(seqs, init, C, R, control=False)
    models = [Model(p) for p in init]
    check_state(sb, models, C, R, "frame 0")
    rng = np.random.default_rng(17)
    modes = {"subset": 0, "whole": 0, "none": 0, "behind": 0}
    n_restarts = 0
    for t in range(1, T):
        # drops, aligned with the current rows
        drop = np.zeros((B, C), bool)
        for b in range(B):
            if b == 1:
                continue
            n = len(models[b].ids)
            mode = ["subset", "whole", "none", "behind"][(t + b) % 4]
            modes[mode] += 1
            if mode == "subset":
                drop[b, :n] = rng.random(n) < 0.2
            elif mode == "whole":
                drop[b, :n] = True
            elif mode == "behind":
                drop[b, n:] = rng.random(C - n) < 0.5
        sb.drop(torch.from_numpy(drop).cuda())
        # restarts of the step into frame t: b -> (points (N, 2), counts, ids, first_points, first_frames)
        staged = {}
        flags = np.zeros(B, bool)
        if t in (3, 9):                                      # sequence 2, twice: no points, then gftt points with a short count
            if t == 3:
                staged[2] = (None, None, None, None, None)
            else:
                p = cv2.goodFeaturesToTrack(seqs[2][t], **DET).reshape(-1, 2)[:120]
                staged[2] = (p, len(p) // 2, None, None, None)
        if t == 4:                                           # sequence 3: gftt points of the restart frame
            staged[3] = (cv2.goodFeaturesToTrack(seqs[3][t], **DET).reshape(-1, 2)[:400], None, None, None, None)
        if t == 6:                                           # sequence 4: given ids / first points / negative frames, and dropped
            p = cv2.goodFeaturesToTrack(seqs[4][t], **DET).reshape(-1, 2)[:250]
            ids = (1000 + 7 * np.arange(len(p))).astype(np.int32)
            fp = rng.uniform(-20, 1200, p.shape).astype(np.float32)
            ff = rng.integers(-30, 1, len(p)).astype(np.int32)
            staged[4] = (p, None, ids, fp, ff)
            drop[4, :len(models[4].ids)] = True
            sb.drop(torch.from_numpy(drop).cuda())           # OR-ed with the drops above
        if t == 11:                                          # the empty sequence 0
            staged[0] = (cv2.goodFeaturesToTrack(seqs[0][t], **DET).reshape(-1, 2)[:60], None, None, None, None)
        if staged:
            # a decoy call first: overwritten for the sequences it shares with the real calls
            decoy = np.zeros(B, bool)
            decoy[list(staged)] = True
            sb.restart(torch.from_numpy(decoy).cuda(), torch.full((B, 3, 2), 50.0, device="cuda"))
        for b, (p, cnt, ids, fp, ff) in staged.items():
            m = np.zeros(B, bool)
            m[b] = flags[b] = True
            n_restarts += 1
            if p is None:
                sb.restart(torch.from_numpy(m).cuda())
                continue
            N = len(p)
            pts_t = torch.full((B, N, 2), -1.0, device="cuda")
            pts_t[b] = torch.from_numpy(p).cuda()
            kw = {}
            if cnt is not None:
                kw["counts"] = torch.full((B,), cnt, dtype=torch.int32, device="cuda")
            if ids is not None:
                kw["ids"] = torch.full((B, N), -5, dtype=torch.int32, device="cuda")
                kw["ids"][b] = torch.from_numpy(ids).cuda()
                kw["first_points"] = torch.zeros((B, N, 2), device="cuda")
                kw["first_points"][b] = torch.from_numpy(fp).cuda()
                kw["first_frames"] = torch.zeros((B, N), dtype=torch.int32, device="cuda")
                kw["first_frames"][b] = torch.from_numpy(ff).cuda()
            sb.restart(torch.from_numpy(m).cuda(), pts_t, **kw)
        frames = frames_at(seqs, t)
        sb.step(frames)
        twin.step(frames)
        sb.check()
        keep = sb.keep.cpu().numpy()
        assert np.array_equal(sb.restarted.cpu().numpy(), flags), "frame %d: restarted" % t
        n_new = sb.n_new.cpu().numpy()
        for b, m in enumerate(models):
            n_in = len(m.ids)
            if b in staged:
                p, cnt, ids, fp, ff = staged[b]
                p = np.zeros((0, 2), np.float32) if p is None else p[: (len(p) if cnt is None else cnt)]
                keep_ref = np.zeros(n_in, bool)
                surv = p
                new = detect(cv2, seqs[b][t], surv, C)
                if ids is None:
                    sids = np.arange(m.next_id, m.next_id + len(p), dtype=np.int32)
                    m.next_id += len(p)
                else:
                    sids = ids[: len(p)]
                    m.next_id = int(sids.max()) + 1 if len(sids) else 0
                m.ids = np.concatenate([sids, np.arange(m.next_id, m.next_id + len(new), dtype=np.int32)])
                m.next_id += len(new)
                m.pts = np.concatenate([surv, new]).astype(np.float32)
                m.f = 0
                first_pts = m.pts.copy() if fp is None else np.concatenate([fp[: len(p)], new])
                first_frames = np.zeros(len(m.pts), np.int32) if ff is None else np.concatenate([ff[: len(p)], np.zeros(len(new), np.int32)])
                m.recs = Records(m.pts, m.ids, first_pts, first_frames)
            else:
                if b == 1:
                    keep_ref, surv, new, _n, _bound = cv2_step(cv2, seqs[b][t - 1], seqs[b][t], m.pts, DET, C)
                else:
                    k0, p1 = lk_keep(cv2, seqs[b][t - 1], seqs[b][t], m.pts)
                    keep_ref = k0 & ~drop[b, :n_in]
                    surv = p1[keep_ref]
                    new = detect(cv2, seqs[b][t], surv, C)
                m.ids = np.concatenate([m.ids[keep_ref], np.arange(m.next_id, m.next_id + len(new), dtype=np.int32)])
                m.next_id += len(new)
                m.pts = np.concatenate([surv, new]).astype(np.float32)
                m.f += 1
                m.recs.step(m.f, m.ids, m.pts)
            assert np.array_equal(keep[b, :n_in], keep_ref) and not keep[b, n_in:].any(), "frame %d sequence %d: keep" % (t, b)
            assert int(n_new[b]) == len(new), "frame %d sequence %d: n_new" % (t, b)
        check_state(sb, models, C, R, "frame %d" % t)
        # sequence 1 equals the twin without control
        for name in ("points", "ids", "keep", "first_points", "first_frames", "lengths"):
            x, y = getattr(sb, name)[1].cpu().numpy(), getattr(twin, name)[1].cpu().numpy()
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "frame %d: sequence 1 %s differs from control=False" % (t, name)
        assert int(sb.counts[1]) == int(twin.counts[1]) and int(sb.n_new[1]) == int(twin.n_new[1])
        assert np.array_equal(sb.window(R)[1].cpu().numpy().view(np.uint32), twin.window(R)[1].cpu().numpy().view(np.uint32))
    assert sb.frame == T - 1 and n_restarts == 5 and min(modes.values()) > 0
    fr = sb.frames.cpu().numpy()
    assert len(set(fr.tolist())) >= 3 and fr[3] > R, fr         # frames differ, and sequence 3's ring wrapped after its restart


def test_idle_control_equals_plain(klt, cv2):
    """control=True without drops or restarts gives the outputs, records, windows and history of control=False."""
    h, w = KITTI
    R = 3
    seqs = [S.sequence(h, w, 6, seed=410 + b) for b in range(3)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 200 + 300 * b] for b, s in enumerate(seqs)]
    a = make(seqs, init, 1200, R, control=True)
    b_ = make(seqs, init, 1200, R, control=False)
    for t in range(1, 6):
        frames = frames_at(seqs, t)
        a.step(frames)
        b_.step(frames)
        for name in ("points", "counts", "ids", "keep", "n_new", "first_points", "first_frames", "lengths", "frames"):
            x, y = getattr(a, name).cpu().numpy(), getattr(b_, name).cpu().numpy()
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "frame %d: %s" % (t, name)
        assert not a.restarted.any()
        assert np.array_equal(a.window(R).cpu().numpy().view(np.uint32), b_.window(R).cpu().numpy().view(np.uint32))
        for name, x, y in zip(a.history()._fields, a.history(), b_.history()):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "frame %d: history().%s" % (t, name)
    a.check()


@pytest.mark.parametrize("B", [4, 6])
@pytest.mark.parametrize("prefilter", [None, (5, 1.5, 1.5)])
def test_graph_replay_equals_eager(klt, cv2, B, prefilter):
    """Ten frames with R = 4: between steps, each object computes on the device, from its own state, a drop mask (every
    track whose id is a multiple of 5) and a restart mask (the sequences with the fewest points, every third frame), and
    restarts them with the first 40 of their own points.  No host read between replays; the graph object equals the
    eager one bit for bit."""
    import torch
    h, w = KITTI
    R = 4
    seqs = [S.sequence(h, w, 11, seed=470 + b) for b in range(B)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 100 + 200 * b] for b, s in enumerate(seqs)]
    init[0] = init[0][:0]
    eager = make(seqs, init, 1800, R, prefilter=prefilter)
    graph = make(seqs, init, 1800, R, prefilter=prefilter)
    restarts = 0
    for t in range(1, 11):
        for sb in (eager, graph):
            c = sb.counts
            sb.drop((sb.ids % 5 == 0) & (torch.arange(sb.capacity, device="cuda")[None, :] < c[:, None]))
            if t % 3 == 0:
                sb.restart(c <= c.min(), sb.points[:, :40].clone(), torch.clamp(c, max=40), ids=sb.ids[:, :40] + 100000)
        frames = frames_at(seqs, t)
        eager.step(frames)
        graph.step(frames)
        if t == 1:
            graph.capture()
        restarts += int(eager.restarted.sum())
        assert eager.frame == graph.frame == t
        for name in ("points", "counts", "ids", "keep", "n_new", "restarted", "frames", "first_points", "first_frames", "lengths"):
            x, y = getattr(eager, name).cpu().numpy(), getattr(graph, name).cpu().numpy()
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "frame %d: %s" % (t, name)
        for k in (1, 2, 4):
            assert np.array_equal(eager.window(k).cpu().numpy().view(np.uint32), graph.window(k).cpu().numpy().view(np.uint32))
        for name, x, y in zip(eager.history()._fields, eager.history(), graph.history()):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "frame %d: history().%s" % (t, name)
        eager.check()
        graph.check()
    assert graph._graphs is not None and restarts >= 3


def test_errors_and_clamped_counts(klt):
    import torch
    from visual_odom_pipeline_b200 import _lib
    from visual_odom_pipeline_b200 import tracker as T
    from visual_odom_pipeline_b200.lk import error
    h, w = 64, 96
    frames = torch.from_numpy(np.stack([S.sequence(h, w, 2, seed=90 + b)[1] for b in range(3)])).cuda()
    pts = torch.full((3, 8, 2), 20.0, device="cuda")
    cnt = torch.tensor([8, 0, 3], dtype=torch.int32, device="cuda")
    C = 16
    plain = T.KLTSequenceBatch(frames, pts, cnt, C, history=2)
    with pytest.raises(error):
        plain.drop(torch.zeros((3, C), dtype=torch.bool, device="cuda"))
    with pytest.raises(error):
        plain.restart(torch.zeros(3, dtype=torch.bool, device="cuda"))
    with pytest.raises(error):
        plain.restarted
    nohist = T.KLTSequenceBatch(frames, pts, cnt, C, control=True)
    with pytest.raises(error):
        nohist.frames
    seqs = torch.tensor([True, False, True], device="cuda")
    with pytest.raises(error):                                        # first points need history >= 1
        nohist.restart(seqs, pts, first_points=pts, first_frames=torch.zeros((3, 8), dtype=torch.int32, device="cuda"))
    sb = T.KLTSequenceBatch(frames, pts, cnt, C, history=2, control=True)
    for bad in (torch.zeros((3, C - 1), dtype=torch.bool, device="cuda"), torch.zeros((3, C), dtype=torch.uint8, device="cuda"),
                torch.zeros((3, C), dtype=torch.bool)):
        with pytest.raises(error):
            sb.drop(bad)
    ff = torch.zeros((3, 8), dtype=torch.int32, device="cuda")
    bad_restarts = [
        dict(seqs=seqs.int()), dict(seqs=seqs[:2]), dict(seqs=seqs.cpu()),
        dict(seqs=seqs, counts=cnt), dict(seqs=seqs, ids=ff), dict(seqs=seqs, first_points=pts, first_frames=ff),
        dict(seqs=seqs, points=torch.zeros((3, C + 1, 2), device="cuda")), dict(seqs=seqs, points=pts.double()),
        dict(seqs=seqs, points=pts[:2]), dict(seqs=seqs, points=pts.cpu()),
        dict(seqs=seqs, points=pts, counts=cnt.long()), dict(seqs=seqs, points=pts, counts=cnt[:2]),
        dict(seqs=seqs, points=pts, ids=ff[:, :4]), dict(seqs=seqs, points=pts, ids=ff.long()),
        dict(seqs=seqs, points=pts, first_points=pts), dict(seqs=seqs, points=pts, first_frames=ff),
        dict(seqs=seqs, points=pts, first_points=pts[:, :4], first_frames=ff), dict(seqs=seqs, points=pts, first_points=pts, first_frames=ff.long()),
    ]
    for kw in bad_restarts:
        with pytest.raises(error):
            sb.restart(**kw)
    sb.step(frames)
    sb.check()
    assert not sb.restarted.any()

    # staged counts outside [0, N]: clamped, flagged, no fault
    sb.restart(seqs, pts, counts=torch.tensor([9, 0, -2], dtype=torch.int32, device="cuda"))
    sb.step(frames)
    with pytest.raises(error):
        sb.check()
    got = sb.counts.cpu().numpy()
    assert sb.restarted.cpu().numpy().tolist() == [True, False, True]
    assert got[0] == 8 + int(sb.n_new[0]) and got[2] == int(sb.n_new[2])
    assert np.array_equal(sb.points[0, :8].cpu().numpy(), pts[0].cpu().numpy()) and bool((sb.frames[[0, 2]] == 0).all())
    sb.check()

    # the entry points' own argument checks
    L = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    cur, nxt = sb._cur, 1 - sb._cur
    prev, new = sb._slots[cur], sb._slots[nxt]

    def step_args(ids=True):
        return [sb.ctx.handle, prev.images.data_ptr(), prev.buffer.data_ptr(), new.images.data_ptr(), new.buffer.data_ptr(),
                prev.layout, 0, 0, 1, 3, sb._pts[cur].data_ptr(), sb._counts[cur].data_ptr(), C, sb.params, sb.max_bidir_error,
                sb.mask_radius, sb.maxCorners, sb.qualityLevel, sb.minDistance, sb.blockSize, sb._pts[nxt].data_ptr(), C,
                sb._keep.data_ptr(), sb._counts[nxt].data_ptr(), sb._n_new.data_ptr(), sb._ids[cur].data_ptr() if ids else None,
                sb._ids[nxt].data_ptr() if ids else None, sb._next_id.data_ptr() if ids else None, sb._flags.data_ptr(), sb._ws_ptr,
                sb._ws_bytes]

    def ctl(**kw):
        c = _lib.klt_step_control(sb._ctl.d_drop, sb._ctl.d_restart, sb._ctl.d_restart_pts, sb._ctl.d_restart_counts,
                                  sb._ctl.d_restart_ids, sb._ctl.d_restart_next_id, sb._ctl.d_restarted)
        for k, v in kw.items():
            setattr(c, k, v)
        return c

    inval = _lib.KLT_ERR_INVALID_ARG
    assert L.klt_frame_step_batch_control_async(*step_args(), None, st) == inval                          # null control
    for kw in (dict(d_restarted=None), dict(d_restart_pts=None), dict(d_restart_counts=None),
               dict(d_restart_ids=None), dict(d_restart_next_id=None)):
        assert L.klt_frame_step_batch_control_async(*step_args(), ctl(**kw), st) == inval, kw
    assert L.klt_frame_step_batch_control_async(*step_args(ids=False), ctl(), st) == inval                # staged ids, no step ids
    assert L.klt_frame_step_batch_control_async(*step_args(ids=False), ctl(d_restart_ids=None), st) == inval
    rgood = [sb.ctx.handle, 3, C, C, sb._keep.data_ptr(), sb._pts[nxt].data_ptr(), sb._ids[nxt].data_ptr(), sb._counts[nxt].data_ptr(),
             sb._first_pts[cur].data_ptr(), sb._first_frames[cur].data_ptr(), sb._first_pts[nxt].data_ptr(),
             sb._first_frames[nxt].data_ptr(), sb._frame.data_ptr(), 2, sb._ring_pts.data_ptr(), sb._ring_ids.data_ptr(),
             sb._ring_src.data_ptr(), sb._ring_counts.data_ptr(), sb._ring_frames.data_ptr(), sb._restarted.data_ptr(),
             sb._rs_counts.data_ptr(), sb._rs_first_pts.data_ptr(), sb._rs_first_frames.data_ptr(), st]
    for i in [0, 4, 5, 6, 7, 8, 12, 14, 19, 20]:
        args = list(rgood)
        args[i] = None
        assert L.klt_track_records_step_control(*args) == inval, "null argument %d" % i
    for i, v in [(13, 0), (3, C - 1), (2, -1), (1, 0)]:
        args = list(rgood)
        args[i] = v
        assert L.klt_track_records_step_control(*args) == inval, (i, v)
    # nothing was launched by the rejected calls
    torch.cuda.synchronize()
    assert bool((sb._frame == torch.tensor([0, 2, 0], dtype=torch.int32, device="cuda")).all())

    # a drop-only control (no restart array) through the C entry point, with staged counts out of range that nobody reads,
    # then a staged count above n_per_seq: clamped and flagged
    rc = L.klt_frame_step_batch_control_async(*step_args(), ctl(d_restart=None, d_restart_pts=None, d_restart_counts=None,
                                                                d_restart_ids=None, d_restart_next_id=None), st)
    assert rc == _lib.KLT_OK
    torch.cuda.synchronize()
    assert int(sb._flags.item()) == 0
    sb._rs_counts.fill_(C + 5)
    sb._rs_flag.fill_(1)
    assert L.klt_frame_step_batch_control_async(*step_args(), ctl(), st) == _lib.KLT_OK
    torch.cuda.synchronize()
    assert int(sb._flags.item()) == 1 and bool((sb._rs_flag == 0).all()) and bool((sb._restarted == 1).all())
    assert bool((sb._counts[nxt] <= C).all())
