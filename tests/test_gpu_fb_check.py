"""GPU tier (pytest -m gpu, B200) of the forward-backward check (second_pass="reverse"): the step's second LK pass runs
from the new frame back into the old one, in KLTSequenceBatch (with every combination of history, control and
motion_prior, eagerly and replayed from the graphs), KLTTracker and trackBidirectional.

Bar: every sequence and frame against the capped cv2 loop whose second call is cv2.calcOpticalFlowPyrLK(im1, im0, p1, b)
(tests/test_fb_check_cpu.py, fb_keep_from): keep, survivors (as uint32), new corners, counts, ids, n_new and bidir_error
(as uint32; NaN where the host's d is NaN, behind the count and for a restarted sequence), and with history the records."""
import json
import os

import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from test_fb_check_cpu import FAST_FB, FAST_MOTIONS, FB_CAP, FB_MAX_ERR, REF_LK, fast_case, fb_keep_from
from test_gpu_frame_step_async import DET, KITTI, LK, pad
from test_gpu_frame_step_lk_shapes import CASES, check_launches, lk_launches
from test_gpu_motion_prior import given_requests, shape_batch, shape_starts, with_restarts
from test_gpu_sequence_control import Model, check_state
from test_gpu_track_history import Records, frames_at
from test_motion_prior_cpu import detect, velocity_starts

pytestmark = pytest.mark.gpu

SNAP = ("points", "counts", "ids", "keep", "n_new", "bidir_error")


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def make(seqs, init, cap, history=0, control=False, motion_prior=None, lk=LK, max_err=FB_MAX_ERR, second_pass="reverse"):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init, n=cap)
    return T.KLTSequenceBatch(frames_at(seqs, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), cap,
                              history=history, control=control, motion_prior=motion_prior, max_bidir_error=max_err,
                              second_pass=second_pass, **lk, **DET)


def same_d(got, want):
    """float32 arrays equal bit for bit, NaN (of any payload) where want is NaN."""
    nan = np.isnan(want)
    return np.array_equal(np.isnan(got), nan) and np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def drive(cv2, seqs, init, C, R, prior, requests, lk=LK, control=False, check_records=True):
    """test_gpu_motion_prior.drive with the reverse second pass: an eager object and a graph-replayed twin (captured after
    the first step), both checked against the host loop every frame, bidir_error included.  Returns the host models and,
    per step, the survivors per sequence."""
    import torch
    B = len(seqs)
    T = len(seqs[0])
    objs = [make(seqs, init, C, R, control, prior, lk) for _ in range(2)]
    models = [Model(np.asarray(p, np.float32).reshape(-1, 2)) for p in init]
    kept = []
    for t in range(1, T):
        req = requests(t, models)
        for sb in objs:
            for pts, mask in req.get("predict", []):
                sb.predict(torch.from_numpy(pts).cuda(), torch.from_numpy(mask).cuda())
            if req.get("drop") is not None:
                sb.drop(torch.from_numpy(req["drop"]).cuda())
            for b, p in req.get("restart", {}).items():
                m = np.zeros(B, bool)
                m[b] = True
                pt = torch.full((B, len(p), 2), -1.0, device="cuda")
                pt[b] = torch.from_numpy(p).cuda()
                sb.restart(torch.from_numpy(m).cuda(), pt)
        frames = frames_at(seqs, t)
        for sb in objs:
            sb.step(frames)
        if t == 1:
            objs[1].capture()
        snaps = [{k: getattr(sb, k).cpu().numpy() for k in SNAP} for sb in objs]
        for sb in objs:
            sb.check()
        drop = req.get("drop")
        kept.append([])
        for b, m in enumerate(models):
            n = len(m.ids)
            if b in req.get("restart", {}):
                p = req["restart"][b]
                keep_ref = np.zeros(n, bool)
                d_ref = np.full(n, np.nan, np.float32)
                surv = p
                new = detect(cv2, seqs[b][t], surv, C)
                sids = np.arange(m.next_id, m.next_id + len(p), dtype=np.int32)
                m.next_id += len(p)
                m.ids = np.concatenate([sids, np.arange(m.next_id, m.next_id + len(new), dtype=np.int32)])
                m.next_id += len(new)
                m.pts = np.concatenate([surv, new]).astype(np.float32)
                m.f = 0
                m.recs = Records(m.pts, m.ids)
            else:
                starts = None
                if prior is not None:
                    starts = m.pts.copy()
                    if prior == "velocity":
                        prev = np.array([m.recs.pos[int(i)].get(m.f - 1, (np.nan, np.nan)) for i in m.ids], np.float32).reshape(-1, 2)
                        starts = velocity_starts(m.pts, prev)
                    for pts, mask in req.get("predict", []):
                        starts[mask[b, :n]] = pts[b, :n][mask[b, :n]]
                keep_ref, p1, d_ref = fb_keep_from(cv2, lk, seqs[b][t - 1], seqs[b][t], m.pts, starts)
                if drop is not None:
                    keep_ref = keep_ref & ~drop[b, :n]
                surv = p1[keep_ref]
                new = detect(cv2, seqs[b][t], surv, C)
                m.ids = np.concatenate([m.ids[keep_ref], np.arange(m.next_id, m.next_id + len(new), dtype=np.int32)])
                m.next_id += len(new)
                m.pts = np.concatenate([surv, new]).astype(np.float32)
                m.f += 1
                if R:
                    m.recs.step(m.f, m.ids, m.pts)
            kept[-1].append(surv)
            for name, g in zip(("eager", "graph"), snaps):
                tag = "%s frame %d sequence %d" % (name, t, b)
                assert np.array_equal(g["keep"][b, :n], keep_ref) and not g["keep"][b, n:].any(), tag + ": keep (%d differ)" % (
                    int((g["keep"][b, :n] != keep_ref).sum()))
                assert same_d(g["bidir_error"][b, :n], d_ref), tag + ": bidir_error"
                assert np.isnan(g["bidir_error"][b, n:]).all(), tag + ": bidir_error behind the count"
                assert int(g["n_new"][b]) == len(new), tag + ": n_new"
                assert int(g["counts"][b]) == len(m.ids), tag + ": counts"
                assert np.array_equal(g["points"][b, :len(m.ids)].view(np.uint32), m.pts.view(np.uint32)), tag + ": points"
                assert np.array_equal(g["ids"][b, :len(m.ids)], m.ids), tag + ": ids"
        if R and check_records:
            for sb, name in zip(objs, ("eager", "graph")):
                check_state(sb, models, C, R, "%s frame %d" % (name, t))
    assert objs[1]._graphs is not None
    return models, kept


def inputs(cv2, B, seed, frames=9, motion=(1.1, -0.6, 0.15, 1.003), empty=True):
    """B KITTI sequences and different initial counts per sequence (the first one empty when `empty`)."""
    h, w = KITTI
    seqs = [S.sequence(h, w, frames, seed=seed + b, motion=motion) for b in range(B)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 300 * b + 150] for b, s in enumerate(seqs)]
    if empty:
        init[0] = np.zeros((0, 2), np.float32)
    return seqs, init


def test_plain_against_cv2_loop(klt, cv2):
    """No history, control or prior: four sequences (one empty), C = 1200, eight steps."""
    seqs, init = inputs(cv2, 4, seed=1100)
    drive(cv2, seqs, init, 1200, 0, None, lambda t, m: {})


def test_history_control_drop_and_restart(klt, cv2):
    """history=4, control=True: random drops every step, and restarts of two sequences at different frames (NaN errors for
    them in that step)."""
    B, C = 4, 1200
    seqs, init = inputs(cv2, B, seed=1120)
    rng = np.random.default_rng(7)

    def req(t, models):
        d = np.zeros((B, C), bool)
        for b, m in enumerate(models):
            d[b, :len(m.ids)] = rng.random(len(m.ids)) < 0.15
        return {"drop": d}

    models, _ = drive(cv2, seqs, init, C, 4, None, with_restarts(cv2, seqs, req, {3: {2: 120}, 5: {0: 40}}), control=True)
    assert models[2].f == 5 and models[0].f == 3


@pytest.mark.parametrize("motion", [(1.1, -0.6, 0.15, 1.003), (10.0, 1.5, 0.2, 1.0)], ids=["default", "10px"])
def test_velocity_prior(klt, cv2, motion):
    """motion_prior="velocity" (R = 2): the reverse pass starts at the mirrored start p1 - (s - p0) with the flag."""
    seqs, init = inputs(cv2, 3, seed=1140, motion=motion)
    drive(cv2, seqs, init, 1500, 2, "velocity", lambda t, m: {})


def test_given_prior_with_nan_and_outside(klt, cv2):
    """motion_prior="given": a random half of the slots every step at positions of every kind (the true next position,
    offsets, outside the image, NaN, +-inf), control with drops, and a restart."""
    B, C = 4, 1200
    motion = (1.1, -0.6, 0.15, 1.003)
    seqs, init = inputs(cv2, B, seed=1160, motion=motion)
    req = with_restarts(cv2, seqs, given_requests(B, C, motion, seed=31, two_calls=(3,), drops=True), {4: {1: 90}})
    drive(cv2, seqs, init, C, 4, "given", req, control=True)


# ---- every LK instance of the step runs both passes with the same shape --------------------------------------------------

@pytest.fixture(scope="module")
def sms(klt):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def launches(klt, tmp_path_factory):
    """The LK launches of each case's first reverse step with start positions, profiled in a child process (this file run
    as a script; see test_gpu_frame_step_lk_shapes.py for why the test process never starts a CUPTI session)."""
    import subprocess
    import sys
    out = tmp_path_factory.mktemp("fb_launches")
    tests = os.path.dirname(os.path.abspath(__file__))
    path = [os.path.dirname(tests), tests] + ([os.environ["PYTHONPATH"]] if os.environ.get("PYTHONPATH") else [])
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, PYTHONPATH=os.pathsep.join(path)), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, "profiling child failed:\n" + r.stdout[-4000:] + r.stderr[-4000:]
    with open(out / "launches.json") as f:
        return {k: [(n, tuple(g), tuple(b)) for n, g, b in v] for k, v in json.load(f).items()}


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_lk_instance_reverse_pass(klt, cv2, sms, launches, capsys, case):
    """The first step (profiled in the `launches` child) ran the forward and the reverse pass with the case's instance,
    grid and block; then three steps with the velocity prior (R = 2) and given starts on half the slots equal the cv2 loop,
    eagerly and replayed."""
    B, C, lk, seqs, init = shape_batch(cv2, case, sms, CASES.index(case))
    lo, hi = case.side
    assert (lo is None or B * C > lo * sms) and (hi is None or B * C <= hi * sms), (case.name, B, C, sms)
    check_launches(case, launches[case.name], B * C, capsys, "KLTSequenceBatch.step, reverse second pass")
    seed = 1200 + CASES.index(case)
    drive(cv2, seqs, init, C, 2, "velocity", lambda t, models: {"predict": [shape_starts(seqs, t, [m.pts for m in models], C, seed)]},
          lk=lk, check_records=False)


# ---- the fast sequences of the CPU tier ------------------------------------------------------------------------------------

@pytest.mark.parametrize("px", sorted(FAST_MOTIONS))
def test_fast_sequences_counts(klt, cv2, px):
    """16 and 20 px per frame, the library's parameters: the device loop equals the cv2 loop, and its survivor counts are the
    CPU tier's pinned numbers, for the reverse check at 1 px and for the reference's check at 30."""
    seq, init = fast_case(cv2, px)
    _models, kept = drive(cv2, [seq], [init], FB_CAP, 0, None, lambda t, m: {}, lk=REF_LK)
    assert [len(k[0]) for k in kept] == [n for n, _o, _l in FAST_FB[(px, "reverse")]]
    sb = make([seq], [init], FB_CAP, lk=REF_LK, max_err=30, second_pass="reference")
    counts = []
    for t in range(1, len(seq)):
        sb.step(frames_at([seq], t))
        counts.append(int(sb.keep.sum()))
    sb.check()
    assert counts == [n for n, _o, _l in FAST_FB[(px, "reference")]]


# ---- KLTTracker and trackBidirectional --------------------------------------------------------------------------------------

def tracker_inputs(cv2, B=2, n=600, seed=1300):
    h, w = KITTI
    seqs = [S.sequence(h, w, 3, seed=seed + b, motion=(6.0, -1.0, 0.3, 1.002)) for b in range(B)]
    pts = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[:n] for s in seqs]
    n = min(len(p) for p in pts)
    pts = np.stack([p[:n] for p in pts]).astype(np.float32)
    pts[0, 3] = np.nan
    pts[-1, 5] = (-30.0, 40.0)
    return seqs, pts


def test_tracker_track_and_track_filtered(klt, cv2):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    seqs, pts = tracker_inputs(cv2)
    B = len(seqs)
    for filtered in (False, True):
        trk = T.KLTTracker(**LK).reset(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda())
        for t in (1, 2):
            im1 = torch.from_numpy(np.stack([s[t] for s in seqs])).cuda()
            p0 = torch.from_numpy(pts).cuda()
            if filtered:
                p1, keep, bidir, _st, _er = [x.cpu().numpy() for x in trk.track_filtered(im1, p0, FB_MAX_ERR, second_pass="reverse")]
            else:
                p1, _st, _er, p0r = [x.cpu().numpy() for x in trk.track(im1, p0, bidirectional=True, second_pass="reverse")]
            for b in range(B):
                keep_ref, p1_ref, d_ref = fb_keep_from(cv2, LK, seqs[b][t - 1], seqs[b][t], pts[b], None)
                assert same_d(p1[b], p1_ref), (filtered, t, b)
                if filtered:
                    assert np.array_equal(keep[b], keep_ref) and same_d(bidir[b], d_ref), (t, b)
                else:
                    want, _s, _e = cv2.calcOpticalFlowPyrLK(seqs[b][t], seqs[b][t - 1], p1_ref.reshape(-1, 1, 2), None, **LK)
                    assert same_d(p0r[b], want.reshape(-1, 2)), (t, b)


def test_tracker_step_and_step_batch(klt, cv2):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    seqs, pts = tracker_inputs(cv2, seed=1320)
    B = len(seqs)
    counts = np.array([len(pts[0]) - 17, len(pts[1])], np.int32)
    single = [T.KLTTracker(**LK).reset(torch.from_numpy(seqs[b][0]).cuda()) for b in range(B)]
    batch = T.KLTTracker(**LK).reset(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda())
    for t in (1, 2):
        for b in range(B):
            p = pts[b, :counts[b]]
            keep_ref, p1_ref, _d = fb_keep_from(cv2, LK, seqs[b][t - 1], seqs[b][t], p, None)
            surv_ref = p1_ref[keep_ref]
            new_ref = detect(cv2, seqs[b][t], surv_ref, 10 ** 9)
            surv, keep, new = single[b].step(torch.from_numpy(seqs[b][t]).cuda(), torch.from_numpy(p).cuda(),
                                             max_bidir_error=FB_MAX_ERR, second_pass="reverse", **DET)
            assert np.array_equal(keep.cpu().numpy(), keep_ref), (t, b)
            assert np.array_equal(surv.cpu().numpy().view(np.uint32), surv_ref.view(np.uint32)), (t, b)
            assert np.array_equal(np.zeros((0, 2), np.float32) if new is None else new.reshape(-1, 2), new_ref), (t, b)
        frames = torch.from_numpy(np.stack([s[t] for s in seqs])).cuda()
        out = batch.step_batch(frames, torch.from_numpy(pts).cuda(), torch.from_numpy(counts).cuda(), max_bidir_error=FB_MAX_ERR,
                               second_pass="reverse", **DET)
        nxt, ncnt, keep, n_new = [x.cpu().numpy() for x in out]
        for b in range(B):
            p = pts[b, :counts[b]]
            keep_ref, p1_ref, _d = fb_keep_from(cv2, LK, seqs[b][t - 1], seqs[b][t], p, None)
            surv_ref = p1_ref[keep_ref]
            new_ref = detect(cv2, seqs[b][t], surv_ref, 10 ** 9)
            s, k = len(surv_ref), len(new_ref)
            assert np.array_equal(keep[b, :counts[b]], keep_ref) and not keep[b, counts[b]:].any(), (t, b)
            assert int(ncnt[b]) == s + k and int(n_new[b]) == k, (t, b)
            assert np.array_equal(nxt[b, :s].view(np.uint32), surv_ref.view(np.uint32)) and np.array_equal(nxt[b, s:s + k], new_ref)


def test_track_bidirectional_reverse(klt, cv2):
    """Pageable numpy frames, as the reference passes them: p1, status, err are cv2's first call, d and keep those of the
    reverse check; N = 0 returns Nones; a NaN point goes through as cv2 takes it."""
    from visual_odom_pipeline_b200 import lk as K
    seqs, pts = tracker_inputs(cv2, B=1, seed=1340)
    im0, im1 = seqs[0][0].copy(), seqs[0][1].copy()
    p0 = pts[0].reshape(-1, 1, 2)
    for max_err in (FB_MAX_ERR, 30.0):
        p1, keep, d, st, er = K.trackBidirectional(im0, im1, p0, max_bidir_error=max_err, second_pass="reverse")
        keep_ref, p1_ref, d_ref = fb_keep_from(cv2, LK, im0, im1, pts[0], None, max_bidir=max_err)
        q, st_ref, er_ref = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **LK)
        assert p1.shape == p0.shape and same_d(p1, q)
        assert np.array_equal(st, st_ref)
        both = (st.reshape(-1) == 1)
        assert np.array_equal(er.reshape(-1)[both].view(np.uint32), er_ref.reshape(-1)[both].view(np.uint32))
        assert np.array_equal(keep, keep_ref) and same_d(d, d_ref)
        assert np.isnan(d[3]) and not keep[3]
    assert K.trackBidirectional(im0, im1, np.zeros((0, 1, 2), np.float32), second_pass="reverse") == (None,) * 5


def test_errors(klt):
    import torch
    from visual_odom_pipeline_b200 import lk as K
    from visual_odom_pipeline_b200 import tracker as T
    from visual_odom_pipeline_b200.lk import error
    h, w = 64, 96
    frames = torch.from_numpy(np.stack([S.sequence(h, w, 2, seed=90 + b)[1] for b in range(3)])).cuda()
    pts = torch.full((3, 8, 2), 20.0, device="cuda")
    cnt = torch.tensor([8, 0, 3], dtype=torch.int32, device="cuda")
    for bad in ("forward", None, "REVERSE", 1):
        with pytest.raises(error):
            T.KLTSequenceBatch(frames, pts, cnt, 16, second_pass=bad)
        with pytest.raises(error):
            K.trackBidirectional(frames[0].cpu().numpy(), frames[1].cpu().numpy(), np.zeros((4, 2), np.float32), second_pass=bad)
    plain = T.KLTSequenceBatch(frames, pts, cnt, 16)
    with pytest.raises(error):
        plain.bidir_error
    sb = T.KLTSequenceBatch(frames, pts, cnt, 16, second_pass="reverse")
    assert np.isnan(sb.bidir_error.cpu().numpy()).all()              # before the first step
    sb.step(frames).check()
    d = sb.bidir_error.cpu().numpy()
    assert d.shape == (3, 16) and d.dtype == np.float32
    assert not np.isnan(d[0, :8]).all() and np.isnan(d[1]).all() and np.isnan(d[2, 3:]).all()


if __name__ == "__main__":
    # the child process of the `launches` fixture: python tests/test_gpu_fb_check.py OUT_DIR
    import sys
    import cv2 as cv2_
    import torch
    sms_ = torch.cuda.get_device_properties(0).multi_processor_count
    res = {}
    for i, case in enumerate(CASES):
        B, C, lk, seqs, init = shape_batch(cv2_, case, sms_, i)
        sb = make(seqs, init, C, 2, False, "velocity", lk)
        p, m = shape_starts(seqs, 1, [np.asarray(x, np.float32).reshape(-1, 2) for x in init], C, 1200 + i)
        sb.predict(torch.from_numpy(p).cuda(), torch.from_numpy(m).cuda())
        frames = frames_at(seqs, 1)
        res[case.name] = lk_launches(torch, lambda: sb.step(frames), os.path.join(sys.argv[1], "%d.json" % i))
    with open(os.path.join(sys.argv[1], "launches.json"), "w") as f:
        json.dump(res, f)
