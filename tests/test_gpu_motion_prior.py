"""GPU tier (pytest -m gpu, B200) of the motion prior of KLTSequenceBatch: the forward LK pass of each step starts at
positions a back end gave with predict(), or at p + (p - q) from each track's own velocity, on the device and inside the
graphs.

Bar: every sequence and frame, eagerly and replayed from the graphs, against the capped cv2 loop whose forward call is
cv2.calcOpticalFlowPyrLK(im0, im1, p0, starts, flags=cv2.OPTFLOW_USE_INITIAL_FLOW), the starts restated on the host
(tests/test_motion_prior_cpu.py): keep, survivors (as uint32), new corners, counts, ids and n_new, and with history the
records of test_gpu_sequence_control.py (first points and frames, windows, history rows and tracks)."""
import json
import os

import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from test_gpu_frame_step_async import DET, KITTI, LK, pad
from test_gpu_frame_step_lk_shapes import CASES, FAST, Case, case_inputs, check_launches, lk_launches
from test_gpu_sequence_control import Model, check_state
from test_gpu_track_history import OUTSIDE, Records, frames_at
from test_motion_prior_cpu import FAST_LK, FAST_ON_MOTION, FAST_STEPS, detect, fine_sequence, host_loop, lk_keep_from, velocity_starts

pytestmark = pytest.mark.gpu

SNAP = ("points", "counts", "ids", "keep", "n_new")


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def make(seqs, init, cap, history=0, control=False, motion_prior=None, lk=LK):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init, n=cap)
    return T.KLTSequenceBatch(frames_at(seqs, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), cap,
                              history=history, control=control, motion_prior=motion_prior, **lk, **DET)


def true_next(pts, motion, h, w):
    """Where synth.warp(motion) moves each point (float32)."""
    tx, ty, rot, scale = motion
    a = np.deg2rad(rot)
    al, be = scale * np.cos(a), scale * np.sin(a)
    cx, cy = w / 2, h / 2
    x, y = pts[:, 0].astype(np.float64), pts[:, 1].astype(np.float64)
    nx = al * x + be * y + (1 - al) * cx - be * cy + tx
    ny = -be * x + al * y + be * cx + (1 - al) * cy + ty
    return np.stack([nx, ny], -1).astype(np.float32)


def drive(cv2, seqs, init, C, R, prior, requests, lk=LK, control=False, check_records=True):
    """Steps an eager object and a graph-replayed twin (captured after the first step) with the same requests, and checks
    both against the host loop every frame.  requests(t, models) -> dict with optional "predict": [(points (B, C, 2),
    mask (B, C))], "drop": (B, C) bool, "restart": {b: points (N, 2)}.  Returns the host models and, per step, the
    survivors per sequence."""
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
                starts = m.pts.copy()
                if prior == "velocity":
                    prev = np.array([m.recs.pos[int(i)].get(m.f - 1, (np.nan, np.nan)) for i in m.ids], np.float32).reshape(-1, 2)
                    starts = velocity_starts(m.pts, prev)
                for pts, mask in req.get("predict", []):
                    starts[mask[b, :n]] = pts[b, :n][mask[b, :n]]
                keep_ref, p1 = lk_keep_from(cv2, lk, seqs[b][t - 1], seqs[b][t], m.pts, starts)
                if drop is not None:
                    keep_ref = keep_ref & ~drop[b, :n]
                surv = p1[keep_ref]
                new = detect(cv2, seqs[b][t], surv, C)
                m.ids = np.concatenate([m.ids[keep_ref], np.arange(m.next_id, m.next_id + len(new), dtype=np.int32)])
                m.next_id += len(new)
                m.pts = np.concatenate([surv, new]).astype(np.float32)
                m.f += 1
                m.recs.step(m.f, m.ids, m.pts)
            kept[-1].append(surv)
            for name, g in zip(("eager", "graph"), snaps):
                tag = "%s frame %d sequence %d" % (name, t, b)
                assert np.array_equal(g["keep"][b, :n], keep_ref) and not g["keep"][b, n:].any(), tag + ": keep (%d differ)" % (
                    int((g["keep"][b, :n] != keep_ref).sum()))
                assert int(g["n_new"][b]) == len(new), tag + ": n_new"
                assert int(g["counts"][b]) == len(m.ids), tag + ": counts"
                assert np.array_equal(g["points"][b, :len(m.ids)].view(np.uint32), m.pts.view(np.uint32)), tag + ": points"
                assert np.array_equal(g["ids"][b, :len(m.ids)], m.ids), tag + ": ids"
        if R and check_records:
            for sb, name in zip(objs, ("eager", "graph")):
                check_state(sb, models, C, R, "%s frame %d" % (name, t))
    assert objs[1]._graphs is not None
    return models, kept


def given_requests(B, C, motion, seed, two_calls=(), drops=False, kinds=6):
    """Random given positions every step: a random half of the slots of each sequence, each of one kind (the warp's true
    next position, an offset of 0.5 - 40 px, a point outside the image, NaN, +inf or -inf; the first `kinds` of them), and
    random marks behind the count.  Steps in two_calls add a second predict() that overrides part of the first and marks
    more slots.  drops: random drops every step (needs control=True)."""
    h, w = KITTI
    rng = np.random.default_rng(seed)

    def req(t, models):
        pts = np.full((B, C, 2), 7.0, np.float32)
        mask = np.zeros((B, C), bool)
        for b, m in enumerate(models):
            n = len(m.ids)
            sel = rng.random(n) < 0.5
            kind = rng.integers(0, kinds, n)
            p = m.pts.copy()
            good = true_next(p, motion, h, w)
            ang = rng.uniform(0, 2 * np.pi, n)
            r = rng.uniform(0.5, 40, n)
            off = (p + np.stack([r * np.cos(ang), r * np.sin(ang)], -1)).astype(np.float32)
            outside = OUTSIDE[rng.integers(0, len(OUTSIDE), n)]
            special = {3: (np.nan, np.nan), 4: (np.inf, 5.0), 5: (10.0, -np.inf)}
            q = np.where((kind == 0)[:, None], good, np.where((kind == 1)[:, None], off, outside))
            for k, v in special.items():
                q[kind == k] = v
            pts[b, :n], mask[b, :n] = q, sel
            mask[b, n:] = rng.random(C - n) < 0.3
            pts[b, n:] = np.nan
        out = {"predict": [(pts, mask)]}
        if t in two_calls:
            pts2 = (pts + np.float32(1.5)).astype(np.float32)
            mask2 = mask & (rng.random((B, C)) < 0.5) | (rng.random((B, C)) < 0.1)
            out["predict"].append((pts2, mask2))
        if drops:
            d = np.zeros((B, C), bool)
            for b, m in enumerate(models):
                d[b, :len(m.ids)] = rng.random(len(m.ids)) < 0.15
            out["drop"] = d
        return out

    return req


def restart_points(cv2, seqs, t, b, k):
    return cv2.goodFeaturesToTrack(seqs[b][t], **DET).reshape(-1, 2)[:k].astype(np.float32)


def with_restarts(cv2, seqs, req, restarts):
    """requests plus restarts {t: {b: k}}: sequence b restarts with the first k corners of frame t."""
    def f(t, models):
        out = req(t, models)
        if t in restarts:
            out["restart"] = {b: restart_points(cv2, seqs, t, b, k) for b, k in restarts[t].items()}
        return out
    return f


def test_idle_prior_is_a_no_op(klt, cv2):
    """motion_prior="given" with no predict() call, and with all-False masks, equals motion_prior=None bit for bit over
    ten frames, eagerly and replayed from the graphs."""
    import torch
    h, w = KITTI
    B, C = 3, 1200
    seqs = [S.sequence(h, w, 11, seed=610 + b) for b in range(B)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 200 + 300 * b] for b, s in enumerate(seqs)]
    objs = {(prior, g): make(seqs, init, C, 0, False, "given" if prior == "given-masked" else prior)
            for prior in (None, "given", "given-masked") for g in (0, 1)}
    for t in range(1, 11):
        for (prior, g), sb in objs.items():
            if prior == "given-masked":
                sb.predict(torch.full((B, C, 2), 3.0, device="cuda"), torch.zeros((B, C), dtype=torch.bool, device="cuda"))
            sb.step(frames_at(seqs, t))
            if t == 1 and g:
                sb.capture()
        ref = {k: getattr(objs[(None, 0)], k).cpu().numpy() for k in SNAP}
        for key, sb in objs.items():
            for k in SNAP:
                assert np.array_equal(getattr(sb, k).cpu().numpy().view(np.uint8), ref[k].view(np.uint8)), "frame %d %r: %s" % (t, key, k)
    for sb in objs.values():
        sb.check()


@pytest.mark.parametrize("setting", ["plain", "control"])
def test_given_positions_against_cv2_loop(klt, cv2, setting):
    """Five KITTI sequences (one empty, one whose capacity binds), C = 1200, ten steps; every step predicts a random half of
    the slots with positions of every kind and marks slots behind the count; steps 3 and 7 make a second predict() call.
    control: R = 4, random drops every step, and restarts of two sequences at different frames (one of them also
    predicted in the same step)."""
    h, w = KITTI
    B, C = 5, 1200
    motion = (1.1, -0.6, 0.15, 1.003)
    seqs = [S.sequence(h, w, 11, seed=640 + b, motion=motion) for b in range(B)]
    init = [np.zeros((0, 2), np.float32)]
    for b in range(1, B):
        init.append(cv2.goodFeaturesToTrack(seqs[b][0], **DET).reshape(-1, 2)[: (1200 if b == 2 else 250 * b)])
    ctl = setting == "control"
    req = given_requests(B, C, motion, seed=11, two_calls=(3, 7), drops=ctl)
    if ctl:
        req = with_restarts(cv2, seqs, req, {4: {3: 150}, 6: {0: 40}})
    models, _ = drive(cv2, seqs, init, C, 4 if ctl else 0, "given", req, control=ctl)
    assert len(models[2].ids) == C                                   # the capacity bound
    if ctl:
        assert models[3].f == 6 and models[0].f == 4


@pytest.mark.parametrize("R", [2, 5])
@pytest.mark.parametrize("motion", [(1.1, -0.6, 0.15, 1.003), (10.0, 1.5, 0.2, 1.0)], ids=["default", "10px"])
def test_velocity_against_cv2_loop(klt, cv2, R, motion):
    """Velocity prior, four KITTI sequences, C = 1500, nine steps (the ring of R = 2 wraps every step, R = 5 after five):
    new corners start at their position, restarts of two sequences at frames 3 and 5 (no velocity at their frame 0), and
    predict() overrides a tenth of the slots every other step."""
    h, w = KITTI
    B, C = 4, 1500
    seqs = [S.sequence(h, w, 10, seed=680 + b, motion=motion) for b in range(B)]
    init = [cv2.goodFeaturesToTrack(s[0], **DET).reshape(-1, 2)[: 300 * (b + 1)] for b, s in enumerate(seqs)]
    rng = np.random.default_rng(R)
    base = given_requests(B, C, motion, seed=20 + R, kinds=3)

    def req(t, models):
        out = base(t, models)
        pts, mask = out["predict"][0]
        if t % 2:
            mask &= rng.random((B, C)) < 0.2
        else:
            mask[:] = False
        return {"predict": [(pts, mask)]}

    models, _ = drive(cv2, seqs, init, C, R, "velocity", with_restarts(cv2, seqs, req, {3: {1: 200}, 5: {2: 0}}), control=True)
    assert [m.f for m in models] == [9, 6, 4, 9]


def test_velocity_follows_fast_motion(klt, cv2):
    """maxLevel 0, 21 x 21 window, fine texture, 6 px then 12 px per frame (the CPU tier's property case): the device
    loop equals the cv2 loop, and the velocity prior keeps more than twice as many tracks on the true motion as no prior."""
    h, w = KITTI
    seq = fine_sequence(cv2, h, w, FAST_STEPS, seed=5)
    init = [cv2.goodFeaturesToTrack(seq[0], **DET).reshape(-1, 2)]
    on_motion = {}
    for prior in (None, "velocity"):
        _models, kept = drive(cv2, [seq], init, 1500, 2 if prior else 0, prior, lambda t, m: {}, lk=FAST_LK, check_records=False)
        ref = host_loop(cv2, seq, init[0], 1500, FAST_LK, prior == "velocity")
        assert [len(k[0]) for k in kept] == [n for n, _o in ref]
        on_motion[prior] = [o for _n, o in ref]
        assert on_motion[prior] == FAST_ON_MOTION[prior]
    assert all(v > 2 * n for v, n in zip(on_motion["velocity"][1:], on_motion[None][1:]))


# ---- every LK instance of the step runs its forward pass from given starts ----------------------------------------------

SHAPES = [CASES[0], CASES[2], CASES[3],
          Case("31x31-4warps-two_pass", (31, 31), 3, 3, FAST % (31, 31, 4), 128, 1, True,
               lambda sms: (3, 1200), (None, 128), lambda C: [0, 600, C]),
          CASES[4], CASES[5]]


def shape_starts(seqs, t, pts_list, C, seed):
    """Given starts for step t of a shapes case: about half of every sequence's slots at the true next position plus up
    to 2 px, the rest left to the velocity prior."""
    h, w = KITTI
    rng = np.random.default_rng(seed + t)
    B = len(pts_list)
    pts = np.zeros((B, C, 2), np.float32)
    mask = np.zeros((B, C), bool)
    for b, p in enumerate(pts_list):
        n = len(p)
        pts[b, :n] = true_next(p, (1.1, -0.6, 0.15, 1.003), h, w) + rng.uniform(-2, 2, (n, 2)).astype(np.float32)
        mask[b, :n] = rng.random(n) < 0.5
    return pts, mask


def shape_batch(cv2, case, sms, i):
    B, C = case.shape(sms)
    lk = dict(winSize=case.win, maxLevel=case.max_level, criteria=(3, 30, 0.03))
    seqs, init = case_inputs(cv2, case, B, C, seed=700 + 10 * i)
    return B, C, lk, seqs, init


@pytest.fixture(scope="module")
def sms(klt):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def launches(klt, tmp_path_factory):
    """The LK launches of each shape's first step with given starts, profiled in a child process (this file run as a
    script; see test_gpu_frame_step_lk_shapes.py for why the test process never starts a CUPTI session)."""
    import subprocess
    import sys
    out = tmp_path_factory.mktemp("prior_launches")
    tests = os.path.dirname(os.path.abspath(__file__))
    path = [os.path.dirname(tests), tests] + ([os.environ["PYTHONPATH"]] if os.environ.get("PYTHONPATH") else [])
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, PYTHONPATH=os.pathsep.join(path)), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, "profiling child failed:\n" + r.stdout[-4000:] + r.stderr[-4000:]
    with open(out / "launches.json") as f:
        return {k: [(n, tuple(g), tuple(b)) for n, g, b in v] for k, v in json.load(f).items()}


@pytest.mark.parametrize("case", SHAPES, ids=[c.name for c in SHAPES])
def test_lk_instance_from_given_starts(klt, cv2, sms, launches, capsys, case):
    """The first step (profiled in the `launches` child) ran the case's LK instance on its grid, both passes; then three
    steps with the velocity prior (R = 2) and given starts on half the slots equal the cv2 loop, eagerly and replayed."""
    B, C, lk, seqs, init = shape_batch(cv2, case, sms, SHAPES.index(case))
    lo, hi = case.side
    assert (lo is None or B * C > lo * sms) and (hi is None or B * C <= hi * sms), (case.name, B, C, sms)
    check_launches(case, launches[case.name], B * C, capsys, "KLTSequenceBatch.step with start positions")
    seed = 900 + SHAPES.index(case)
    drive(cv2, seqs, init, C, 2, "velocity", lambda t, models: {"predict": [shape_starts(seqs, t, [m.pts for m in models], C, seed)]},
          lk=lk, check_records=False)


def test_errors(klt):
    import torch
    from visual_odom_pipeline_b200 import _lib
    from visual_odom_pipeline_b200 import tracker as T
    from visual_odom_pipeline_b200.lk import error
    h, w = 64, 96
    frames = torch.from_numpy(np.stack([S.sequence(h, w, 2, seed=90 + b)[1] for b in range(3)])).cuda()
    pts = torch.full((3, 8, 2), 20.0, device="cuda")
    cnt = torch.tensor([8, 0, 3], dtype=torch.int32, device="cuda")
    C = 16
    for kw in (dict(motion_prior="velocity"), dict(motion_prior="velocity", history=1), dict(motion_prior="nearest"),
               dict(motion_prior=True)):
        with pytest.raises(error):
            T.KLTSequenceBatch(frames, pts, cnt, C, **kw)
    plain = T.KLTSequenceBatch(frames, pts, cnt, C, history=2)
    good_p, good_m = torch.zeros((3, C, 2), device="cuda"), torch.zeros((3, C), dtype=torch.bool, device="cuda")
    with pytest.raises(error):
        plain.predict(good_p, good_m)
    sb = T.KLTSequenceBatch(frames, pts, cnt, C, history=2, motion_prior="velocity")
    for p, m in ((good_p[:, :8], good_m), (good_p.double(), good_m), (good_p.cpu(), good_m), (good_p[:2], good_m),
                 (good_p, good_m[:, :8]), (good_p, good_m.to(torch.uint8)), (good_p, good_m.cpu()), (good_p[..., :1], good_m)):
        with pytest.raises(error):
            sb.predict(p, m)
    sb.predict(good_p, good_m).step(frames).check()

    # the entry points' own argument checks, with a real context and buffers
    L = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    inval = _lib.KLT_ERR_INVALID_ARG
    good = [sb.ctx.handle, 3, C, sb._pts[0].data_ptr(), sb._counts[0].data_ptr(), sb._guess_pts.data_ptr(), sb._guess_mask.data_ptr(),
            2, sb._ring_pts.data_ptr(), sb._ring_src.data_ptr(), sb._ring_counts.data_ptr(), sb._frame.data_ptr(), sb._init.data_ptr(), st]
    assert L.klt_track_predict(*good) == _lib.KLT_OK
    for i, v in [(1, 0), (2, -1), (3, None), (4, None), (5, None), (6, None), (7, -1), (7, 1), (8, None), (9, None), (10, None),
                 (11, None), (12, None)]:
        a = list(good)
        a[i] = v
        assert L.klt_track_predict(*a) == inval, (i, v)
    a = list(good)
    a[5] = a[6] = None
    a[7] = 0
    a[8:12] = [None] * 4
    assert L.klt_track_predict(*a) == _lib.KLT_OK                    # no given positions, no velocity
    a[2] = 0
    a[3] = a[12] = None
    assert L.klt_track_predict(*a) == _lib.KLT_OK                    # nothing to do
    cur, nxt = sb._cur, 1 - sb._cur
    prev, new = sb._slots[cur], sb._slots[nxt]
    step = [sb.ctx.handle, prev.images.data_ptr(), prev.buffer.data_ptr(), new.images.data_ptr(), new.buffer.data_ptr(),
            prev.layout, 0, 0, 1, 3, sb._pts[cur].data_ptr(), sb._counts[cur].data_ptr(), C, sb.params, sb.max_bidir_error,
            sb.mask_radius, sb.maxCorners, sb.qualityLevel, sb.minDistance, sb.blockSize, sb._pts[nxt].data_ptr(), C,
            sb._keep.data_ptr(), sb._counts[nxt].data_ptr(), sb._n_new.data_ptr(), sb._ids[cur].data_ptr(), sb._ids[nxt].data_ptr(),
            sb._next_id.data_ptr(), sb._flags.data_ptr(), sb._ws_ptr, sb._ws_bytes]
    assert L.klt_frame_step_batch_init_async(*step, None, None, st) == inval            # no start positions
    flagged = _lib.klt_lk_params.from_buffer_copy(sb.params)
    flagged.flags |= 4                                                                  # KLT_OPTFLOW_USE_INITIAL_FLOW
    s2 = list(step)
    s2[13] = flagged
    assert L.klt_frame_step_batch_init_async(*s2, sb._init.data_ptr(), None, st) == inval
    assert L.klt_frame_step_batch_async(*s2, st) == inval                               # still refused there
    torch.cuda.synchronize()


if __name__ == "__main__":
    # the child process of the `launches` fixture: python tests/test_gpu_motion_prior.py OUT_DIR
    import sys
    import cv2 as cv2_
    import torch
    sms_ = torch.cuda.get_device_properties(0).multi_processor_count
    res = {}
    for i, case in enumerate(SHAPES):
        B, C, lk, seqs, init = shape_batch(cv2_, case, sms_, i)
        sb = make(seqs, init, C, 2, False, "velocity", lk)
        p, m = shape_starts(seqs, 1, [np.asarray(x, np.float32).reshape(-1, 2) for x in init], C, 900 + i)
        sb.predict(torch.from_numpy(p).cuda(), torch.from_numpy(m).cuda())
        frames = frames_at(seqs, 1)
        res[case.name] = lk_launches(torch, lambda: sb.step(frames), os.path.join(sys.argv[1], "%d.json" % i))
    with open(os.path.join(sys.argv[1], "launches.json"), "w") as f:
        json.dump(res, f)
