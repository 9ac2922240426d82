"""GPU tier (pytest -m gpu, B200) of the minimum track distance of KLTSequenceBatch (min_track_distance=d): the
compaction of the frame step ends a survivor that lies closer than d to an earlier kept one, in slot order.

Bar: every sequence and frame against the capped cv2 loop plus the host thinning of tests/test_thin_cpu.py: keep,
thinned, survivors and new corners (as uint32), ids, counts, n_new, and bidir_error with second_pass="reverse"; with
history the records (thinned tracks end, and no window reaches past their end).  An eager object and a graph-replayed
twin (captured after the first step) are both checked.  With the option off the step launches what it launched before;
with it on it launches the same kernels, grids and blocks, one compaction instance swapped for the thinning one."""
import json
import os
import re

import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from test_fb_check_cpu import fb_keep_from, same_direction_keep
from test_gpu_frame_step_async import DET, KITTI, LK, pad
from test_gpu_motion_prior import with_restarts
from test_gpu_sequence_control import Model, check_state
from test_gpu_track_history import Records, frames_at
from test_motion_prior_cpu import detect, lk_keep_from, velocity_starts
from test_thin_cpu import SHRINK, thin

pytestmark = pytest.mark.gpu

SNAP = ("points", "counts", "ids", "keep", "n_new", "thinned")


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def make(seqs, init, cap, dist, history=0, control=False, motion_prior=None, second_pass="reference", max_err=30.0):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init, n=cap)
    return T.KLTSequenceBatch(frames_at(seqs, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), cap,
                              history=history, control=control, motion_prior=motion_prior, second_pass=second_pass,
                              max_bidir_error=max_err, min_track_distance=dist, **LK, **DET)


def host_track(cv2, im0, im1, pts, starts, reverse, max_err):
    """The tracking half of the step -> keep (n,) bool, p1 (n, 2), d (n,) float32 (None for the reference's pass)."""
    if not len(pts):
        return np.zeros(0, bool), np.zeros((0, 2), np.float32), np.zeros(0, np.float32)
    if reverse:
        return fb_keep_from(cv2, LK, im0, im1, pts, starts, max_bidir=max_err)
    if starts is None:
        keep, p1 = same_direction_keep(cv2, LK, im0, im1, pts, max_bidir=max_err)
    else:
        keep, p1 = lk_keep_from(cv2, LK, im0, im1, pts, starts, max_bidir=max_err)
    return keep, p1, None


def same_d(got, want):
    nan = np.isnan(want)
    return np.array_equal(np.isnan(got), nan) and np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def drive(cv2, seqs, init, C, dist, R=0, prior=None, requests=lambda t, m: {}, second_pass="reference", max_err=30.0,
          control=False):
    """Both objects against the host loop every frame -> (models, per step and sequence the thinned mask, per step and
    sequence the ids of the tracks thinned)."""
    import torch
    B, T_ = len(seqs), len(seqs[0])
    reverse = second_pass == "reverse"
    objs = [make(seqs, init, C, dist, R, control, prior, second_pass, max_err) for _ in range(2)]
    models = [Model(np.asarray(p, np.float32).reshape(-1, 2)) for p in init]
    thinned, ended = [], []
    for t in range(1, T_):
        req = requests(t, models)
        for sb in objs:
            if req.get("drop") is not None:
                sb.drop(torch.from_numpy(req["drop"]).cuda())
            for b, p in req.get("restart", {}).items():
                m = np.zeros(B, bool)
                m[b] = True
                pt = torch.full((B, len(p), 2), -1.0, device="cuda")
                pt[b] = torch.from_numpy(p).cuda()
                sb.restart(torch.from_numpy(m).cuda(), pt)
        for sb in objs:
            sb.step(frames_at(seqs, t))
        if t == 1:
            objs[1].capture()
        snaps = []
        for sb in objs:
            s = {k: getattr(sb, k).cpu().numpy() for k in SNAP}
            if reverse:
                s["bidir_error"] = sb.bidir_error.cpu().numpy()
            snaps.append(s)
            sb.check()
        drop = req.get("drop")
        thinned.append([])
        ended.append([])
        for b, m in enumerate(models):
            n = len(m.ids)
            if b in req.get("restart", {}):
                p = req["restart"][b]
                keep_ref, th_ref = np.zeros(n, bool), np.zeros(n, bool)
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
                if prior == "velocity":
                    prev = np.array([m.recs.pos[int(i)].get(m.f - 1, (np.nan, np.nan)) for i in m.ids], np.float32).reshape(-1, 2)
                    starts = velocity_starts(m.pts, prev)
                keep_ref, p1, d_ref = host_track(cv2, seqs[b][t - 1], seqs[b][t], m.pts, starts, reverse, max_err)
                if drop is not None:
                    keep_ref = keep_ref & ~drop[b, :n]
                th_ref = thin(p1, keep_ref, dist)
                keep_ref = keep_ref & ~th_ref
                ended[-1].append(set(int(i) for i in m.ids[th_ref]))
                surv = p1[keep_ref]
                new = detect(cv2, seqs[b][t], surv, C)
                m.ids = np.concatenate([m.ids[keep_ref], np.arange(m.next_id, m.next_id + len(new), dtype=np.int32)])
                m.next_id += len(new)
                m.pts = np.concatenate([surv, new]).astype(np.float32)
                m.f += 1
                if R:
                    m.recs.step(m.f, m.ids, m.pts)
            if len(ended[-1]) <= b:
                ended[-1].append(set())
            thinned[-1].append(th_ref)
            for name, g in zip(("eager", "graph"), snaps):
                tag = "%s frame %d sequence %d" % (name, t, b)
                assert np.array_equal(g["thinned"][b, :n].astype(bool), th_ref) and not g["thinned"][b, n:].any(), \
                    tag + ": thinned (%d differ)" % int((g["thinned"][b, :n].astype(bool) != th_ref).sum())
                assert np.array_equal(g["keep"][b, :n], keep_ref) and not g["keep"][b, n:].any(), tag + ": keep"
                if reverse:
                    assert same_d(g["bidir_error"][b, :n], d_ref), tag + ": bidir_error"
                assert int(g["n_new"][b]) == len(new), tag + ": n_new"
                assert int(g["counts"][b]) == len(m.ids), tag + ": counts"
                assert np.array_equal(g["points"][b, :len(m.ids)].view(np.uint32), m.pts.view(np.uint32)), tag + ": points"
                assert np.array_equal(g["ids"][b, :len(m.ids)], m.ids), tag + ": ids"
        if R:
            for sb, name in zip(objs, ("eager", "graph")):
                check_state(sb, models, C, R, "%s frame %d" % (name, t))
    assert objs[1]._graphs is not None
    return models, thinned, ended


def shrink_inputs(cv2, B, seed, frames, counts, shape=KITTI):
    h, w = shape
    seqs = [S.sequence(h, w, frames, seed=seed + b, motion=SHRINK) for b in range(B)]
    init = [cv2.goodFeaturesToTrack(s[0], **dict(DET, maxCorners=max(n, 1))).reshape(-1, 2)[:n] for s, n in zip(seqs, counts)]
    return seqs, init


def total_thinned(thinned):
    return sum(int(m.sum()) for step in thinned for m in step)


def test_a_contracting_sequences(klt, cv2):
    """Scale 0.99 per frame, four sequences (one empty) with different initial counts, d = 10, C = 3000."""
    seqs, init = shrink_inputs(cv2, 4, seed=1500, frames=8, counts=[0, 600, 1400, 2000])
    _models, thinned, _ended = drive(cv2, seqs, init, 3000, 10.0)
    assert total_thinned(thinned) >= 300, total_thinned(thinned)
    assert len(thinned[0][0]) == 0                     # the empty sequence has no slot in the first step


def test_b_records_control_velocity_reverse(klt, cv2):
    """history=2, control with drops every step and a restart, motion_prior="velocity", second_pass="reverse" at max
    error 1: thinned tracks end in the records, and no later row or window holds their ids."""
    B, C = 3, 2500
    seqs, init = shrink_inputs(cv2, B, seed=1520, frames=7, counts=[900, 1500, 2000])
    rng = np.random.default_rng(11)

    def req(t, models):
        d = np.zeros((B, C), bool)
        for b, m in enumerate(models):
            d[b, :len(m.ids)] = rng.random(len(m.ids)) < 0.1
        return {"drop": d}

    models, thinned, ended = drive(cv2, seqs, init, C, 10.0, R=2, prior="velocity",
                                   requests=with_restarts(cv2, seqs, req, {3: {1: 150}}), second_pass="reverse", max_err=1.0,
                                   control=True)
    assert total_thinned(thinned) >= 100, total_thinned(thinned)
    gone = [set() for _ in range(B)]
    for step in ended:
        for b in range(B):
            gone[b] |= step[b]
    for b, m in enumerate(models):
        assert not (gone[b] & set(int(i) for i in m.ids)), b


def test_c_duplicated_initial_rows(klt, cv2):
    """Every initial point two and three times at d = 0.5: every later copy that passes the filter is thinned at the first
    step, and no first copy is."""
    seqs, init = shrink_inputs(cv2, 2, seed=1540, frames=4, counts=[400, 700])
    rows, first = [], []
    for p in init:
        reps = np.where(np.arange(len(p)) % 2 == 0, 2, 3)
        rows.append(np.repeat(p, reps, axis=0))
        first.append(np.concatenate([[True] + [False] * (r - 1) for r in reps]))
    _models, thinned, _ended = drive(cv2, seqs, rows, 2400, 0.5)
    for b, (row, f) in enumerate(zip(rows, first)):
        keep, _p1 = same_direction_keep(cv2, LK, seqs[b][0], seqs[b][1], row)
        assert np.array_equal(thinned[0][b], keep & ~f), b
        assert thinned[0][b].sum() >= len(init[b])


def test_d_conflicts_across_chunks(klt, cv2):
    """d = 60 with 2300 and 1800 initial points (chunks of 1024 slots), C = 2333 (not a multiple of 32)."""
    seqs, init = shrink_inputs(cv2, 2, seed=1560, frames=4, counts=[2300, 1800])
    assert min(len(p) for p in init) > 1024
    _models, thinned, _ended = drive(cv2, seqs, init, 2333, 60.0)
    assert all(thinned[0][b][1024:].any() for b in range(2))


def test_e_tracks_at_the_border(klt, cv2):
    """Points along all four borders, 6 px apart, corners of the image included, at d = 10."""
    h, w = KITTI
    xs = np.arange(0.0, w + 0.5, 6.0, dtype=np.float32)
    ys = np.arange(0.0, h + 0.5, 6.0, dtype=np.float32)
    edge = np.concatenate([np.stack([xs, np.zeros_like(xs)], 1), np.stack([xs, np.full_like(xs, h - 0.5)], 1),
                           np.stack([np.zeros_like(ys), ys], 1), np.stack([np.full_like(ys, w - 0.25), ys], 1),
                           np.float32([[0, 0], [w, h], [w, 0], [0, h], [3.0, 2.0]])]).astype(np.float32)
    seqs = [S.sequence(h, w, 4, seed=1580 + b, motion=(0.2, 0.1, 0.0, 1.0)) for b in range(2)]
    init = [edge, edge[::-1].copy()]
    _models, thinned, _ended = drive(cv2, seqs, init, 1800, 10.0)
    assert all(thinned[0][b].sum() >= 50 for b in range(2))


def test_f_4k_frames(klt, cv2):
    """Two 3840 x 2160 contracting sequences, d = 10."""
    seqs, init = shrink_inputs(cv2, 2, seed=1600, frames=3, counts=[2000, 1200], shape=(2160, 3840))
    _models, thinned, _ended = drive(cv2, seqs, init, 4000, 10.0)
    assert total_thinned(thinned) > 0


# ---- launches ---------------------------------------------------------------------------------------------------------------

CONFIGS = {"plain": {}, "everything": dict(history=2, control=True, motion_prior="velocity", second_pass="reverse", max_err=1.0)}


def all_launches(torch, fn, trace):
    """Runs fn under torch.profiler -> [(kernel name with template arguments, grid, block)] of every kernel, in order."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(trace))
    with open(trace) as f:
        events = json.load(f)["traceEvents"]
    out = []
    for e in sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"]):
        name = re.sub(r"\(.*$", "", e["name"].replace("(anonymous namespace)", "anon")).replace(" ", "")
        out.append((name, list(e["args"]["grid"]), list(e["args"]["block"])))
    return out


@pytest.fixture(scope="module")
def launches(klt, tmp_path_factory):
    """The launches of one eager step per configuration, with the option off and on, profiled in a child process (this
    file run as a script; see test_gpu_frame_step_lk_shapes.py for why the test process never starts a CUPTI session)."""
    import subprocess
    import sys
    out = tmp_path_factory.mktemp("thin_launches")
    tests = os.path.dirname(os.path.abspath(__file__))
    path = [os.path.dirname(tests), tests] + ([os.environ["PYTHONPATH"]] if os.environ.get("PYTHONPATH") else [])
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, PYTHONPATH=os.pathsep.join(path)), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, "profiling child failed:\n" + r.stdout[-4000:] + r.stderr[-4000:]
    with open(out / "launches.json") as f:
        return json.load(f)


@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_g_launches(klt, launches, config):
    """Off: the step's kernels with the compaction instance it used before the option existed.  On: the same kernels,
    grids and blocks in the same order, that compaction swapped for the thinning instance; no launch is added."""
    off, on = launches[config]["off"], launches[config]["on"]
    want_off = "track_compact_kernel<true,false,false,false>" if config == "plain" else "track_compact_kernel<true,true,true,false>"
    compact = [i for i, (n, _g, _b) in enumerate(off) if "track_compact_kernel" in n]
    assert len(compact) == 1 and off[compact[0]][0].endswith(want_off), off
    assert len(on) == len(off)
    for i, (a, b) in enumerate(zip(off, on)):
        if i == compact[0]:
            assert b[0].endswith("track_compact_kernel<true,true,true,true>") and a[1:] == b[1:], (a, b)
        else:
            assert a == b, (i, a, b)


def test_h_errors(klt):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    from visual_odom_pipeline_b200.lk import error
    h, w = 64, 96
    frames = torch.from_numpy(np.stack([S.sequence(h, w, 2, seed=90 + b)[1] for b in range(3)])).cuda()
    pts = torch.full((3, 8, 2), 20.0, device="cuda")
    cnt = torch.tensor([8, 0, 3], dtype=torch.int32, device="cuda")
    for bad in (float("nan"), float("inf"), 0.0, -1.0, 1e6, "3", True):
        with pytest.raises(error):
            T.KLTSequenceBatch(frames, pts, cnt, 16, min_track_distance=bad)
    plain = T.KLTSequenceBatch(frames, pts, cnt, 16)
    with pytest.raises(error):
        plain.thinned
    sb = T.KLTSequenceBatch(frames, pts, cnt, 16, min_track_distance=5.0)
    assert sb.thinned.shape == (3, 16) and sb.thinned.dtype == torch.uint8 and not sb.thinned.any()
    sb.step(frames).check()
    th, keep = sb.thinned.cpu().numpy(), sb.keep.cpu().numpy()
    # eight and three copies of one point: the first is kept when the copies survive, the others thinned
    for b, n in ((0, 8), (2, 3)):
        assert keep[b].sum() <= 1 and not th[b, 0] and bool(th[b, 1:n].all()) == bool(keep[b, 0]) and not th[b, n:].any(), b
    assert not th[1].any()


if __name__ == "__main__":
    # the child process of the `launches` fixture: python tests/test_gpu_thin.py OUT_DIR
    import sys
    import cv2 as cv2_
    import torch
    seqs_, init_ = shrink_inputs(cv2_, 3, seed=1620, frames=3, counts=[500, 0, 1500])
    res = {}
    for cname, kw in sorted(CONFIGS.items()):
        res[cname] = {}
        for arm, dist in (("off", None), ("on", 10.0)):
            sb = make(seqs_, init_, 2048, dist, **kw)
            sb.step(frames_at(seqs_, 1))
            f2 = frames_at(seqs_, 2)
            res[cname][arm] = all_launches(torch, lambda: sb.step(f2), os.path.join(sys.argv[1], "%s_%s.json" % (cname, arm)))
    with open(os.path.join(sys.argv[1], "launches.json"), "w") as f:
        json.dump(res, f)
