"""GPU tier (pytest -m gpu, B200) of grid detection in KLTSequenceBatch (detect_grid=(cols, rows), tracks_per_cell=q) and
of the batched grid detector.

Bar: every sequence and frame against the capped cv2 loop plus the host rule of tests/test_grid_detect_cpu.py: keep,
survivors and new corners (as uint32) in row order, counts, n_new, ids, and with history the records.  An eager object
and a graph-replayed twin (captured after the first step) are both checked.  detect_grid=(1, 1) with q = C equals the
step without the option, ids and records included.  With the option off the step launches what it launched before."""
import json
import os
import re

import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from test_gpu_frame_step_async import DET, KITTI, LK, pad
from test_gpu_motion_prior import with_restarts
from test_gpu_sequence_control import Model, check_state
from test_gpu_thin import host_track, same_d
from test_gpu_track_history import Records, frames_at
from test_grid_detect_cpu import edges, grid_detect, step_mask
from test_motion_prior_cpu import detect, velocity_starts
from test_thin_cpu import SHRINK, thin

pytestmark = pytest.mark.gpu

SNAP = ("points", "counts", "ids", "keep", "n_new")


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def make(seqs, init, cap, grid, q, history=0, control=False, motion_prior=None, second_pass="reference", max_err=30.0, dist=None,
         det=DET):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init, n=cap)
    return T.KLTSequenceBatch(frames_at(seqs, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), cap,
                              history=history, control=control, motion_prior=motion_prior, second_pass=second_pass,
                              max_bidir_error=max_err, min_track_distance=dist, detect_grid=grid, tracks_per_cell=q, **LK, **det)


def drive(cv2, seqs, init, C, grid, q, R=0, prior=None, requests=lambda t, m: {}, second_pass="reference", max_err=30.0,
          control=False, dist=None, det=DET):
    """An eager object and a graph-replayed twin against the host loop every frame -> (models, new corners per step)."""
    import torch
    B, T_ = len(seqs), len(seqs[0])
    reverse = second_pass == "reverse"
    objs = [make(seqs, init, C, grid, q, R, control, prior, second_pass, max_err, dist, det) for _ in range(2)]
    models = [Model(np.asarray(p, np.float32).reshape(-1, 2)) for p in init]
    news = []

    def det_fn(im, surv):
        if grid is None:
            return detect(cv2, im, surv, C)
        return grid_detect(cv2, im, surv, C, grid, q, det=det)
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
        news.append([])
        for b, m in enumerate(models):
            n = len(m.ids)
            d_ref = None
            if b in req.get("restart", {}):
                p = req["restart"][b]
                keep_ref = np.zeros(n, bool)
                surv = p
                new = det_fn(seqs[b][t], surv)
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
                if dist is not None:
                    keep_ref = keep_ref & ~thin(p1, keep_ref, dist)
                surv = p1[keep_ref]
                new = det_fn(seqs[b][t], surv)
                m.ids = np.concatenate([m.ids[keep_ref], np.arange(m.next_id, m.next_id + len(new), dtype=np.int32)])
                m.next_id += len(new)
                m.pts = np.concatenate([surv, new]).astype(np.float32)
                m.f += 1
                if R:
                    m.recs.step(m.f, m.ids, m.pts)
            news[-1].append(new)
            for name, g in zip(("eager", "graph"), snaps):
                tag = "%s frame %d sequence %d" % (name, t, b)
                assert np.array_equal(g["keep"][b, :n], keep_ref) and not g["keep"][b, n:].any(), tag + ": keep"
                if reverse and d_ref is not None:
                    assert same_d(g["bidir_error"][b, :n], d_ref), tag + ": bidir_error"
                assert int(g["n_new"][b]) == len(new), tag + ": n_new %d, want %d" % (int(g["n_new"][b]), len(new))
                assert int(g["counts"][b]) == len(m.ids), tag + ": counts"
                assert np.array_equal(g["points"][b, :len(m.ids)].view(np.uint32), m.pts.view(np.uint32)), tag + ": points"
                assert np.array_equal(g["ids"][b, :len(m.ids)], m.ids), tag + ": ids"
        if R:
            for sb, name in zip(objs, ("eager", "graph")):
                check_state(sb, models, C, R, "%s frame %d" % (name, t))
    assert objs[1]._graphs is not None
    return models, news


def uneven(B, seed, frames, gain=0.1, shape=KITTI):
    return [S.uneven_sequence(*shape, frames, seed=seed + b, left_gain=gain) for b in range(B)]


def initial(cv2, seqs, counts):
    return [cv2.goodFeaturesToTrack(s[0], **dict(DET, maxCorners=max(n, 1))).reshape(-1, 2)[:n] for s, n in zip(seqs, counts)]


@pytest.mark.parametrize("grid,q", [((8, 4), 64), ((4, 3), 100), ((7, 5), 40)])
def test_a_uneven_contrast(klt, cv2, grid, q):
    """Low-contrast left third, three sequences (one empty); the 1000-corner cap binds on the empty one's first frame."""
    seqs = uneven(3, 2000, 4)
    init = initial(cv2, seqs, [0, 300, 900])
    _models, news = drive(cv2, seqs, init, 3000, grid, q)
    cols, rows = grid
    left = edges(cols, KITTI[1])[cols // 3]
    assert any((n[:, 0] < left).any() for step in news for n in step)


def test_b_identity_against_the_off_arm(klt, cv2):
    """detect_grid=(1, 1), q = C: the same rows, ids and records as the step without the option, every frame."""
    import torch
    seqs = [S.sequence(*KITTI, 5, seed=2100 + b) for b in range(3)]
    init = initial(cv2, seqs, [500, 0, 1500])
    C = 2200
    objs = [make(seqs, init, C, None, None, history=3), make(seqs, init, C, (1, 1), C, history=3)]
    for t in range(1, 5):
        for sb in objs:
            sb.step(frames_at(seqs, t))
        if t == 1:
            objs[1].capture()
        a, b = ({k: getattr(sb, k).cpu().numpy() for k in SNAP + ("first_points", "first_frames")} for sb in objs)
        for k in a:
            assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), (t, k)
        ha, hb = objs[0].history(), objs[1].history()
        for x, y in zip(ha, hb):
            assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), t
    torch.cuda.synchronize()


def test_c_identity_against_the_host_loop(klt, cv2):
    """(1, 1) with q = C against the global host loop, the capacity binding (C = 1400)."""
    seqs = [S.sequence(*KITTI, 4, seed=2120 + b) for b in range(2)]
    init = initial(cv2, seqs, [900, 1300])
    drive(cv2, seqs, init, 1400, None, None)
    drive(cv2, seqs, init, 1400, (1, 1), 1400)


def test_d_flat_band_and_caps(klt, cv2):
    """A flat band (cells with no candidate), odd grid (7, 5) off the 32-px tiles; capacity binding (C = 700) and a
    small maxCorners (150) binding on the interleave."""
    h, w = KITTI
    seqs = []
    for b in range(2):
        s = S.sequence(h, w, 4, seed=2140 + b)
        for f in s:
            f[:, 300:620] = 128
        seqs.append(s)
    init = initial(cv2, seqs, [200, 500])
    drive(cv2, seqs, init, 700, (7, 5), 30)
    drive(cv2, seqs, init, 3000, (7, 5), 30, det=dict(DET, maxCorners=150))


def test_e_large_cell_radix_path(klt, cv2):
    """(1, 1) and (2, 1) at qualityLevel 0.001 on KITTI frames: cells with more than 4096 candidates (the radix sort)."""
    seqs = [S.sequence(*KITTI, 3, seed=2160)]
    init = [np.zeros((0, 2), np.float32)]
    det = dict(DET, qualityLevel=0.001, minDistance=3)
    im = seqs[0][1]
    eig = cv2.cornerMinEigenVal(im, 31, ksize=3)
    assert (eig > eig.max() * 0.001).sum() > 20000
    drive(cv2, seqs, init, 3000, (2, 1), 900, det=det)
    drive(cv2, seqs, init, 3000, (1, 1), 3000, det=det)


def test_f_control_priors_reverse_thinning(klt, cv2):
    """history=2, control with drops and restarts (staged points with NaN and outside the image), motion_prior
    velocity, second_pass="reverse" at max error 1 and min_track_distance 10, on the uneven sequence, grid (8, 4)."""
    B, C = 3, 2500
    seqs = uneven(B, 2180, 6)
    init = initial(cv2, seqs, [400, 800, 1200])
    rng = np.random.default_rng(5)
    h, w = KITTI

    def req(t, models):
        d = np.zeros((B, C), bool)
        for b, m in enumerate(models):
            d[b, :len(m.ids)] = rng.random(len(m.ids)) < 0.1
        out = {"drop": d}
        if t == 5:   # the last step: NaN rows are never tracked
            p = np.float32([[np.nan, 5.0], [-20.0, 40.0], [w + 30.0, 10.0], [w, h], [50.5, np.nan], [100.0, 100.0], [0.0, 0.0]])
            out["restart"] = {2: p}
        return out
    drive(cv2, seqs, init, C, (8, 4), 48, R=2, prior="velocity", requests=req, second_pass="reverse", max_err=1.0, control=True,
          dist=10.0)


def test_g_given_prior_and_restart_helper(klt, cv2):
    """motion_prior="given" (nothing predicted: the start is the point) and with_restarts of the motion-prior tier."""
    seqs = uneven(2, 2200, 5, gain=0.3)
    init = initial(cv2, seqs, [700, 300])
    drive(cv2, seqs, init, 2000, (4, 3), 80, R=1, prior="given", control=True,
          requests=with_restarts(cv2, seqs, lambda t, m: {}, {2: {0: 120}}))


def test_h_small_odd_size(klt, cv2):
    """97 x 61 frames, grids (5, 3) (cells 19-20 px wide) and (32, 32) (the largest grid: cells 3-4 x 1-2 px)."""
    seqs = [S.sequence(61, 97, 4, seed=2220 + b, motion=(0.7, -0.3, 0.5, 1.004)) for b in range(3)]
    init = initial(cv2, seqs, [10, 0, 25])
    det = dict(DET, blockSize=7, minDistance=4)
    drive(cv2, seqs, init, 120, (5, 3), 6, det=det)
    drive(cv2, seqs, init, 120, (32, 32), 1, det=dict(det, maxCorners=40))   # KLT_MAX_GRID_CELLS cells


def test_i_standalone_detector(klt, cv2):
    """detector.good_features_to_track_grid against cv2 per cell, with and without a mask, on two grids."""
    import torch
    from visual_odom_pipeline_b200 import detector as D
    from test_grid_detect_cpu import cell_lists
    frames = [S.uneven_sequence(*KITTI, 1, seed=2240 + b, left_gain=g)[0] for b, g in enumerate((0.1, 1.0, 0.3))]
    img = torch.from_numpy(np.stack(frames)).cuda()
    masks = [step_mask(f, cv2.goodFeaturesToTrack(f, **dict(DET, maxCorners=300)).reshape(-1, 2)) for f in frames]
    for grid, q, use_mask in (((8, 4), 32, False), ((7, 5), 20, True), ((1, 1), 900, True)):
        kw = dict(qualityLevel=0.03, minDistance=10, blockSize=31)
        m = torch.from_numpy(np.stack(masks)).cuda() if use_mask else None
        corners, counts = D.good_features_to_track_grid(img, grid, q, mask=m, **kw)
        corners, counts = corners.cpu().numpy(), counts.cpu().numpy()
        for b, f in enumerate(frames):
            mk = masks[b] if use_mask else np.full_like(f, 255)
            want = cell_lists(cv2, f, mk, grid, [q] * (grid[0] * grid[1]), det=dict(DET, **kw))
            for k, L in enumerate(want):
                assert counts[b, k] == len(L), (grid, b, k)
                assert np.array_equal(corners[b, k, :len(L)].view(np.uint32), L.view(np.uint32)), (grid, b, k)


def test_j_contracting_tracks_per_cell(klt, cv2):
    """Contracting sequence with thinning and a (6, 4) grid: survivors fill cells beyond q, those get no quota."""
    seqs = [S.sequence(*KITTI, 5, seed=2260 + b, motion=SHRINK) for b in range(2)]
    init = initial(cv2, seqs, [1500, 600])
    _models, news = drive(cv2, seqs, init, 4096, (6, 4), 50, dist=8.0)
    assert all(len(n) < 1000 for n in news[-1])


# ---- launches ---------------------------------------------------------------------------------------------------------------

def all_launches(torch, fn, trace):
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


# the detection launches of one step with the option off, in order: the kernels of the step before grid detection existed
OFF_DETECTION = ["mask_fill_kernel", "mask_from_points_kernel", "cov_kernel", "row_scan_kernel", "col_scan_kernel", "candidates_kernel",
                 "rank_keys_kernel", "scatter_keys_kernel", "radix_sort_keys_kernel", "select_corners_kernel"]
ON_DETECTION = ["mask_fill_kernel", "mask_from_points_kernel", "cov_kernel", "row_scan_kernel", "col_scan_kernel", "cell_quota_kernel",
                "cell_threshold_kernel", "cell_candidates_kernel", "cell_rank_sort_kernel", "cell_radix_sort_kernel", "cell_select_kernel",
                "cell_interleave_kernel"]


@pytest.fixture(scope="module")
def launches(klt, tmp_path_factory):
    """One eager step with the option off and on, profiled in a child process (this file run as a script; see
    test_gpu_frame_step_lk_shapes.py for why the test process never starts a CUPTI session)."""
    import subprocess
    import sys
    out = tmp_path_factory.mktemp("grid_launches")
    tests = os.path.dirname(os.path.abspath(__file__))
    path = [os.path.dirname(tests), tests] + ([os.environ["PYTHONPATH"]] if os.environ.get("PYTHONPATH") else [])
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, PYTHONPATH=os.pathsep.join(path)), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, "profiling child failed:\n" + r.stdout[-4000:] + r.stderr[-4000:]
    with open(out / "launches.json") as f:
        return json.load(f)


def short(name):
    return re.sub(r"<.*$", "", name.split("::")[-1])


def test_k_launches(klt, launches):
    """Off: the step's detection kernels as before the option existed, and the same list as an object built without
    the arguments.  On: the tracking launches unchanged, the detection tail replaced by the grid kernels."""
    off, plain, on = launches["off"], launches["plain"], launches["on"]
    assert off == plain
    i = [short(n) for n, _g, _b in off].index("mask_fill_kernel")
    assert [short(n) for n, _g, _b in off[i:]] == OFF_DETECTION, off[i:]
    assert on[:i] == off[:i]
    assert [short(n) for n, _g, _b in on[i:]] == ON_DETECTION, on[i:]


if __name__ == "__main__":
    # the child process of the `launches` fixture: python tests/test_gpu_grid_detect.py OUT_DIR
    import sys
    import cv2 as cv2_
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    seqs_ = uneven(3, 2280, 3)
    init_ = initial(cv2_, seqs_, [500, 0, 1500])
    res = {}
    for arm, grid_, q_ in (("off", None, None), ("on", (8, 4), 64), ("plain", "plain", None)):
        if grid_ == "plain":
            padded, cnt = pad(init_, n=2048)
            sb = T.KLTSequenceBatch(frames_at(seqs_, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), 2048, **LK, **DET)
        else:
            sb = make(seqs_, init_, 2048, grid_, q_)
        sb.step(frames_at(seqs_, 1))
        f2 = frames_at(seqs_, 2)
        res[arm] = all_launches(torch, lambda: sb.step(f2), os.path.join(sys.argv[1], "%s.json" % arm))
    with open(os.path.join(sys.argv[1], "launches.json"), "w") as f:
        json.dump(res, f)
