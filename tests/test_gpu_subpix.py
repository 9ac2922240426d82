"""GPU tier (pytest -m gpu, B200) of sub-pixel corner refinement: the cornerSubPix drop-in, the batched device entry point
and KLTSequenceBatch(subpix=...).

Bar: bit for bit against cv2.cornerSubPix with cv2.ipp.setUseIPP(False) (OpenCV's own code path) or its restatement
oracle/subpix_oracle.c, which tests/test_subpix_cpu.py pins to it.  The frame step with the option is checked every frame
and sequence against the host loop of tests/test_gpu_grid_detect.py with cv2.cornerSubPix applied to each frame's new
corners, eagerly and replayed from the graphs.  With the option off the step launches what it launched before; with it
on, exactly one more kernel, between the step's last kernel and the records kernel."""
import ctypes
import json
import os

import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from subpix_cases import cases, images
from test_gpu_frame_step_async import DET, KITTI, LK, pad
from test_gpu_grid_detect import SNAP, all_launches, initial, short, uneven
from test_gpu_motion_prior import with_restarts
from test_gpu_sequence_control import Model, check_state
from test_gpu_thin import host_track, same_d
from test_gpu_track_history import Records, frames_at
from test_grid_detect_cpu import grid_detect
from test_motion_prior_cpu import detect, velocity_starts
from test_thin_cpu import thin

pytestmark = pytest.mark.gpu

SUBPIX = ((5, 5), (-1, -1), (3, 40, 0.001))


@pytest.fixture(scope="module")
def subpix_oracle():
    """oracle/subpix_oracle.c through its ctypes front-end (compiled with gcc on first use)."""
    from oracle import subpix_oracle
    subpix_oracle.build()
    return subpix_oracle


@pytest.fixture()
def cv2():
    cv2 = pytest.importorskip("cv2")
    was = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield cv2
    cv2.ipp.setUseIPP(was)


def same(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


# ---- the drop-in ---------------------------------------------------------------------------------------------------------

def test_drop_in_bit_exact_with_opencv(klt, cv2):
    n = 0
    for name, img, pts, win, zz, crit in cases(cv2):
        ref = cv2.cornerSubPix(img, pts.copy(), win, zz, crit)
        mine = pts.copy()
        out = klt.cornerSubPix(img, mine, win, zz, crit)
        assert out is mine
        bad = np.nonzero((mine.view(np.uint32) != ref.view(np.uint32)).any(-1).ravel())[0]
        assert bad.size == 0, "%s: %d of %d differ, first %s -> want %s got %s" % (name, bad.size, len(pts), pts[bad[0], 0],
                                                                                  ref[bad[0], 0], mine[bad[0], 0])
        n += len(pts)
    assert n >= 6000


def test_drop_in_shapes_and_errors(klt, cv2):
    img = images()["kitti"]
    c = cv2.goodFeaturesToTrack(img, 300, 0.01, 8)
    flat = c.reshape(-1, 2).copy()
    ref = cv2.cornerSubPix(img, c.copy(), *SUBPIX)
    assert klt.cornerSubPix(img, flat, *SUBPIX) is flat and same(flat, ref.reshape(-1, 2))
    row = c.reshape(1, -1, 2).copy()
    assert klt.cornerSubPix(img, row, *SUBPIX) is row and same(row, ref.reshape(1, -1, 2))
    bad = c.copy()
    bad[7, 0, 0] = np.nan
    keep = bad.copy()
    with pytest.raises(klt.error, match="contains"):
        klt.cornerSubPix(img, bad, *SUBPIX)
    assert np.array_equal(bad, keep, equal_nan=True)
    with pytest.raises(klt.error, match="count >= 0"):
        klt.cornerSubPix(img, c.astype(np.float64), *SUBPIX)
    with pytest.raises(klt.error, match="win.width > 0"):
        klt.cornerSubPix(img, c.copy(), (0, 3), (-1, -1), (3, 40, 0.001))


# ---- the batched device entry point --------------------------------------------------------------------------------------

def batch_inputs(cv2, B, h, w, N, seed):
    rng = np.random.default_rng(seed)
    imgs = np.stack([S.texture(h, w, seed=seed + b).astype(np.uint8) for b in range(B)])
    pts = np.zeros((B, N, 2), np.float32)
    for b in range(B):
        c = cv2.goodFeaturesToTrack(imgs[b], N, 0.01, 4, blockSize=5).reshape(-1, 2)
        k = len(c)
        pts[b, :k] = c + rng.uniform(-0.6, 0.6, (k, 2)).astype(np.float32)
        pts[b, k:] = np.stack([rng.uniform(0, w, N - k), rng.uniform(0, h, N - k)], 1)
    pts[:, :, 0] = np.clip(pts[:, :, 0], 0, w - 1)
    pts[:, :, 1] = np.clip(pts[:, :, 1], 0, h - 1)
    return imgs, pts


@pytest.mark.parametrize("B", [1, 5, 64])
def test_batched_against_the_oracle(klt, cv2, subpix_oracle, B):
    """counts with 0 and N, NaN and outside points left unchanged, slots behind the count untouched."""
    import torch
    from visual_odom_pipeline_b200 import detector as D
    h, w, N = 120, 167, 150
    imgs, pts = batch_inputs(cv2, B, h, w, N, seed=300 + B)
    pts[0, 3] = (np.nan, 10.0)
    pts[0, 4] = (-0.25, 30.0)
    pts[B - 1, 5] = (w, 20.0)
    pts[B - 1, 6] = (40.0, np.inf)
    counts = np.random.default_rng(B).integers(0, N + 1, B).astype(np.int32)
    counts[0] = N
    if B > 1:
        counts[1] = 0
    for win, zz, crit in [SUBPIX, ((3, 4), (1, 1), (1, 10, 0.0)), ((15, 15), (-1, -1), (2, 0, 0.01))]:
        d_img = torch.from_numpy(imgs).cuda()
        d_pts = torch.from_numpy(pts).cuda()
        out = D.corner_sub_pix(d_img, d_pts, win, zz, crit, counts=torch.from_numpy(counts).cuda())
        assert out is d_pts
        got = d_pts.cpu().numpy()
        for b in range(B):
            n = int(counts[b])
            ok = np.isfinite(pts[b]).all(1) & (pts[b, :, 0] >= 0) & (pts[b, :, 0] < w) & (pts[b, :, 1] >= 0) & (pts[b, :, 1] < h)
            ok[n:] = False
            want = pts[b].copy()
            want[ok] = subpix_oracle.corner_sub_pix(imgs[b], pts[b][ok], win, zz, crit)
            assert same(got[b], want), "B=%d sequence %d win %r" % (B, b, win)


def test_end_and_n_select_the_slots(klt, cv2, subpix_oracle):
    """The C ABI with distinct end and n arrays: slots [end - n, end) only, out-of-range values clamped."""
    import torch
    from visual_odom_pipeline_b200 import _lib
    B, h, w, N = 6, 90, 130, 80
    imgs, pts = batch_inputs(cv2, B, h, w, N, seed=77)
    end = np.array([80, 50, 200, 30, -5, 60], np.int32)
    n = np.array([30, 50, 10, 99, 4, -3], np.int32)
    d_img, d_pts = torch.from_numpy(imgs).cuda(), torch.from_numpy(pts).cuda()
    d_end, d_n = torch.from_numpy(end).cuda(), torch.from_numpy(n).cuda()
    ctx = _lib.default_context(0)
    L = _lib.load()
    win, zz, crit = SUBPIX
    rc = L.klt_corner_sub_pix(ctx.handle, d_img.data_ptr(), w, h, w, h * w, B, d_pts.data_ptr(), N, d_end.data_ptr(), d_n.data_ptr(),
                              win[0], win[1], zz[0], zz[1], crit[0], crit[1], crit[2], ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    got = d_pts.cpu().numpy()
    for b in range(B):
        e = min(max(int(end[b]), 0), N)
        s = e - min(max(int(n[b]), 0), e)
        want = pts[b].copy()
        if e > s:
            want[s:e] = subpix_oracle.corner_sub_pix(imgs[b], pts[b, s:e], win, zz, crit)
        assert same(got[b], want), b
    # argument checks before any device work
    args = [ctx.handle, d_img.data_ptr(), w, h, w, h * w, B, d_pts.data_ptr(), N, d_end.data_ptr(), d_n.data_ptr(), 5, 5, -1, -1, 3, 40, 0.001, None]
    for i, v, want in [(11, 0, _lib.KLT_ERR_INVALID_ARG), (2, 14, _lib.KLT_ERR_INVALID_ARG), (6, 0, _lib.KLT_ERR_INVALID_ARG),
                       (7, None, _lib.KLT_ERR_INVALID_ARG), (9, None, _lib.KLT_ERR_INVALID_ARG), (12, 16, _lib.KLT_ERR_UNSUPPORTED)]:
        a = list(args)
        a[i] = v
        if i == 12:
            a[2], a[3], a[4], a[5] = 200, 200, 200, 200 * 200
        assert L.klt_corner_sub_pix(*a) == want, (i, v)
    assert same(d_pts.cpu().numpy(), got)


# ---- KLTSequenceBatch(subpix=...) ----------------------------------------------------------------------------------------

def make(seqs, init, C, subpix, grid=None, q=None, history=0, control=False, motion_prior=None, second_pass="reference",
         max_err=30.0, dist=None):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init, n=C)
    return T.KLTSequenceBatch(frames_at(seqs, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), C,
                              history=history, control=control, motion_prior=motion_prior, second_pass=second_pass,
                              max_bidir_error=max_err, min_track_distance=dist, detect_grid=grid, tracks_per_cell=q,
                              subpix=subpix, **LK, **DET)


def drive(cv2, seqs, init, C, subpix=SUBPIX, grid=None, q=None, R=0, prior=None, requests=lambda t, m: {},
          second_pass="reference", max_err=30.0, control=False, dist=None):
    """An eager object and a graph-replayed twin against the host loop with cv2.cornerSubPix on every frame's new corners."""
    import torch
    B, T_ = len(seqs), len(seqs[0])
    reverse = second_pass == "reverse"
    objs = [make(seqs, init, C, subpix, grid, q, R, control, prior, second_pass, max_err, dist) for _ in range(2)]
    models = [Model(np.asarray(p, np.float32).reshape(-1, 2)) for p in init]
    refined = 0

    def det_fn(im, surv):
        nonlocal refined
        new = detect(cv2, im, surv, C) if grid is None else grid_detect(cv2, im, surv, C, grid, q)
        new = np.ascontiguousarray(new, np.float32).reshape(-1, 2)
        if len(new):
            r = cv2.cornerSubPix(im, new.reshape(-1, 1, 2).copy(), *subpix).reshape(-1, 2)
            refined += int((r != new).any(1).sum())
            new = r
        return new
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
        for b, m in enumerate(models):
            n = len(m.ids)
            d_ref = None
            if b in req.get("restart", {}):
                p = req["restart"][b]
                keep_ref = np.zeros(n, bool)
                new = det_fn(seqs[b][t], p)
                sids = np.arange(m.next_id, m.next_id + len(p), dtype=np.int32)
                m.next_id += len(p)
                m.ids = np.concatenate([sids, np.arange(m.next_id, m.next_id + len(new), dtype=np.int32)])
                m.next_id += len(new)
                m.pts = np.concatenate([p, new]).astype(np.float32)
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
            for name, g in zip(("eager", "graph"), snaps):
                tag = "%s frame %d sequence %d" % (name, t, b)
                assert np.array_equal(g["keep"][b, :n], keep_ref) and not g["keep"][b, n:].any(), tag + ": keep"
                if reverse and d_ref is not None:
                    assert same_d(g["bidir_error"][b, :n], d_ref), tag + ": bidir_error"
                assert int(g["n_new"][b]) == len(new), tag + ": n_new %d, want %d" % (int(g["n_new"][b]), len(new))
                assert int(g["counts"][b]) == len(m.ids), tag + ": counts"
                assert same(g["points"][b, :len(m.ids)], m.pts), tag + ": points"
                assert np.array_equal(g["ids"][b, :len(m.ids)], m.ids), tag + ": ids"
        if R:
            for sb, name in zip(objs, ("eager", "graph")):
                check_state(sb, models, C, R, "%s frame %d" % (name, t))
    assert objs[1]._graphs is not None
    assert refined > 0
    return objs, models


def test_step_refines_new_corners_every_frame(klt, cv2):
    """Three KITTI sequences, 9 frames, capacity 3000: points, counts, ids and keep as uint32 against the host loop."""
    seqs = [S.sequence(*KITTI, 9, seed=3100 + b) for b in range(3)]
    init = initial(cv2, seqs, [600, 0, 1500])
    drive(cv2, seqs, init, 3000)


def test_step_history_first_points_are_refined(klt, cv2):
    """history=3: the records (first_points of the new tracks among them) hold the refined positions."""
    import torch
    seqs = [S.sequence(*KITTI, 8, seed=3200 + b) for b in range(2)]
    init = initial(cv2, seqs, [400, 900])
    objs, models = drive(cv2, seqs, init, 2500, R=3)
    for sb in objs:
        fp, ff, ids = sb.first_points.cpu().numpy(), sb.first_frames.cpu().numpy(), sb.ids.cpu().numpy()
        for b, m in enumerate(models):
            born = ff[b, :len(m.ids)] == m.f
            assert born.any()
            assert same(fp[b, :len(m.ids)][born], m.pts[born])
            assert (m.pts[born] != np.round(m.pts[born])).any()
    torch.cuda.synchronize()


def test_step_restarts_refine_only_the_new_corners(klt, cv2):
    """control restarts: the corners detected behind the staged points are refined, the staged points are not."""
    seqs = [S.sequence(*KITTI, 8, seed=3300 + b) for b in range(3)]
    init = initial(cv2, seqs, [500, 700, 300])
    drive(cv2, seqs, init, 2500, R=2, control=True,
          requests=with_restarts(cv2, seqs, lambda t, m: {}, {3: {0: 150, 2: 30}, 6: {1: 40}}))


def test_step_with_grid_thinning_reverse_and_velocity(klt, cv2):
    """detect_grid, min_track_distance, second_pass="reverse" and motion_prior="velocity" together, with drops."""
    B, C = 3, 2500
    seqs = uneven(B, 3400, 8)
    init = initial(cv2, seqs, [400, 800, 1200])
    rng = np.random.default_rng(9)

    def req(t, models):
        d = np.zeros((B, C), bool)
        for b, m in enumerate(models):
            d[b, :len(m.ids)] = rng.random(len(m.ids)) < 0.05
        return {"drop": d}
    drive(cv2, seqs, init, C, subpix=((4, 3), (0, 0), (3, 20, 0.01)), grid=(8, 4), q=48, R=2, prior="velocity", requests=req,
          second_pass="reverse", max_err=1.0, control=True, dist=10.0)


def test_step_rejects_a_window_the_frame_cannot_hold(klt):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    f = torch.zeros((1, 20, 40), dtype=torch.uint8, device="cuda")
    p = torch.zeros((1, 0, 2), dtype=torch.float32, device="cuda")
    c = torch.zeros((1,), dtype=torch.int32, device="cuda")
    for bad in [((5, 8), (-1, -1), (3, 40, 0.001)), ((0, 2), (-1, -1), (3, 40, 0.001)), ((16, 2), (-1, -1), (3, 40, 0.001)), (5, 5)]:
        with pytest.raises(klt.error):
            T.KLTSequenceBatch(f, p, c, 16, winSize=(5, 5), maxLevel=0, subpix=bad)
    T.KLTSequenceBatch(f, p, c, 16, winSize=(5, 5), maxLevel=0, subpix=((7, 5), (-1, -1), (3, 40, 0.001)))


# ---- launches ------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def launches(klt, tmp_path_factory):
    """One eager step with the option off, on, and from an object built without the argument, profiled in a child
    process (this file run as a script; the test process never starts a CUPTI session)."""
    import subprocess
    import sys
    out = tmp_path_factory.mktemp("subpix_launches")
    tests = os.path.dirname(os.path.abspath(__file__))
    path = [os.path.dirname(tests), tests] + ([os.environ["PYTHONPATH"]] if os.environ.get("PYTHONPATH") else [])
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, PYTHONPATH=os.pathsep.join(path)), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, "profiling child failed:\n" + r.stdout[-4000:] + r.stderr[-4000:]
    with open(out / "launches.json") as f:
        return json.load(f)


def test_launches(klt, launches):
    """Off: the same launches as an object built without the argument.  On: exactly one more kernel, the refinement,
    right before the records kernel."""
    off, plain, on = launches["off"], launches["plain"], launches["on"]
    assert off == plain
    names = [short(n) for n, _g, _b in on]
    i = names.index("subpix_kernel")
    assert names.count("subpix_kernel") == 1 and len(on) == len(off) + 1
    assert on[:i] + on[i + 1:] == off
    assert names[i + 1].startswith("track_records"), names[i - 1:i + 2]


if __name__ == "__main__":
    # the child process of the `launches` fixture: python tests/test_gpu_subpix.py OUT_DIR
    import sys
    import cv2 as cv2_
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    seqs_ = [S.sequence(*KITTI, 3, seed=3500 + b) for b in range(3)]
    init_ = initial(cv2_, seqs_, [500, 0, 1500])
    res = {}
    for arm in ("off", "on", "plain"):
        padded, cnt = pad(init_, n=2048)
        kw = {} if arm == "plain" else {"subpix": SUBPIX if arm == "on" else None}
        sb = T.KLTSequenceBatch(frames_at(seqs_, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), 2048, history=2,
                                **kw, **LK, **DET)
        sb.step(frames_at(seqs_, 1))
        f2 = frames_at(seqs_, 2)
        res[arm] = all_launches(torch, lambda: sb.step(f2), os.path.join(sys.argv[1], "%s.json" % arm))
    with open(os.path.join(sys.argv[1], "launches.json"), "w") as f:
        json.dump(res, f)
