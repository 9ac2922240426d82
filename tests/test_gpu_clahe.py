"""GPU tier (pytest -m gpu, B200) of contrast-limited equalisation: the createCLAHE drop-in, the batched filters.clahe and
KLTTracker / KLTSequenceBatch(equalize=...).

Bar: bit for bit against cv2.createCLAHE(clipLimit, tileGridSize).apply (oracle/clahe_oracle.py restates it and
tests/test_clahe_cpu.py pins it).  The frame step with the option is checked every frame and sequence against the host
loop of tests/test_gpu_subpix.py run on clahe.apply(frame), eagerly and replayed from the graphs.  With the option off
the objects launch what they launched before; with it on, exactly the two CLAHE kernels more, before the new frame's
pyramid build."""
import ctypes
import json
import os

import numpy as np
import pytest

from visual_odom_pipeline_b200 import synth as S
from clahe_cases import cases, image
from test_gpu_frame_step_async import DET, KITTI, LK, cv2_step, pad
from test_gpu_grid_detect import SNAP, all_launches, initial, short
from test_gpu_motion_prior import with_restarts
from test_gpu_sequence_control import Model, check_state
from test_gpu_thin import host_track, same_d
from test_gpu_track_history import Records, frames_at
from test_grid_detect_cpu import grid_detect
from test_motion_prior_cpu import detect, velocity_starts
from test_thin_cpu import thin

pytestmark = pytest.mark.gpu

EQ = (3.0, (8, 8))
GAINS = [1.0, 1.0, 0.7, 0.7, 1.0, 0.5, 0.5, 1.0, 1.4, 1.0]


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


@pytest.fixture()
def cv2_own_code(cv2):
    """cv2 with IPP off: cornerSubPix is bit-exact with OpenCV's own code path only (tests/test_gpu_subpix.py)."""
    was = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield cv2
    cv2.ipp.setUseIPP(was)


def equalized(cv2, seqs, eq=EQ):
    c = cv2.createCLAHE(*eq)
    return [[c.apply(f) for f in s] for s in seqs]


# ---- the drop-in ---------------------------------------------------------------------------------------------------------

def test_drop_in_bit_exact_with_opencv(klt, cv2):
    n = 0
    for name, img, clip, grid in cases():
        ref = cv2.createCLAHE(clip, grid).apply(img)
        got = klt.createCLAHE(clip, grid).apply(img)
        bad = int((got != ref).sum())
        assert bad == 0, "%s: %d of %d pixels differ" % (name, bad, ref.size)
        n += ref.size
    assert n > 20_000_000


def test_drop_in_views_dst_and_errors(klt, cv2):
    big = image("texture", 400, 1300, 5)
    view = big[7:383, 11:1252]                              # KITTI-size view with a row stride of 1300
    strided = big[::2, ::3]                                 # non-unit column stride
    c, ref_c = klt.createCLAHE(2.0, (8, 8)), cv2.createCLAHE(2.0, (8, 8))
    for src in (view, strided, big[:, :, None][5:100, 3:70]):
        assert np.array_equal(c.apply(src), ref_c.apply(src))
    dst = np.empty(view.shape, np.uint8)
    assert c.apply(view, dst) is dst and np.array_equal(dst, ref_c.apply(view))
    pitched = np.zeros((376, 1400), np.uint8)[:, 5:1246]
    assert c.apply(view, pitched) is pitched and np.array_equal(pitched, ref_c.apply(view))
    inplace = view.copy()
    want = ref_c.apply(inplace)
    assert c.apply(inplace, inplace) is inplace and np.array_equal(inplace, want)
    wrong = np.empty((3, 3), np.uint8)
    out = c.apply(view, wrong)
    assert out is not wrong and np.array_equal(out, ref_c.apply(view))
    assert issubclass(klt.error, cv2.error)
    for bad in (view.astype(np.uint16), np.dstack([view] * 3), view.astype(np.float32)):
        with pytest.raises(cv2.error):
            c.apply(bad)
    with pytest.raises(cv2.error):
        klt.createCLAHE(3.0, (0, 8))


# ---- the batched device entry point --------------------------------------------------------------------------------------

def test_batched_equals_cv2_per_image(klt, cv2):
    """(B, H, W) batches: default output, a pitched `out`, in place, (H, W) input; several grids and clip limits."""
    import torch
    from visual_odom_pipeline_b200 import filters as F
    from visual_odom_pipeline_b200 import tracker as T
    for (h, w), B in [(KITTI, 5), ((101, 37), 3), ((9, 17), 64), ((768, 1024), 2)]:
        imgs = np.stack([image(("noise", "texture", "levels", "constant")[b % 4], h, w, 40 + b) for b in range(B)])
        for clip, grid in [(3.0, (8, 8)), (40.0, (7, 5)), (0.0, (1, 1)), (1.0, (20, 20))]:
            want = np.stack([cv2.createCLAHE(clip, grid).apply(x) for x in imgs])
            d = torch.from_numpy(imgs).cuda()
            out = F.clahe(d, clip, grid)
            assert out.stride(1) % 128 == 0
            assert np.array_equal(out.cpu().numpy(), want), ((h, w), B, clip, grid)
            pitched = torch.zeros((B, h + 3, w + 77), dtype=torch.uint8, device="cuda")[:, 1:h + 1, 5:w + 5]
            assert F.clahe(d, clip, grid, out=pitched) is pitched
            assert np.array_equal(pitched.cpu().numpy(), want)
            own = T.alloc_image_batch(B, h, w)
            own.copy_(d)
            F.clahe(own, clip, grid, out=own)
            assert np.array_equal(own.cpu().numpy(), want)
            assert np.array_equal(d.cpu().numpy(), imgs)
        single = F.clahe(torch.from_numpy(imgs[0]).cuda(), *EQ)
        assert tuple(single.shape) == (h, w) and np.array_equal(single.cpu().numpy(), cv2.createCLAHE(*EQ).apply(imgs[0]))


def test_unpadded_narrow_tiles_and_2d_in_place(klt, cv2):
    """Grids that divide the image into tiles of 4 pixels or fewer with w % 4 != 0 (the last 4-pixel group of a row runs past
    it), each through klt_clahe with a workspace of exactly klt_clahe_ws_bytes; and an (H, W) tensor equalized in place."""
    import torch
    from visual_odom_pipeline_b200 import _lib
    from visual_odom_pipeline_b200 import filters as F
    L = _lib.load()
    ctx = _lib.default_context(0)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for (h, w), grid, B in [((8, 9), (9, 8), 3), ((1, 1), (1, 1), 2), ((376, 1241), (1241, 47), 2), ((7, 13), (13, 7), 5),
                            ((12, 30), (10, 4), 4)]:
        imgs = np.stack([image(("noise", "texture", "levels")[b % 3], h, w, 70 + b) for b in range(B)])
        want = np.stack([cv2.createCLAHE(2.0, grid).apply(x) for x in imgs])
        src = torch.from_numpy(imgs).cuda()
        dst = torch.zeros_like(src)
        ws = torch.empty((int(L.klt_clahe_ws_bytes(B, *grid)),), dtype=torch.uint8, device="cuda")
        assert L.klt_clahe(ctx.handle, src.data_ptr(), w, h, w, h * w, dst.data_ptr(), w, h * w, B, 2.0, grid[0], grid[1],
                           ws.data_ptr(), ws.numel(), st) == 0
        assert np.array_equal(dst.cpu().numpy(), want), ((h, w), grid)
    img = torch.from_numpy(image("texture", 101, 37, 3)).cuda()
    want = cv2.createCLAHE(*EQ).apply(img.cpu().numpy())
    assert F.clahe(img, *EQ, out=img) is img
    assert np.array_equal(img.cpu().numpy(), want)


def test_c_abi_checks(klt):
    """Every argument error of klt_clahe is returned before any device work: the output stays untouched."""
    import torch
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    ctx = _lib.default_context(0)
    B, h, w = 2, 40, 50
    src = torch.randint(0, 256, (B, h, w), dtype=torch.uint8, device="cuda")
    dst = torch.zeros_like(src)
    ws = torch.zeros((int(L.klt_clahe_ws_bytes(B, 8, 8)),), dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    args = [ctx.handle, src.data_ptr(), w, h, w, h * w, dst.data_ptr(), w, h * w, B, 3.0, 8, 8, ws.data_ptr(), ws.numel(), st]
    INV, UNS = _lib.KLT_ERR_INVALID_ARG, _lib.KLT_ERR_UNSUPPORTED
    for changes, want in [({1: None}, INV), ({6: None}, INV), ({13: None}, INV), ({2: 0}, INV), ({3: 0}, INV), ({9: 0}, INV),
                          ({4: w - 1}, INV), ({7: w - 1}, INV), ({11: 0}, INV), ({12: -1}, INV), ({10: float("nan")}, INV),
                          ({10: float("inf")}, INV), ({10: 1e12}, INV), ({14: ws.numel() - 1}, INV), ({13: ws.data_ptr() + 4}, INV),
                          ({6: src.data_ptr(), 7: w + 1}, INV), ({11: 257, 12: 256}, UNS), ({9: 65536}, UNS)]:
        a = list(args)
        for i, v in changes.items():
            a[i] = v
        assert L.klt_clahe(*a) == want, changes
    torch.cuda.synchronize()
    assert int(dst.count_nonzero()) == 0
    assert L.klt_clahe(*args) == 0
    torch.cuda.synchronize()
    assert int(dst.count_nonzero()) > 0


# ---- KLTTracker / KLTSequenceBatch(equalize=...) -------------------------------------------------------------------------

def test_tracker_step_batch_equalized(klt, cv2):
    """KLTTracker(equalize=...).step_batch, every frame, against the reference's step with cv2 on clahe.apply(frame)."""
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    B = 3
    seqs = [S.exposure_sequence(*KITTI, 5, GAINS[:5], seed=600 + b) for b in range(B)]
    host = equalized(cv2, seqs)
    init = initial(cv2, host, [0, 400, 900])
    trk = T.KLTTracker(**LK, equalize=EQ).reset(frames_at(seqs, 0))
    padded, cnt = pad(init)
    pts, counts = torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda()
    hp = [p.reshape(-1, 2) for p in init]
    for t in range(1, 5):
        nxt, ncnt, keep, n_new = trk.step_batch(frames_at(seqs, t), pts, counts, **DET)
        hn, hc, hk = nxt.cpu().numpy(), ncnt.cpu().numpy(), keep.cpu().numpy()
        for b in range(B):
            keep_ref, surv, new, _n, _bound = cv2_step(cv2, host[b][t - 1], host[b][t], hp[b], DET, 10 ** 9)
            tag = "frame %d sequence %d" % (t, b)
            assert np.array_equal(hk[b, :len(hp[b])], keep_ref), tag + ": keep"
            ref = np.concatenate([surv, new]).astype(np.float32)
            assert int(hc[b]) == len(ref), tag + ": counts"
            assert np.array_equal(hn[b, :len(ref)].view(np.uint32), ref.view(np.uint32)), tag + ": points"
            hp[b] = ref
        pts, counts = nxt.contiguous(), ncnt
    # step (one sequence) and the pyramid's level 0 hold the equalized frame
    one = T.KLTTracker(**LK, equalize=EQ).reset(frames_at(seqs[:1], 0))
    surv, keep, new = one.step(frames_at(seqs[:1], 1)[0], torch.from_numpy(hp[0][:0]).cuda())
    assert np.array_equal(one.prev.images[0].cpu().numpy(), host[0][1])
    want = cv2.goodFeaturesToTrack(host[0][1], **DET)
    assert np.array_equal(new, want)


def make(seqs, init, C, equalize, prefilter=None, subpix=None, grid=None, q=None, history=0, control=False, motion_prior=None,
         second_pass="reference", max_err=30.0, dist=None):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init, n=C)
    return T.KLTSequenceBatch(frames_at(seqs, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), C,
                              history=history, control=control, motion_prior=motion_prior, second_pass=second_pass,
                              max_bidir_error=max_err, min_track_distance=dist, detect_grid=grid, tracks_per_cell=q,
                              subpix=subpix, prefilter=prefilter, equalize=equalize, **LK, **DET)


def drive(cv2, seqs, host, init, C, equalize=EQ, prefilter=None, subpix=None, grid=None, q=None, R=0, prior=None,
          requests=lambda t, m: {}, second_pass="reference", max_err=30.0, control=False, dist=None):
    """An eager object and a graph-replayed twin on the raw frames `seqs` against the host loop on `host`, the frames the
    object should see (clahe.apply(frame), or of the bilateral frame) -> the objects, the models and the kept fraction of
    every step and sequence."""
    import torch
    B, T_ = len(seqs), len(seqs[0])
    reverse = second_pass == "reverse"
    objs = [make(seqs, init, C, equalize, prefilter, subpix, grid, q, R, control, prior, second_pass, max_err, dist) for _ in range(2)]
    models = [Model(np.asarray(p, np.float32).reshape(-1, 2)) for p in init]
    kept = []

    def det_fn(im, surv):
        new = detect(cv2, im, surv, C) if grid is None else grid_detect(cv2, im, surv, C, grid, q)
        new = np.ascontiguousarray(new, np.float32).reshape(-1, 2)
        if subpix is not None and len(new):
            new = cv2.cornerSubPix(im, new.reshape(-1, 1, 2).copy(), *subpix).reshape(-1, 2)
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
        kept.append([])
        for b, m in enumerate(models):
            n = len(m.ids)
            d_ref = None
            if b in req.get("restart", {}):
                p = req["restart"][b]
                keep_ref = np.zeros(n, bool)
                new = det_fn(host[b][t], p)
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
                keep_ref, p1, d_ref = host_track(cv2, host[b][t - 1], host[b][t], m.pts, starts, reverse, max_err)
                if n:
                    kept[-1].append(float(keep_ref.mean()))
                if drop is not None:
                    keep_ref = keep_ref & ~drop[b, :n]
                if dist is not None:
                    keep_ref = keep_ref & ~thin(p1, keep_ref, dist)
                surv = p1[keep_ref]
                new = det_fn(host[b][t], surv)
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
                assert np.array_equal(g["points"][b, :len(m.ids)].view(np.uint32), m.pts.view(np.uint32)), tag + ": points"
                assert np.array_equal(g["ids"][b, :len(m.ids)], m.ids), tag + ": ids"
        if R:
            for sb, name in zip(objs, ("eager", "graph")):
                check_state(sb, models, C, R, "%s frame %d" % (name, t))
    assert objs[1]._graphs is not None
    return objs, models, kept


def test_sequence_batch_equalized_every_frame(klt, cv2):
    """Three KITTI sequences under changing exposure, capacity 3000: points, counts, ids and keep as uint32."""
    seqs = [S.exposure_sequence(*KITTI, 7, GAINS[:7], seed=700 + b) for b in range(3)]
    host = equalized(cv2, seqs)
    drive(cv2, seqs, host, initial(cv2, host, [600, 0, 1500]), 3000)


def test_sequence_batch_prefilter_then_equalize(klt, cv2):
    """prefilter=(5, 1.5, 1.5) and equalize: the host loop runs on clahe.apply of the device's bilateral frame (that filter
    equals cv2 only up to rounding ties)."""
    import torch
    from visual_odom_pipeline_b200 import filters as F
    pre = (5, 1.5, 1.5)
    seqs = [S.exposure_sequence(*KITTI, 6, GAINS[3:9], seed=800 + b) for b in range(2)]
    filtered = [[F.bilateral_filter(torch.from_numpy(f).cuda(), *pre).cpu().numpy() for f in s] for s in seqs]
    host = equalized(cv2, filtered, (2.0, (7, 5)))
    drive(cv2, seqs, host, initial(cv2, host, [700, 300]), 2500, equalize=(2.0, (7, 5)), prefilter=pre)


def test_sequence_batch_equalize_with_every_option(klt, cv2_own_code):
    """history, control (drops and restarts), motion_prior="velocity", second_pass="reverse", min_track_distance,
    detect_grid and subpix together with equalize."""
    cv2 = cv2_own_code
    B, C = 3, 2500
    seqs = [S.exposure_sequence(*KITTI, 8, GAINS[:8], seed=900 + b) for b in range(B)]
    host = equalized(cv2, seqs)
    init = initial(cv2, host, [400, 800, 1200])
    rng = np.random.default_rng(9)

    def req(t, models):
        d = np.zeros((B, C), bool)
        for b, m in enumerate(models):
            d[b, :len(m.ids)] = rng.random(len(m.ids)) < 0.05
        return {"drop": d}
    drive(cv2, seqs, host, init, C, subpix=((4, 3), (0, 0), (3, 20, 0.01)), grid=(8, 4), q=48, R=2, prior="velocity",
          requests=with_restarts(cv2, host, req, {4: {1: 60}}), second_pass="reverse", max_err=1.0, control=True, dist=10.0)


def test_exposure_changes_keep_tracks_only_when_equalized(klt, cv2):
    """The forward-backward check at 1 px on gains 1, 1, .7, .7, 1, .5, .5, 1, 1.4, 1: with equalize=(3.0, (8, 8)) every
    step keeps >= 0.95 of its tracks; without it the steps at a gain change keep < 0.7."""
    seqs = [S.exposure_sequence(*KITTI, len(GAINS), GAINS, seed=11)]
    host = equalized(cv2, seqs)
    _o, _m, kept_on = drive(cv2, seqs, host, initial(cv2, host, [1000]), 4096, second_pass="reverse", max_err=1.0)
    _o, _m, kept_off = drive(cv2, seqs, seqs, initial(cv2, seqs, [1000]), 4096, equalize=None, second_pass="reverse",
                             max_err=1.0)
    on = [k[0] for k in kept_on]
    off = [k[0] for k in kept_off]
    assert min(on) >= 0.95, on
    changes = [t - 1 for t in range(1, len(GAINS)) if GAINS[t] != GAINS[t - 1]]
    assert all(off[i] < 0.7 for i in changes), (off, changes)


def test_rejects_what_klt_clahe_rejects(klt):
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    f = torch.zeros((1, 40, 60), dtype=torch.uint8, device="cuda")
    p = torch.zeros((1, 0, 2), dtype=torch.float32, device="cuda")
    c = torch.zeros((1,), dtype=torch.int32, device="cuda")
    for bad in [(3.0, (0, 8)), (float("nan"), (8, 8)), (3.0, (300, 300)), (1e12, (1, 1)), 3.0, (3.0, 8)]:
        with pytest.raises(klt.error):
            T.KLTSequenceBatch(f, p, c, 16, winSize=(5, 5), maxLevel=0, equalize=bad)
        with pytest.raises(klt.error):
            T.DevicePyramid(f, (5, 5), 0, equalize=bad)
    T.KLTSequenceBatch(f, p, c, 16, winSize=(5, 5), maxLevel=0, equalize=(3.0, (61, 41)))


# ---- launches ------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def launches(klt, tmp_path_factory):
    """One eager step with the option off, on, and from an object built without the argument, profiled in a child
    process (this file run as a script; the test process never starts a CUPTI session)."""
    import subprocess
    import sys
    out = tmp_path_factory.mktemp("clahe_launches")
    tests = os.path.dirname(os.path.abspath(__file__))
    path = [os.path.dirname(tests), tests] + ([os.environ["PYTHONPATH"]] if os.environ.get("PYTHONPATH") else [])
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, PYTHONPATH=os.pathsep.join(path)), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, "profiling child failed:\n" + r.stdout[-4000:] + r.stderr[-4000:]
    with open(out / "launches.json") as f:
        return json.load(f)


def test_launches(klt, launches):
    """Off: the same launches as an object built without the argument.  On: exactly the two CLAHE kernels more, right
    before the first pyramid kernel of the new frame."""
    off, plain, on = launches["off"], launches["plain"], launches["on"]
    assert off == plain
    names = [short(n) for n, _g, _b in on]
    i = names.index("clahe_lut_kernel")
    assert names.count("clahe_lut_kernel") == 1 and names.count("clahe_apply_kernel") == 1 and names[i + 1] == "clahe_apply_kernel"
    assert len(on) == len(off) + 2 and on[:i] + on[i + 2:] == off
    assert "pyr" in names[i + 2].lower() or "down" in names[i + 2].lower(), names[i - 1:i + 3]


if __name__ == "__main__":
    # the child process of the `launches` fixture: python tests/test_gpu_clahe.py OUT_DIR
    import sys
    import cv2 as cv2_
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    seqs_ = [S.exposure_sequence(*KITTI, 3, [1.0, 0.7, 1.0], seed=950 + b) for b in range(3)]
    init_ = initial(cv2_, seqs_, [500, 0, 1500])
    res = {}
    for arm in ("off", "on", "plain"):
        padded, cnt = pad(init_, n=2048)
        kw = {} if arm == "plain" else {"equalize": EQ if arm == "on" else None}
        sb = T.KLTSequenceBatch(frames_at(seqs_, 0), torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda(), 2048, history=2,
                                **kw, **LK, **DET)
        sb.step(frames_at(seqs_, 1))
        f2 = frames_at(seqs_, 2)
        res[arm] = all_launches(torch, lambda: sb.step(f2), os.path.join(sys.argv[1], "%s.json" % arm))
    with open(os.path.join(sys.argv[1], "launches.json"), "w") as f:
        json.dump(res, f)
