"""GPU tier (pytest -m gpu, B200): every LK kernel instance the batched frame step can launch, against the reference's
capped cv2 loop.

The step's two LK passes carry per-sequence counts, so they run the instances with counts: lk_fast_kernel<W, H, WPP,
true> for 21x21 and 31x31, the generic lk_kernel for every other window.  Which one runs, and on which grid, depends on the
window and on B x n_per_seq (n_per_seq = the capacity C in KLTSequenceBatch, the points tensor's width in step_batch),
measured against the SM count.  Each case reads the name, grid and block of its first step's LK launches from a
torch.profiler trace (taken in a child process on the same inputs), so it shows that it ran the instance it is named after.  Then, per sequence and frame, keep, the survivors (float32
compared as uint32), the new corners (value and order), the counts and the ids equal the cv2 loop, eagerly and replayed
from the CUDA graphs (lk_fast_kernel is launched with programmatic dependent launch, lk_kernel is not)."""
import collections
import json
import os
import re

import numpy as np
import pytest

from test_gpu_frame_step_async import DET, KITTI, pad, snapshot
from visual_odom_pipeline_b200 import synth as S

pytestmark = pytest.mark.gpu

CRITERIA = (3, 30, 0.03)
FRAMES = 4          # three steps: the first eager, then one replay of each graph parity

Case = collections.namedtuple("Case", "name win max_level top kernel block pts_per_cta two_pass shape side counts")
FAST = "lk_fast_kernel<%d,%d,%d,true>"
# shape(sms) -> (B, C); side = (lo, hi): lo x SMs < B x C <= hi x SMs (None: no bound), the launcher's thresholds are
# 32 x SMs (21x21: 2 warps per point above it) and 128 x SMs (the 4-warp shapes: two-pass grid at or below it);
# counts(C) -> points per sequence
CASES = [
    Case("a-21x21-4warps-two_pass-B2", (21, 21), 3, 3, FAST % (21, 21, 4), 128, 1, True,
         lambda sms: (2, 2048), (None, 32), lambda C: [0, 1900]),
    Case("a-21x21-4warps-two_pass-B1-at_32xSMs", (21, 21), 3, 3, FAST % (21, 21, 4), 128, 1, True,
         lambda sms: (1, 32 * sms), (None, 32), lambda C: [1900]),
    Case("b-21x21-2warps-C_odd", (21, 21), 3, 3, FAST % (21, 21, 2), 128, 2, False,
         lambda sms: (5, 1501), (32, None), lambda C: [0, 1, 2, 750, C]),
    Case("c-31x31-4warps-one_pass-past_128xSMs", (31, 31), 3, 3, FAST % (31, 31, 4), 128, 1, False,
         lambda sms: (5, 128 * sms // 5 + 1), (128, None), lambda C: [0, 1, 777, 2001, C]),
    Case("d-15x15-lk_kernel-4warps", (15, 15), 3, 3, "lk_kernel<true>", 128, 4, False,
         lambda sms: (3, 1003), (None, None), lambda C: [0, 7, C]),
    Case("e-11x372-lk_kernel-2warps", (11, 372), 3, 0, "lk_kernel<false>", 64, 2, False,
         lambda sms: (3, 301), (None, None), lambda C: [0, 1, C]),
    Case("f-21x21-2warps-maxLevel0", (21, 21), 0, 0, FAST % (21, 21, 2), 128, 2, False,
         lambda sms: (5, 1501), (32, None), lambda C: [0, 1, 2, 750, C]),
    Case("f-21x21-2warps-maxLevel5", (21, 21), 5, 4, FAST % (21, 21, 2), 128, 2, False,
         lambda sms: (5, 1501), (32, None), lambda C: [0, 1, 2, 750, C]),
]
CASE_B = CASES[2]


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def sms(klt):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def lk_launches(torch, fn, trace):
    """Runs fn under torch.profiler -> [(instance, grid, block)] of every LK kernel it launched, in order.  instance is the
    kernel's name with its template arguments, without spaces (e.g. 'lk_fast_kernel<21,21,2,true>')."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(trace))
    with open(trace) as f:
        events = json.load(f)["traceEvents"]
    launches = []
    for e in sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"]):
        m = re.search(r"\b(lk_fast_kernel|lk_kernel)<([^>]*)>", e["name"])
        if m:
            args = e.get("args", {})
            assert "grid" in args and "block" in args, "the profiler trace carries no launch dimensions: %r" % e
            launches.append(("%s<%s>" % (m.group(1), m.group(2).replace(" ", "")), list(args["grid"]), list(args["block"])))
    return launches


def first_step_launches(torch, cv2, sms, out_dir):
    """The LK launches of each case's first eager KLTSequenceBatch step, and of KLTTracker.step_batch on case b's initial
    rows (width C) -> {case name or 'step_batch': launches}.  Runs in the child process of the `launches` fixture."""
    from visual_odom_pipeline_b200 import tracker as T
    res = {}
    for i, case in enumerate(CASES):
        B, C = case.shape(sms)
        lk = dict(winSize=case.win, maxLevel=case.max_level, criteria=CRITERIA)
        seqs, init = case_inputs(cv2, case, B, C, seed=400 + 10 * i)
        frames = torch.from_numpy(np.stack([s[1] for s in seqs])).cuda()
        sb = make_batch(torch, seqs, init, C, lk)
        res[case.name] = lk_launches(torch, lambda: sb.step(frames), os.path.join(out_dir, "%d.json" % i))
        if case is CASE_B:
            trk = T.KLTTracker(**lk).reset(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda())
            padded, cnt = pad(init, n=C)
            pts, cnt = torch.from_numpy(padded).cuda(), torch.from_numpy(cnt).cuda()
            res["step_batch"] = lk_launches(torch, lambda: trk.step_batch(frames, pts, cnt, max_bidir_error=30, mask_radius=10, **DET),
                                            os.path.join(out_dir, "step_batch.json"))
    return res


@pytest.fixture(scope="module")
def launches(klt, tmp_path_factory):
    """first_step_launches, profiled in a child process (this file run as a script).  A CUPTI session in the test process
    made the profiler sessions of a later module (tests/test_gpu_pyramid_cluster.py) lose their kernel records (B200,
    torch 2.11, with or without TEARDOWN_CUPTI=0), so this process never starts one."""
    import subprocess
    import sys
    out = tmp_path_factory.mktemp("lk_launches")
    tests = os.path.dirname(os.path.abspath(__file__))
    path = [os.path.dirname(tests), tests] + ([os.environ["PYTHONPATH"]] if os.environ.get("PYTHONPATH") else [])
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, PYTHONPATH=os.pathsep.join(path)), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, "profiling child failed:\n" + r.stdout[-4000:] + r.stderr[-4000:]
    with open(out / "launches.json") as f:
        return {k: [(n, tuple(g), tuple(b)) for n, g, b in v] for k, v in json.load(f).items()}


def check_launches(case, launches, total, capsys, what):
    """Both LK passes ran case.kernel, on case's grid, and no other LK kernel ran."""
    blocks = -(-total // case.pts_per_cta) * (2 if case.two_pass else 1)
    want = (case.kernel, (blocks, 1, 1), (case.block, 1, 1))
    assert launches == [want, want], "%s: expected two launches of %r, got %r" % (what, want, launches)
    with capsys.disabled():
        print("\n%s: %s ran %s x 2, grid %d x %d threads (B x C = %d, %s)"
              % (case.name, what, case.kernel, blocks, case.block, total, "two-pass grid" if case.two_pass else "one pass"))


def band_points(n, seed):
    """n points of the 30-px band around and across the image border (some windows overlap it, some points lie outside)."""
    h, w = KITTI
    p = S.uniform_points(4 * n + 64, h, w, seed=seed, margin=30).reshape(-1, 2)
    m = np.minimum(np.minimum(p[:, 0], w - 1 - p[:, 0]), np.minimum(p[:, 1], h - 1 - p[:, 1]))
    p = p[m < 30]
    assert len(p) >= n
    return p[:n]


def case_inputs(cv2, case, B, C, seed):
    """B KITTI-size sequences of FRAMES frames and their initial points: goodFeaturesToTrack corners of the first frame
    mixed with border-band points (shuffled, so neighbouring slots fall into both passes of a two-pass grid); in the
    cases whose last sequence is full at a capacity of thousands, that one holds uniform points over the image and band."""
    h, w = KITTI
    counts = case.counts(C)
    assert len(counts) == B and max(counts) <= C
    seqs = [S.sequence(h, w, FRAMES, seed=seed + b) for b in range(B)]
    init = []
    for b, n in enumerate(counts):
        if n == C and C > 3000:
            p = S.uniform_points(n, h, w, seed=seed + 50 + b, margin=30).reshape(-1, 2)
        else:
            c = cv2.goodFeaturesToTrack(seqs[b][0], **DET).reshape(-1, 2)[: (n + 1) // 2]
            p = np.concatenate([c, band_points(n - len(c), seed + 50 + b)])
            np.random.default_rng(seed + b).shuffle(p)
        assert len(p) == n
        init.append(p.astype(np.float32))
    return seqs, init


def make_batch(torch, seqs, init, C, lk):
    from visual_odom_pipeline_b200 import tracker as T
    padded, cnt = pad(init, n=C)
    return T.KLTSequenceBatch(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda(), torch.from_numpy(padded).cuda(),
                              torch.from_numpy(cnt).cuda(), C, max_bidir_error=30, mask_radius=10, **lk, **DET)


def cv2_step(cv2, lk, im0, im1, pts, cap, radius=10, max_bidir=30):
    """The reference's step (src/extractor/extractor.py:38-59,102-111) at the LK parameters lk, with the capacity cap
    (maxCorners = min(maxCorners, cap - survivors), no detection when that is 0) -> keep (n,) bool, survivors (s, 2),
    new corners (k, 2)."""
    h, w = im1.shape
    if len(pts):
        p0 = pts.reshape(-1, 1, 2)
        p1, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **lk)
        p0r, _s, _e = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **lk)
        good = abs(p0 - p0r).reshape(-1, 2).max(-1) < max_bidir
        p1 = p1.reshape(-1, 2)
        keep = good & (0 <= p1[:, 0]) & (p1[:, 0] <= w) & (0 <= p1[:, 1]) & (p1[:, 1] <= h)
        surv = p1[keep]
    else:
        keep, surv = np.zeros(0, bool), np.zeros((0, 2), np.float32)
    mask = np.full_like(im1, 255)
    for x, y in [np.int32(p) for p in surv]:
        cv2.circle(mask, (int(x), int(y)), radius, 0, -1)
    k = min(DET["maxCorners"], cap - len(surv))
    new = np.zeros((0, 2), np.float32)
    if k > 0:
        c = cv2.goodFeaturesToTrack(im1, mask=mask, **dict(DET, maxCorners=k))
        new = new if c is None else c.reshape(-1, 2)
    return keep, surv, new


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_lk_instance_against_capped_cv2(klt, cv2, sms, launches, capsys, case):
    """The first step of an eager KLTSequenceBatch (profiled in the `launches` child): both LK passes ran the case's
    instance on its grid.
    A graph twin steps the same frames (first step eager, then capture and replay); every frame of both equals the cv2
    loop with ids kept on the host, and the twins equal each other bit for bit."""
    import torch
    B, C = case.shape(sms)
    lo, hi = case.side
    assert (lo is None or B * C > lo * sms) and (hi is None or B * C <= hi * sms), (case.name, B, C, sms)
    lk = dict(winSize=case.win, maxLevel=case.max_level, criteria=CRITERIA)
    seqs, init = case_inputs(cv2, case, B, C, seed=400 + 10 * CASES.index(case))
    check_launches(case, launches[case.name], B * C, capsys, "KLTSequenceBatch.step")
    eager, graph = make_batch(torch, seqs, init, C, lk), make_batch(torch, seqs, init, C, lk)
    assert eager._slots[0].top == case.top
    pts = list(init)
    ids = [np.arange(len(p), dtype=np.int32) for p in pts]
    next_id = [len(p) for p in pts]
    for t in range(1, FRAMES):
        frames = torch.from_numpy(np.stack([s[t] for s in seqs])).cuda()
        eager.step(frames)
        graph.step(frames)
        if t == 1:
            graph.capture()
        out, rep = snapshot(eager), snapshot(graph)
        eager.check()
        graph.check()
        for k in out:
            assert np.array_equal(out[k].view(np.uint8), rep[k].view(np.uint8)), "frame %d: graph replay differs in %s" % (t, k)
        for b in range(B):
            keep_ref, surv_ref, new_ref = cv2_step(cv2, lk, seqs[b][t - 1], seqs[b][t], pts[b], C)
            n, s, k = len(pts[b]), len(surv_ref), len(new_ref)
            tag = "%s sequence %d frame %d" % (case.name, b, t)
            assert np.array_equal(out["keep"][b, :n], keep_ref), tag + ": keep (%d of %d differ)" % (
                int((out["keep"][b, :n] != keep_ref).sum()), n)
            assert not out["keep"][b, n:].any(), tag + ": keep behind the count"
            assert int(out["counts"][b]) == s + k and int(out["n_new"][b]) == k, tag + ": counts (%d + %d expected, %d + %d)" % (
                s, k, int(out["counts"][b]) - int(out["n_new"][b]), int(out["n_new"][b]))
            assert np.array_equal(out["points"][b, :s].view(np.uint32), surv_ref.view(np.uint32)), tag + ": survivors"
            assert np.array_equal(out["points"][b, s:s + k], new_ref), tag + ": new corners"
            ids_ref = np.concatenate([ids[b][keep_ref], np.arange(next_id[b], next_id[b] + k, dtype=np.int32)])
            assert np.array_equal(out["ids"][b, :s + k], ids_ref), tag + ": ids"
            ids[b], next_id[b] = ids_ref, next_id[b] + k
            pts[b] = np.concatenate([surv_ref, new_ref])
    assert graph._graphs is not None


def test_step_batch_twin_of_case_b(klt, cv2, sms, launches, capsys):
    """KLTTracker.step_batch sizes its launch by the points tensor's width: given case b's rows (width C) frame after
    frame, it runs the same instance, and its outputs equal KLTSequenceBatch's, whose new corners are the first
    min(n_new, C - survivors) of step_batch's."""
    import torch
    from visual_odom_pipeline_b200 import tracker as T
    case = CASE_B
    B, C = case.shape(sms)
    assert B * C > 32 * sms and C % 2 == 1
    lk = dict(winSize=case.win, maxLevel=case.max_level, criteria=CRITERIA)
    seqs, init = case_inputs(cv2, case, B, C, seed=400 + 10 * CASES.index(case))
    check_launches(case, launches["step_batch"], B * C, capsys, "KLTTracker.step_batch")
    sb = make_batch(torch, seqs, init, C, lk)
    trk = T.KLTTracker(**lk).reset(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda())
    for t in range(1, FRAMES):
        frames = torch.from_numpy(np.stack([s[t] for s in seqs])).cuda()
        pts, cnt = sb.points.clone(), sb.counts.clone()
        n_in = cnt.cpu().numpy()
        out = trk.step_batch(frames, pts, cnt, max_bidir_error=30, mask_radius=10, **DET)
        nxt, ncnt, keep, n_new = [x.cpu().numpy() for x in out]
        sb.step(frames)
        got = snapshot(sb)
        sb.check()
        assert keep.shape == (B, C)
        assert np.array_equal(got["keep"], keep), "frame %d: keep" % t
        for b in range(B):
            tag = "sequence %d frame %d" % (b, t)
            s = int(keep[b].sum())
            assert not keep[b, n_in[b]:].any(), tag + ": keep behind the count"
            k = min(int(n_new[b]), C - s)
            assert int(ncnt[b]) == s + int(n_new[b]), tag + ": step_batch counts"
            assert int(got["counts"][b]) == s + k and int(got["n_new"][b]) == k, tag + ": counts"
            assert np.array_equal(got["points"][b, :s + k].view(np.uint32), nxt[b, :s + k].view(np.uint32)), tag + ": points"


if __name__ == "__main__":
    # the child process of the `launches` fixture: python tests/test_gpu_frame_step_lk_shapes.py OUT_DIR
    import sys
    import cv2
    import torch
    res = first_step_launches(torch, cv2, torch.cuda.get_device_properties(0).multi_processor_count, sys.argv[1])
    with open(os.path.join(sys.argv[1], "launches.json"), "w") as f:
        json.dump(res, f)
