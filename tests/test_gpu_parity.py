"""GPU tier (pytest -m gpu, B200): the CUDA path, called through the C ABI (ctypes), against the C
oracle, the committed golden vectors and live cv2 on the same seeded inputs.

Bars (BASELINE.json north_star): pyramid levels bit-exact; positions within 0.01 px; status identical
on >= 99.9 % of points.  The kernels reproduce OpenCV's arithmetic exactly (SURVEY.md Appendix A), so
these tests assert the stronger bit-exact property and log every mismatching point."""
import ctypes

import numpy as np
import pytest

from conftest import assert_lk_equal, load_golden
from visual_odom_pipeline_b200 import synth as S

pytestmark = pytest.mark.gpu

POS_TOL_PX = 0.01        # north_star tolerance, stated here although the expected difference is 0
STATUS_AGREE_MIN = 0.999


def crit_of(g):
    return (int(g["criteria"][0]), int(g["criteria"][1]), float(g["criteria"][2]))


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tier needs a CUDA device"
    return torch


def test_native_library_is_loaded_and_bound_to_b200(klt):
    ctx = klt.default_context(0)
    assert ctx.cc[0] == 10 and ctx.sm_count >= 100, (ctx.name, ctx.cc, ctx.sm_count)
    with open("/proc/self/maps") as f:
        assert "libklt_b200.so" in f.read()


# ---------------------------------------------------------------- pyramid ------------------------
@pytest.mark.parametrize("hw", [(376, 1241), (480, 640), (768, 1024), (135, 241), (47, 156), (33, 17), (50, 70), (2160, 3840)])
def test_pyramid_bit_exact_vs_oracle(klt, oracle, hw):
    h, w = hw
    img = S.texture(h, w, seed=h * 3 + w).astype(np.uint8)
    top, levels = klt.buildOpticalFlowPyramid(img, (5, 5), 8)
    otop, olevels = oracle.build_pyramid(img, (5, 5), 8)
    assert top == otop and len(levels) == len(olevels)
    for l, (a, b) in enumerate(zip(levels, olevels)):
        assert a.shape == b.shape and np.array_equal(a, b), "level %d of %s" % (l, hw)


def test_pyramid_matches_golden_and_cv2(klt, cv2):
    g = load_golden("pyramid")
    top, levels = klt.buildOpticalFlowPyramid(g["img"], (21, 21), 8)
    assert top == int(g["top_win21_max8"])
    top, levels = klt.buildOpticalFlowPyramid(g["img"], (3, 3), 4)
    for l, k in enumerate(("l1", "l2", "l3", "l4"), 1):
        assert np.array_equal(levels[l], g[k]), k
    ctop, clevels = cv2.buildOpticalFlowPyramid(g["img"], (21, 21), 8, None, False)
    ktop, klevels = klt.buildOpticalFlowPyramid(g["img"], (21, 21), 8)
    assert ctop == ktop and all(np.array_equal(a, b) for a, b in zip(klevels, clevels))


def test_pyramid_noncontiguous_and_constant_inputs(klt, oracle):
    big = S.texture(200, 300, seed=5).astype(np.uint8)
    view = big[3:190:1, 7:250]                      # row-strided view, like a cv2 ROI
    assert not view.flags["C_CONTIGUOUS"]
    _, lv = klt.buildOpticalFlowPyramid(view, (5, 5), 3)
    _, ol = oracle.build_pyramid(np.ascontiguousarray(view), (5, 5), 3)
    assert all(np.array_equal(a, b) for a, b in zip(lv, ol))
    for val in (0, 255):                            # saturation: 255 * 256 sums must not wrap
        _, lv = klt.buildOpticalFlowPyramid(np.full((64, 96), val, np.uint8), (5, 5), 2)
        assert all((x == val).all() for x in lv)


def test_device_pyramid_batched_aligned_and_unaligned(klt, oracle, torch_cuda):
    torch = torch_cuda
    from visual_odom_pipeline_b200 import tracker as T
    B, H, W = 5, 94, 311
    imgs = np.stack([S.texture(H, W, seed=40 + i).astype(np.uint8) for i in range(B)])
    for aligned in (True, False):
        if aligned:
            d = T.alloc_image_batch(B, H, W)
            d.copy_(torch.from_numpy(imgs))
        else:
            d = torch.from_numpy(imgs).cuda()      # W = 311: rows are not 16-byte aligned -> byte path
        pyr = T.DevicePyramid(d, (5, 5), 4)
        torch.cuda.synchronize()
        for b in range(B):
            _, ol = oracle.build_pyramid(imgs[b], (5, 5), 4)
            for l in range(pyr.top + 1):
                assert np.array_equal(pyr.level(l)[b].cpu().numpy(), ol[l]), (aligned, b, l)


# ---------------------------------------------------------------- LK -----------------------------
@pytest.mark.parametrize("name", ["lk_default", "lk_reference", "lk_hard", "lk_count_only", "lk_eps_only", "lk_mineig_flag", "lk_level0"])
def test_lk_matches_golden(klt, name):
    g = load_golden(name)
    got = klt.calcOpticalFlowPyrLK(g["prev"], g["next"], g["prevPts"], None, winSize=tuple(int(v) for v in g["winSize"]),
                                   maxLevel=int(g["maxLevel"]), criteria=crit_of(g), flags=int(g["flags"]))
    assert got[0].shape == g["nextPts"].shape and got[1].shape == g["status"].shape and got[2].shape == g["err"].shape
    assert got[0].dtype == np.float32 and got[1].dtype == np.uint8 and got[2].dtype == np.float32
    assert_lk_equal(got, (g["nextPts"], g["status"], g["err"]), name)


CONFIGS = [
    # id, h, w, n, win, maxLevel, criteria, motion, margin, extra   (BASELINE.json configs at oracle-friendly N)
    ("parking", 480, 640, 500, (21, 21), 3, (3, 30, 0.01), S.BENIGN, 0, {}),
    ("kitti", 376, 1241, 2000, (21, 21), 3, (3, 30, 0.01), S.BENIGN, 0, {}),
    ("kitti_ref_params", 376, 1241, 2000, (31, 31), 3, (3, 30, 0.03), S.BENIGN, 0, {}),
    ("kitti_hard", 376, 1241, 2000, (21, 21), 3, (3, 30, 0.01), S.HARD, 60, dict(noise_sigma=3.0, flat_cols=(400, 700))),
    ("kitti_hard31", 376, 1241, 2000, (31, 31), 3, (3, 30, 0.03), S.HARD, 60, dict(noise_sigma=3.0, flat_cols=(400, 700))),
    ("malaga", 768, 1024, 3000, (21, 21), 3, (3, 30, 0.01), S.BENIGN, 0, {}),
    ("nonsquare", 240, 320, 400, (20, 12), 3, (3, 30, 0.01), S.HARD, 30, {}),
    ("tall_win", 240, 320, 400, (13, 29), 3, (3, 30, 0.01), S.HARD, 30, {}),
    ("win3", 240, 320, 400, (3, 3), 3, (3, 30, 0.01), S.HARD, 30, {}),
    ("win8", 240, 320, 400, (8, 8), 3, (3, 30, 0.01), S.HARD, 30, {}),
    ("win40", 240, 320, 400, (40, 40), 3, (3, 30, 0.01), S.HARD, 30, {}),
    ("win64", 240, 320, 200, (64, 64), 3, (3, 30, 0.01), S.HARD, 30, {}),
    ("truncated_pyr", 376, 1241, 500, (21, 21), 8, (3, 30, 0.01), S.BENIGN, 30, {}),
    ("level0_only", 376, 1241, 500, (21, 21), 0, (3, 30, 0.01), S.BENIGN, 30, {}),
    ("count_only", 240, 320, 400, (21, 21), 3, (1, 10, 0.01), S.BENIGN, 30, {}),
    ("eps_only", 240, 320, 400, (21, 21), 3, (2, 30, 0.05), S.BENIGN, 30, {}),
    ("clamped_crit", 240, 320, 400, (21, 21), 3, (3, 200, 20.0), S.BENIGN, 30, {}),
    ("zero_iters", 240, 320, 400, (21, 21), 3, (3, 0, 0.01), S.BENIGN, 30, {}),
    ("tiny_image", 50, 70, 100, (21, 21), 3, (3, 30, 0.01), S.BENIGN, 30, {}),
]


@pytest.mark.parametrize("case", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_lk_bit_exact_vs_oracle_and_cv2(klt, oracle, cv2, case):
    _, h, w, n, win, lvl, crit, motion, margin, kw = case
    a, b = S.frame_pair(h, w, seed=7, motion=motion, **kw)
    p = S.uniform_points(n, h, w, seed=3, margin=margin)
    got = klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=win, maxLevel=lvl, criteria=crit)
    want = oracle.calc_optical_flow_pyr_lk(a, b, p, None, win, lvl, crit)
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=win, maxLevel=lvl, criteria=crit)
    # the north-star gates first (tolerances stated), then the stronger bit-exact check
    agree = (got[1] == ref[1]).mean()
    assert agree >= STATUS_AGREE_MIN, "status agreement %.5f" % agree
    both = ((got[1] == 1) & (ref[1] == 1)).ravel()
    if both.any():
        assert np.abs(got[0].reshape(-1, 2)[both] - ref[0].reshape(-1, 2)[both]).max() <= POS_TOL_PX
    assert_lk_equal(got, want, "vs oracle")
    assert_lk_equal(got, ref, "vs cv2")


@pytest.mark.parametrize("wpp", ["1", "2", "4"], ids=["wpp1", "wpp2", "wpp4"])
def test_lk_team_sizes_bit_exact(klt, wpp):
    """Every team size of the specialised kernel (1, 2 or 4 warps per keypoint) ships in the library and is picked by
    window / point count: same bit-exactness bar for each, forced through KLT_LK_WPP."""
    import os, subprocess, sys
    e = dict(os.environ)
    e["KLT_LK_WPP"] = wpp
    r = subprocess.run([sys.executable, os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lk_variant_check.py")], env=e,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_lk_one_pass_grid_bit_exact(klt):
    """Single-pair launches of the 4-warp shape dispatch the points near the image border first (a grid that holds every
    point twice); KLT_LK_TWO_PASS=0 is the plain grid.  Both orders must give cv2's bits -- the default order is what
    every other test of this file runs."""
    import os, subprocess, sys
    e = dict(os.environ)
    e["KLT_LK_TWO_PASS"] = "0"
    e["KLT_LK_WPP"] = "4"
    r = subprocess.run([sys.executable, os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lk_variant_check.py")], env=e,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_lk_point_layouts_and_special_points(klt, cv2):
    a, b = S.frame_pair(120, 160, seed=2)
    base = S.uniform_points(40, 120, 160, seed=9)
    for shape in [(40, 1, 2), (40, 2), (1, 40, 2)]:
        p = base.reshape(shape)
        got = klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
        ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
        assert got[0].shape == ref[0].shape == shape and got[1].shape == ref[1].shape and got[2].shape == ref[2].shape
        assert_lk_equal(got, ref, str(shape))
    p = np.array([[np.nan, 10], [1e9, 1e9], [-500, 20], [0, 0], [159.9, 119.9], [80, 60], [-10.5, -10.5], [np.inf, 3]], np.float32).reshape(-1, 1, 2)
    got = klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    assert np.array_equal(got[1], ref[1])
    fin = np.isfinite(ref[0]).all(-1).ravel()
    assert np.array_equal(got[0].reshape(-1, 2)[fin].view(np.uint32), ref[0].reshape(-1, 2)[fin].view(np.uint32))
    assert np.array_equal(np.isnan(got[0]), np.isnan(ref[0]))
    one = klt.calcOpticalFlowPyrLK(a, b, base[:1], None)
    assert_lk_equal(one, cv2.calcOpticalFlowPyrLK(a, b, base[:1], None), "N=1")
    assert klt.calcOpticalFlowPyrLK(a, b, base[:0], None) == (None, None, None)


def test_lk_initial_flow_flag(klt, cv2):
    a, b = S.frame_pair(120, 160, seed=4)
    p = S.uniform_points(50, 120, 160, seed=1)
    guess = (p + np.float32(2.0)).astype(np.float32)
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, guess.copy(), winSize=(21, 21), maxLevel=2, criteria=(3, 30, 0.01), flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
    got = klt.calcOpticalFlowPyrLK(a, b, p, guess.copy(), winSize=(21, 21), maxLevel=2, criteria=(3, 30, 0.01), flags=klt.OPTFLOW_USE_INITIAL_FLOW)
    assert_lk_equal(got, ref)


def test_inputs_not_mutated_and_outputs_fresh(klt):
    a, b = S.frame_pair(96, 128, seed=6)
    p = S.uniform_points(30, 96, 128, seed=2)
    a0, b0, p0 = a.copy(), b.copy(), p.copy()
    r1 = klt.calcOpticalFlowPyrLK(a, b, p, None)
    r2 = klt.calcOpticalFlowPyrLK(a, b, p, None)
    assert np.array_equal(a, a0) and np.array_equal(b, b0) and np.array_equal(p, p0)
    assert r1[0] is not r2[0] and np.array_equal(r1[0], r2[0]) and np.array_equal(r1[1], r2[1])


def test_reference_call_pattern_extend_tracks(klt, cv2):
    """The exact sequence of reference src/extractor/extractor.py:43-57 (forward call, second call from
    the result, bidirectional distance, inclusive bounds filter) gives the same survivors."""
    lk = dict(winSize=(31, 31), maxLevel=3, criteria=(cv2.TERM_CRITERIA_EPS | cv2.TERM_CRITERIA_COUNT, 30, 0.03))
    im0, im1 = S.frame_pair(376, 1241, seed=12)
    uv = S.uniform_points(600, 376, 1241, seed=8).reshape(-1, 2)
    p0 = np.float32([u.reshape(2, 1).T for u in uv]).reshape(-1, 1, 2)

    def run(fn):
        p1, _st, _err = fn(im0, im1, p0, None, **lk)
        p0r, _st, _err = fn(im0, im1, p1, None, **lk)
        d = abs(p0 - p0r).reshape(-1, 2).max(-1)
        good = d < np.inf
        keep = [i for i, ((x, y), g) in enumerate(zip(p1.reshape(-1, 2), good)) if g and 0 <= x <= im1.shape[1] and 0 <= y <= im1.shape[0]]
        return p1, p0r, keep
    a, b = run(cv2.calcOpticalFlowPyrLK), run(klt.calcOpticalFlowPyrLK)
    assert a[2] == b[2]
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32)) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))


@pytest.mark.parametrize("max_err", [np.inf, 30, 28.5])
def test_fused_tracking_step_equals_reference_pattern(klt, cv2, max_err):
    """klt.trackBidirectional = the cv2 sequence of reference src/extractor/extractor.py:43-53 / :64-75 in one call:
    p1 bit-exact, bidirectional distance bit-exact, survivor mask identical (hard motion + out-of-frame points)."""
    lk = dict(winSize=(31, 31), maxLevel=3, criteria=(cv2.TERM_CRITERIA_EPS | cv2.TERM_CRITERIA_COUNT, 30, 0.03))
    im0, im1 = S.frame_pair(240, 320, seed=5, motion=S.HARD)
    p0 = S.uniform_points(700, 240, 320, seed=9, margin=25)          # some points start outside the frame
    p0[3, 0, 0] = np.nan
    p1, st, er = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **lk)
    p0r, _, _ = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **lk)
    with np.errstate(invalid="ignore"):
        d = abs(p0 - p0r).reshape(-1, 2).max(-1)
        good = d < max_err
    x, y = p1.reshape(-1, 2).T
    want = good & (0 <= x) & (x <= im1.shape[1]) & (0 <= y) & (y <= im1.shape[0])
    q1, keep, bd, st2, er2 = klt.trackBidirectional(im0, im1, p0, max_bidir_error=max_err, **lk)
    assert q1.shape == p0.shape and keep.dtype == np.bool_ and keep.shape == (700,)
    fin = np.isfinite(p1).all(-1).ravel()
    assert np.array_equal(q1.reshape(-1, 2)[fin].view(np.uint32), p1.reshape(-1, 2)[fin].view(np.uint32))
    assert np.array_equal(st2, st)
    m = st.ravel() == 1
    assert np.array_equal(er2.ravel()[m].view(np.uint32), er.ravel()[m].view(np.uint32))
    both = np.isfinite(d) & np.isfinite(bd)
    assert np.array_equal(np.isfinite(d), np.isfinite(bd))
    assert np.array_equal(bd[both].view(np.uint32), d[both].astype(np.float32).view(np.uint32))
    assert np.array_equal(keep, want), "survivors differ at %s" % np.nonzero(keep != want)[0][:10]
    assert want.sum() > 0 or max_err != np.inf
    assert klt.trackBidirectional(im0, im1, np.empty((0, 1, 2), np.float32)) == (None,) * 5


def test_device_track_filtered_equals_host_fused_step(klt, torch_cuda):
    torch = torch_cuda
    from visual_odom_pipeline_b200 import tracker as T
    lk = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    pairs = [S.frame_pair(120, 160, seed=30 + i, motion=S.HARD if i % 2 else S.BENIGN) for i in range(3)]
    pts = np.stack([S.uniform_points(150, 120, 160, seed=40 + i, margin=15).reshape(-1, 2) for i in range(3)])
    trk = T.KLTTracker(**lk).reset(torch.from_numpy(np.stack([a for a, _ in pairs])).cuda())
    p1, keep, bd, st, er = trk.track_filtered(torch.from_numpy(np.stack([b for _, b in pairs])).cuda(), torch.from_numpy(pts).cuda(), max_bidir_error=5.0)
    for i, (a, b) in enumerate(pairs):
        h1, hk, hb, hs, he = klt.trackBidirectional(a, b, pts[i], max_bidir_error=5.0, **lk)
        assert np.array_equal(p1[i].cpu().numpy().view(np.uint32), h1.view(np.uint32))
        assert np.array_equal(keep[i].cpu().numpy(), hk)
        assert np.array_equal(bd[i].cpu().numpy().view(np.uint32), hb.view(np.uint32))
        assert np.array_equal(st[i].cpu().numpy(), hs.ravel())


# ---------------------------------------------------------------- device / batch API -------------
def test_batched_device_api_equals_per_pair_host_calls(klt, oracle, torch_cuda):
    torch = torch_cuda
    from visual_odom_pipeline_b200 import tracker as T
    B, H, W, N = 6, 188, 621, 300
    pairs = [S.frame_pair(H, W, seed=70 + i) for i in range(B)]
    pts = np.stack([S.uniform_points(N, H, W, seed=i, margin=20).reshape(N, 2) for i in range(B)])
    prev = T.alloc_image_batch(B, H, W); prev.copy_(torch.from_numpy(np.stack([p[0] for p in pairs])))
    nxt = T.alloc_image_batch(B, H, W); nxt.copy_(torch.from_numpy(np.stack([p[1] for p in pairs])))
    P0 = T.DevicePyramid(prev, (21, 21), 3)
    P1 = T.DevicePyramid(nxt, (21, 21), 3)
    q, st, er, it = T.lk_track(P0, P1, torch.from_numpy(pts).cuda(), criteria=(3, 30, 0.01), return_iters=True)
    torch.cuda.synchronize()
    for b in range(B):
        want = oracle.calc_optical_flow_pyr_lk(pairs[b][0], pairs[b][1], pts[b], None, (21, 21), 3, (3, 30, 0.01), return_iters=True)
        assert_lk_equal((q[b].cpu().numpy(), st[b].cpu().numpy(), er[b].cpu().numpy()), want[:3], "pair %d" % b)
        assert np.array_equal(it[b].cpu().numpy(), want[3]), "iteration counts, pair %d" % b


def test_torch_tensor_dropin_and_tracker_sequence(klt, cv2, torch_cuda):
    torch = torch_cuda
    from visual_odom_pipeline_b200 import tracker as T
    frames = S.sequence(120, 160, 5, seed=31)
    p = S.uniform_points(80, 120, 160, seed=4)
    # drop-in with CUDA tensors
    got = klt.calcOpticalFlowPyrLK(torch.from_numpy(frames[0]).cuda(), torch.from_numpy(frames[1]).cuda(), torch.from_numpy(p).cuda(), None,
                                   winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
    ref = cv2.calcOpticalFlowPyrLK(frames[0], frames[1], p, None, winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
    assert tuple(got[0].shape) == ref[0].shape
    assert_lk_equal(tuple(t.cpu().numpy() for t in got), ref)
    # tracker keeps the pyramid of the last frame: same results as pairwise cv2 calls
    trk = T.KLTTracker(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03)).reset(torch.from_numpy(frames[0]).cuda())
    cur = p.copy()
    for t in range(1, len(frames)):
        q, st, er, back = trk.track(torch.from_numpy(frames[t]).cuda(), torch.from_numpy(cur.reshape(1, -1, 2)).cuda(), bidirectional=True)
        ref = cv2.calcOpticalFlowPyrLK(frames[t - 1], frames[t], cur, None, winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
        refb = cv2.calcOpticalFlowPyrLK(frames[t - 1], frames[t], ref[0], None, winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
        assert_lk_equal((q.cpu().numpy(), st.cpu().numpy(), er.cpu().numpy()), ref, "frame %d" % t)
        assert np.array_equal(back.cpu().numpy().reshape(-1, 2).view(np.uint32), refb[0].reshape(-1, 2).view(np.uint32))
        cur = ref[0]


# ---------------------------------------------------------------- full-size properties -----------
def test_full_size_stress_config_vs_cv2_and_properties(klt, cv2):
    """BASELINE configs[4]: 3840x2160, dense grid ~100k points, win 31, maxLevel 5 (too big for the scalar
    oracle in seconds -> live cv2 is the checker, plus size-independent properties)."""
    h, w = 2160, 3840
    a, b = S.frame_pair(h, w, seed=7)
    p = S.grid_points(422, 237, h, w)
    assert p.shape[0] == 100014
    got = klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=(31, 31), maxLevel=5, criteria=(3, 30, 0.01))
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=(31, 31), maxLevel=5, criteria=(3, 30, 0.01))
    assert_lk_equal(got, ref, "4K")
    again = klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=(31, 31), maxLevel=5, criteria=(3, 30, 0.01))
    assert all(np.array_equal(x, y) for x, y in zip(got, again)), "not deterministic"
    perm = np.random.default_rng(0).permutation(p.shape[0])          # per-point independence
    shuf = klt.calcOpticalFlowPyrLK(a, b, p[perm], None, winSize=(31, 31), maxLevel=5, criteria=(3, 30, 0.01))
    assert np.array_equal(shuf[0], got[0][perm]) and np.array_equal(shuf[1], got[1][perm])


def test_integer_shift_is_recovered_at_kitti_size(klt):
    """Property: next = prev shifted by whole pixels -> interior points move by exactly that shift
    (to the eps of the criteria), independent of any reference implementation."""
    h, w = 376, 1241
    base = S.texture(h + 16, w + 16, seed=3).astype(np.uint8)
    prev = np.ascontiguousarray(base[8:8 + h, 8:8 + w])
    dx, dy = 5, -3
    nxt = np.ascontiguousarray(base[8 - dy:8 - dy + h, 8 - dx:8 - dx + w])
    p = S.uniform_points(2000, h - 80, w - 80, seed=1) + np.float32(40)
    q, st, er = klt.calcOpticalFlowPyrLK(prev, nxt, p, None, winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    ok = st.ravel() == 1
    assert ok.mean() > 0.98
    d = (q - p).reshape(-1, 2)[ok]
    assert np.abs(d - np.array([dx, dy], np.float32)).max() < 0.05
    assert (er.ravel()[ok] < 1.0).all()


def test_pyramid_levels_match_cv2_pyrdown(klt):
    """Every level up to maxLevel 6 equals cv2.pyrDown applied level by level."""
    import cv2
    for hw in [(376, 1241), (480, 640), (135, 241), (97, 203), (2160, 3840)]:
        img = S.texture(hw[0], hw[1], seed=hw[1]).astype(np.uint8)
        top, levels = klt.buildOpticalFlowPyramid(img, (5, 5), 6)
        ref = img
        for l in range(1, top + 1):
            ref = cv2.pyrDown(ref)
            assert np.array_equal(levels[l], ref), (hw, l)


def test_second_device_in_the_same_process(klt, cv2):
    """One process driving two GPUs (a context per device): the kernels' dynamic shared-memory opt-in is per device."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    a, b = S.frame_pair(376, 1241, seed=8)
    p = S.uniform_points(500, 376, 1241, seed=9)
    lk = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk)
    refc = cv2.goodFeaturesToTrack(a, 1000, 0.03, 10, blockSize=31)
    for dev in (0, 1, 0, 1):
        assert_lk_equal(klt.calcOpticalFlowPyrLK(a, b, p, None, device=dev, **lk), ref, "device %d" % dev)
        got = klt.goodFeaturesToTrack(a, 1000, 0.03, 10, blockSize=31, device=dev)
        assert got.shape == refc.shape and np.array_equal(got, refc)


# ---------------------------------------------------------------- host-path properties of round 2 -----------
def test_pageable_and_pinned_inputs_give_the_same_results(klt, cv2):
    """Pageable numpy arrays (what the un-edited reference passes: loader.py:86, pipeline.py:103) are staged by the helper
    threads of the context, pinned ones are DMA'd in place; odd sizes exercise the slice boundaries of the staging copy."""
    lk = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    for (h, w, n) in [(376, 1241, 700), (601, 1000, 300), (768, 1024, 300)]:
        a, b = S.frame_pair(h, w, seed=h)
        p = S.uniform_points(n, h, w, seed=w)
        ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk)
        pa, pb, pp = klt.pinned_empty(a.shape), klt.pinned_empty(b.shape), klt.pinned_empty(p.shape, np.float32)
        pa[...] = a; pb[...] = b; pp[...] = p
        for _ in range(3):      # the helpers are started by the first call, asleep or spinning afterwards
            assert_lk_equal(klt.calcOpticalFlowPyrLK(a, b, p, None, **lk), ref, "pageable %dx%d" % (w, h))
        assert_lk_equal(klt.calcOpticalFlowPyrLK(pa, pb, pp, None, **lk), ref, "pinned %dx%d" % (w, h))
        assert_lk_equal(klt.calcOpticalFlowPyrLK(a, pb, p, None, **lk), ref, "mixed %dx%d" % (w, h))
    import time
    time.sleep(0.01)            # helpers have gone to sleep on their condition variable: the next job wakes them
    assert_lk_equal(klt.calcOpticalFlowPyrLK(a, b, p, None, **lk), ref, "after sleep")


def test_concurrent_callers_share_one_context(klt, cv2):
    """A klt_ctx serialises its *_host entry points internally (include/klt_b200.h): threads calling the drop-in at the
    same time -- LK, the fused bidirectional step and detection, all on the shared default context -- get the same
    results as cv2."""
    import threading
    lk = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    jobs = []
    for i in range(4):
        a, b = S.frame_pair(240, 320 + 16 * i, seed=40 + i)
        p = S.uniform_points(200, 240, 320 + 16 * i, seed=50 + i)
        jobs.append((a, b, p, cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk)))
    errors = []

    def work(job):
        try:
            for _ in range(20):
                assert_lk_equal(klt.calcOpticalFlowPyrLK(job[0], job[1], job[2], None, **lk), job[3])
        except Exception as ex:   # noqa: BLE001
            errors.append(ex)

    def bidirectional_ref(a, b, p, ref):   # the cv2 sequence of extractor.py:43-53
        p0r = cv2.calcOpticalFlowPyrLK(a, b, ref[0], None, **lk)[0]
        d = abs(p - p0r).reshape(-1, 2).max(-1)
        x, y = ref[0].reshape(-1, 2).T
        return a, b, p, ref, (d < 30) & (0 <= x) & (x <= a.shape[1]) & (0 <= y) & (y <= a.shape[0]), d

    def work_bidirectional(a, b, p, ref, want_keep, want_d):
        try:
            for _ in range(20):
                q1, keep, d, st, er = klt.trackBidirectional(a, b, p, 30, **lk)
                assert_lk_equal((q1, st, er), ref)
                assert np.array_equal(d, want_d, equal_nan=True) and np.array_equal(keep, want_keep)
        except Exception as ex:   # noqa: BLE001
            errors.append(ex)

    def work_detection(img, want):
        try:
            for _ in range(20):
                got = klt.goodFeaturesToTrack(img, 500, 0.03, 10, blockSize=15)
                assert got.shape == want.shape and np.array_equal(got, want)
        except Exception as ex:   # noqa: BLE001
            errors.append(ex)
    ts = [threading.Thread(target=work, args=(j,)) for j in jobs]
    ts += [threading.Thread(target=work_bidirectional, args=bidirectional_ref(*j)) for j in jobs[:2]]
    ts += [threading.Thread(target=work_detection, args=(j[1], cv2.goodFeaturesToTrack(j[1], 500, 0.03, 10, blockSize=15)))
           for j in jobs[2:]]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errors, errors[:1]


def test_tracker_owns_its_frames(klt, cv2, torch_cuda):
    """KLTTracker copies every frame into storage of its own: the caller may upload frame t+1 into the SAME device tensor."""
    torch = torch_cuda
    from visual_odom_pipeline_b200 import tracker as T
    lk = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    frames = S.sequence(120, 160, 4, seed=77)
    p = S.uniform_points(60, 120, 160, seed=5)
    buf = torch.from_numpy(frames[0]).cuda()
    trk = T.KLTTracker(**lk).reset(buf)
    cur = p.copy()
    for t in range(1, len(frames)):
        buf.copy_(torch.from_numpy(frames[t]))            # overwrites what reset() / the last track() was given
        q, st, er = trk.track(buf, torch.from_numpy(cur.reshape(1, -1, 2)).cuda())
        ref = cv2.calcOpticalFlowPyrLK(frames[t - 1], frames[t], cur, None, **lk)
        assert_lk_equal((q.cpu().numpy(), st.cpu().numpy(), er.cpu().numpy()), ref, "frame %d" % t)
        cur = ref[0]


def test_calls_do_not_change_the_current_device(klt, torch_cuda):
    """The C ABI makes its context's device current for the duration of a call only."""
    torch = torch_cuda
    a, b = S.frame_pair(120, 160, seed=3)
    p = S.uniform_points(30, 120, 160, seed=4)
    before = torch.cuda.current_device()
    klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=(21, 21), maxLevel=2, device=0)
    klt.goodFeaturesToTrack(a, 100, 0.03, 10, blockSize=15, device=0)
    assert torch.cuda.current_device() == before
    if torch.cuda.device_count() >= 2:
        from visual_odom_pipeline_b200 import tracker as T
        klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=(21, 21), maxLevel=2, device=1)
        assert torch.cuda.current_device() == before
        # device-pointer entry points on tensors of cuda:1 while cuda:0 is current
        ta, tb = torch.from_numpy(a).to("cuda:1"), torch.from_numpy(b).to("cuda:1")
        q, st, er = T.calc_optical_flow_pyr_lk_device(ta, tb, torch.from_numpy(p).to("cuda:1"), None, winSize=(21, 21), maxLevel=2)
        ref = klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=(21, 21), maxLevel=2, device=0)
        assert_lk_equal((q.cpu().numpy(), st.cpu().numpy(), er.cpu().numpy()), ref)
        assert torch.cuda.current_device() == before


def test_pyramid_reuse_across_calls_detects_changed_images(klt, cv2):
    """The host entry point keeps the pyramids of its last call and skips the build of an image whose content hash (computed
    on the device from the uploaded bytes) is unchanged -- the reference passes the same pair four times per frame
    (extractor.py:44,45,65,66).  Hashing is switched on while the caller keeps passing the same two arrays: the first repeat
    records the hashes, the following calls skip.  Results never depend on it: edits in place, new pairs, other geometries
    and calls that overwrite the workspace in between are all detected."""
    import ctypes
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    ctx = klt.default_context(0)
    L.klt_debug_pyr_reuse_count.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_ulonglong)]
    L.klt_debug_pyr_reuse_count.restype = ctypes.c_int

    def skipped():
        v = ctypes.c_ulonglong()
        assert L.klt_debug_pyr_reuse_count(ctx.handle, ctypes.byref(v)) == 0
        return v.value
    lk = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.03))
    a, b = S.frame_pair(376, 1241, seed=61)
    c = S.frame_pair(376, 1241, seed=62)[1]
    p = S.uniform_points(400, 376, 1241, seed=63)

    def call(x, y, pts, what, kw=lk):
        assert_lk_equal(klt.calcOpticalFlowPyrLK(x, y, pts, None, **kw), cv2.calcOpticalFlowPyrLK(x, y, pts, None, **kw), what)
    call(c, c, p, "some other pair first")
    s0 = skipped()
    call(a, b, p, "call 1 of the frame")               # new arrays: no hashing
    call(a, b, p, "call 2: same arrays")               # hashes recorded, both pyramids built
    assert skipped() == s0
    p1 = cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk)[0][:333]
    call(a, b, p1, "call 3: same arrays, other points")
    assert skipped() == s0 + 2
    call(a, b, p, "call 4")
    assert skipped() == s0 + 4
    # one pixel of the next image edited IN PLACE: same array object, same address
    b[100, 200] ^= 0x40
    call(a, b, p, "edited in place")
    assert skipped() == s0 + 5                                          # only the previous image was kept
    b[375, 1240] ^= 0x01                                                # the last pixel of the last row
    call(a, b, p, "last pixel edited")
    assert skipped() == s0 + 6
    call(a, b, p, "unchanged again")
    assert skipped() == s0 + 8
    # next frame: (b, c) -- other arrays: no hashing on the first call, nothing to compare with on the second
    call(b, c, p, "next frame, call 1")
    call(b, c, p, "next frame, call 2")
    assert skipped() == s0 + 8
    call(b, c, p, "next frame, call 3")
    assert skipped() == s0 + 10
    # another window size (same arrays): another pyramid depth rule -> never reused across parameter sets
    lk21 = dict(winSize=(21, 21), maxLevel=2, criteria=(3, 30, 0.01))
    call(b, c, p, "other parameters", lk21)
    assert skipped() == s0 + 10
    call(b, c, p, "back to the first parameters")
    assert skipped() == s0 + 10
    call(b, c, p, "and again")
    assert skipped() == s0 + 12
    # every other host call overwrites the workspace: the same pair is rebuilt after it, and skipped again on the next call
    overwriting = [("detection", lambda: klt.goodFeaturesToTrack(b, 500, 0.03, 10, blockSize=31)),
                   ("buildOpticalFlowPyramid", lambda: klt.buildOpticalFlowPyramid(b, (31, 31), 3)),
                   ("cornerMinEigenVal", lambda: klt.cornerMinEigenVal(b, 31)),
                   ("bilateralFilter", lambda: klt.bilateralFilter(b, 5, 1.5, 1.5)),
                   ("detectNewFeatures", lambda: klt.detectNewFeatures(b, p, 10))]
    n = s0 + 12
    for what, overwrite in overwriting:
        overwrite()
        call(b, c, p, "after " + what)
        assert skipped() == n, what
        call(b, c, p, "after %s, again" % what)
        n += 2
        assert skipped() == n, what
    # fused bidirectional call shares the mechanism
    got = klt.trackBidirectional(b, c, p, 30, **lk)
    assert_lk_equal((got[0], got[3], got[4]), cv2.calcOpticalFlowPyrLK(b, c, p, None, **lk), "bidirectional")
    assert skipped() == n + 2


def test_lk_windows_larger_than_the_image(klt, cv2):
    """Regression (found by tests/test_gpu_random.py): on a 12 x 12 white-noise image with a 21 x 21 window almost the whole
    gradient energy of a window sits in one or two threads of the team; the per-thread clamp of the exactness bounds used to
    be 2^25 / WPP, so for the 4-warp team a clamped thread no longer proved "not exact" and one float32 sum was taken from the
    integer total although OpenCV's partial sums round."""
    rng = np.random.default_rng(0)
    for (h, w, win) in [(12, 12, (21, 21)), (12, 12, (31, 31)), (9, 40, (21, 21)), (25, 25, (31, 31))]:
        a = rng.integers(0, 256, (h, w), dtype=np.uint8)
        b = np.roll(a, (0, 1), axis=(0, 1))
        p = np.stack([rng.uniform(-8, w + 8, 200), rng.uniform(-8, h + 8, 200)], -1).astype(np.float32).reshape(-1, 1, 2)
        for lvl in (0, 2):
            ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=win, maxLevel=lvl, criteria=(3, 30, 0.01))
            assert_lk_equal(klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=win, maxLevel=lvl, criteria=(3, 30, 0.01)), ref,
                            "%dx%d win %s level %d" % (w, h, win, lvl))


def test_pyramid_and_lk_replay_from_a_cuda_graph(klt, cv2, torch_cuda):
    """The device-pointer entry points are plain launches once their scratch exists (the one-launch pyramid build keeps its
    launch counter on the device), so a frame's work -- both pyramids + LK -- can be captured once and replayed from a CUDA
    graph with new frame contents in the same buffers."""
    torch = torch_cuda
    from visual_odom_pipeline_b200 import tracker as T
    h, w, win, crit = 240, 320, (21, 21), (3, 30, 0.01)
    frames = S.sequence(h, w, 5, seed=12)
    a, b = T.alloc_image_batch(1, h, w), T.alloc_image_batch(1, h, w)
    a[0].copy_(torch.from_numpy(frames[0])); b[0].copy_(torch.from_numpy(frames[1]))
    pts = torch.from_numpy(S.uniform_points(300, h, w, seed=2).reshape(1, -1, 2)).cuda()
    P0, P1 = T.DevicePyramid(a, win, 3), T.DevicePyramid(b, win, 3)
    assert P0.top >= 2                                   # the one-launch build is the path under test
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                        # warm-up on the capture stream: scratch is allocated per stream
        for _ in range(2):
            P0.build(); P1.build()
            T.lk_track(P0, P1, pts, criteria=crit)
    side.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        P0.build(); P1.build()
        q, st, er = T.lk_track(P0, P1, pts, criteria=crit)
    for t in range(1, len(frames)):
        a[0].copy_(torch.from_numpy(frames[t - 1])); b[0].copy_(torch.from_numpy(frames[t]))
        p_h = S.uniform_points(300, h, w, seed=20 + t)
        pts.copy_(torch.from_numpy(p_h.reshape(1, -1, 2)))
        torch.cuda.synchronize()
        for _ in range(2):                               # replayed twice: the counters of the pyramid build keep advancing
            g.replay()
        torch.cuda.synchronize()
        ref = cv2.calcOpticalFlowPyrLK(frames[t - 1], frames[t], p_h, None, winSize=win, maxLevel=3, criteria=crit)
        assert_lk_equal((q.cpu().numpy(), st.cpu().numpy(), er.cpu().numpy()), ref, "replay %d" % t)
