"""GPU tier (pytest -m gpu, B200) of the generic LK kernel (lk_kernel, csrc/klt_lk.cu), which serves every window but
21x21 and 31x31: every window shape the header accepts, against cv2 and the CPU oracle bit for bit.

- The window sweep runs the largest and most elongated windows, at 4, 3 and 2 warps per CTA, and the refusals.
- The replay cases drive each of the kernel's serial float32 replays (G, b, err) at points where the integer shortcut
  would give another output bit (tests/test_lk_windows_cpu.py shows that without a GPU).
- The batched device path runs at each warp count, with per-pair iteration counts, and the frame step with ragged counts.
- The minEigThreshold gate is tested at its float32 boundary, in both kernels."""
import numpy as np
import pytest

from conftest import assert_lk_equal
from test_lk_windows_cpu import REPLAY_CASES, REPLAY_MIN, shortcut_vs_cv2
from visual_odom_pipeline_b200 import synth as S

pytestmark = pytest.mark.gpu

B200_SMEM_OPTIN = 232448          # bytes of opt-in shared memory per block on a B200 (227 KB)

WINDOWS = [
    # window, warps per CTA lk_launch picks on a B200 (the most of 4 whose shared-memory slices fit B200_SMEM_OPTIN)
    ((42, 42), 4),                 # the first size above the randomised tests' range
    ((45, 45), 4), ((46, 46), 4),  # either side of the 2056-px area past which err may need its replay
    ((63, 65), 4), ((64, 64), 4),  # area 4095 and 4096
    ((128, 32), 4), ((32, 128), 4),
    ((504, 8), 4), ((504, 3), 4),  # the widest windows: 64 eight-pixel runs per derivative row
    ((50, 81), 4),                 # scalar tail of 2
    ((8, 504), 3), ((3, 483), 3), ((41, 96), 3), ((35, 115), 3),
    ((9, 455), 2), ((11, 372), 2),
]
REFUSED = [(64, 65), (505, 8), (1000, 4)]


def warp_bytes(win_w, win_h, margin=3):
    """make_geom (csrc/klt_lk.cu): shared memory of one warp's slice."""
    ru = lambda v, a: (v + a - 1) // a * a
    pw = 8 * ((win_w + 7) // 8)
    sj = ru(pw + 2 * margin + 2, 4)
    off = ru(2 * pw * win_h, 16) + ru(4 * pw * win_h, 16) + ru(sj * (win_h + 1 + 2 * margin), 16)
    ireg, dreg, diff = ru((pw + 12) * (win_h + 3), 16), ru(4 * (pw + 1) * (win_h + 1), 16), ru(2 * pw * win_h, 16)
    return ru(off + max(ireg + dreg, diff), 128)


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def b200(klt):
    import torch
    assert torch.cuda.get_device_properties(0).shared_memory_per_block_optin == B200_SMEM_OPTIN
    return torch


def border_points(n, h, w, seed):
    """n points over the image and a 30-px band around it: some windows overlap the border, some points lie outside."""
    rng = np.random.default_rng(seed)
    return np.stack([rng.uniform(-30, w + 30, n), rng.uniform(-30, h + 30, n)], -1).astype(np.float32).reshape(-1, 1, 2)


def check_all(klt, oracle, cv2, a, b, p, win, what, **lk):
    got = klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=win, **lk)
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=win, **lk)
    want = oracle.calc_optical_flow_pyr_lk(a, b, p, None, win, lk["maxLevel"], lk["criteria"], flags=lk.get("flags", 0),
                                           min_eig_threshold=lk.get("minEigThreshold", 1e-4))
    assert_lk_equal(got, ref, what + " vs cv2")
    assert_lk_equal(got, want, what + " vs oracle")
    return got


# ---- a. window sweep ---------------------------------------------------------------------------
@pytest.mark.parametrize("win,warps", WINDOWS, ids=["%dx%d_%dwarps" % (w[0], w[1], k) for w, k in WINDOWS])
def test_window_sweep_bit_exact(klt, oracle, cv2, b200, win, warps):
    assert min(4, B200_SMEM_OPTIN // warp_bytes(*win)) == warps
    for h, w in ((376, 1241), (768, 1024)):
        for seed, motion in ((7, S.BENIGN), (8, S.HARD)):
            a, b = S.frame_pair(h, w, seed=seed, motion=motion)
            p = border_points(300, h, w, seed)
            check_all(klt, oracle, cv2, a, b, p, win, "%dx%d %dx%d seed %d" % (win + (w, h, seed)),
                      maxLevel=3, criteria=(3, 30, 0.01))


@pytest.mark.parametrize("win", REFUSED, ids=["%dx%d" % w for w in REFUSED])
def test_windows_past_the_limits_are_refused(klt, cv2, b200, win):
    """cv2 accepts these windows; the library raises its error (a cv2.error) with the unsupported status."""
    import re
    from visual_odom_pipeline_b200 import _lib
    a, b = S.frame_pair(120, 160, seed=1)
    p = S.uniform_points(16, 120, 160, seed=2)
    assert cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=win, maxLevel=0)[1].shape == (16, 1)
    with pytest.raises(klt.error, match=re.escape(_lib.status_string(_lib.KLT_ERR_UNSUPPORTED))) as e:
        klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=win, maxLevel=0)
    assert isinstance(e.value, cv2.error)
    # the library still works afterwards
    assert_lk_equal(klt.calcOpticalFlowPyrLK(a, b, p, None, winSize=(21, 21)), cv2.calcOpticalFlowPyrLK(a, b, p, None))


# ---- b. the replays ----------------------------------------------------------------------------
@pytest.mark.parametrize("case", REPLAY_CASES, ids=[c[0] for c in REPLAY_CASES])
def test_each_replay_reached_relevant_and_exact(klt, oracle, cv2, b200, case):
    """Reach: at least REPLAY_MIN points pass the kernel's bound.  Relevance: at least REPLAY_MIN of them get another
    output bit from the integer shortcut than from cv2.  Correctness: the GPU equals cv2 and the oracle."""
    _, kind, make = case
    prev, nxt, pts, win, lk = make()
    got = check_all(klt, oracle, cv2, prev, nxt, pts, win, kind, **lk)
    reached, relevant, within, wrong = shortcut_vs_cv2(kind, prev, nxt, pts, win, got)
    assert reached >= REPLAY_MIN and relevant >= REPLAY_MIN and wrong == 0, (reached, relevant, within, wrong)


# ---- c. batched device path at each warp count -------------------------------------------------
@pytest.mark.parametrize("win", [(64, 64), (41, 96), (9, 455)], ids=["64x64_4warps", "41x96_3warps", "9x455_2warps"])
def test_batched_lk_track_with_iteration_counts(klt, oracle, b200, win):
    """B = 5 pairs of N = 301 points: at 3 and 2 warps per CTA, CTAs straddle pairs."""
    torch = b200
    from visual_odom_pipeline_b200 import tracker as T
    B, H, W, N = 5, 376, 1241, 301
    pairs = [S.frame_pair(H, W, seed=90 + i, motion=S.HARD if i % 2 else S.BENIGN) for i in range(B)]
    pts = np.stack([border_points(N, H, W, seed=i).reshape(N, 2) for i in range(B)])
    prev = T.alloc_image_batch(B, H, W); prev.copy_(torch.from_numpy(np.stack([p[0] for p in pairs])))
    nxt = T.alloc_image_batch(B, H, W); nxt.copy_(torch.from_numpy(np.stack([p[1] for p in pairs])))
    P0, P1 = T.DevicePyramid(prev, win, 3), T.DevicePyramid(nxt, win, 3)
    q, st, er, it = T.lk_track(P0, P1, torch.from_numpy(pts).cuda(), criteria=(3, 30, 0.01), return_iters=True)
    torch.cuda.synchronize()
    for b in range(B):
        want = oracle.calc_optical_flow_pyr_lk(pairs[b][0], pairs[b][1], pts[b], None, win, 3, (3, 30, 0.01), return_iters=True)
        assert_lk_equal((q[b].cpu().numpy(), st[b].cpu().numpy(), er[b].cpu().numpy()), want[:3], "pair %d" % b)
        assert np.array_equal(it[b].cpu().numpy(), want[3]), "iteration counts, pair %d" % b


def test_step_batch_ragged_counts_at_3_warps(klt, cv2, b200):
    """KLTTracker.step_batch at 41x96 (3 warps per CTA) with counts 0, 1, 7, N: the kernel's early exit past a pair's
    count indexes points by the CTA's warp count.  Against the reference's cv2 step per sequence."""
    torch = b200
    from visual_odom_pipeline_b200 import tracker as T
    lk = dict(winSize=(41, 96), maxLevel=3, criteria=(3, 30, 0.03))
    det = dict(maxCorners=500, qualityLevel=0.03, minDistance=10, blockSize=31)
    h, w = 376, 1241
    seqs = [S.sequence(h, w, 3, seed=60 + b) for b in range(4)]
    pts = [cv2.goodFeaturesToTrack(s[0], **det).reshape(-1, 2) for s in seqs]
    pts = [p[:n] for p, n in zip(pts, (0, 1, 7, 301))]
    assert len(pts[3]) == 301
    trk = T.KLTTracker(**lk).reset(torch.from_numpy(np.stack([s[0] for s in seqs])).cuda())
    for t in range(1, 3):
        n = max(len(p) for p in pts)
        padded = np.full((4, n, 2), np.nan, np.float32)
        for b, p in enumerate(pts):
            padded[b, :len(p)] = p
        cnt = np.array([len(p) for p in pts], np.int32)
        out = trk.step_batch(torch.from_numpy(np.stack([s[t] for s in seqs])).cuda(), torch.from_numpy(padded).cuda(),
                             torch.from_numpy(cnt).cuda(), **det)
        nxt_pts, ncnt, keep, n_new = [x.cpu().numpy() for x in out]
        nxt = []
        for b in range(4):
            im0, im1 = seqs[b][t - 1], seqs[b][t]
            if len(pts[b]):
                p0 = pts[b].reshape(-1, 1, 2)
                p1 = cv2.calcOpticalFlowPyrLK(im0, im1, p0, None, **lk)[0]
                p0r = cv2.calcOpticalFlowPyrLK(im0, im1, p1, None, **lk)[0]
                p1 = p1.reshape(-1, 2)
                keep_ref = ((abs(p0 - p0r).reshape(-1, 2).max(-1) < 30) & (0 <= p1[:, 0]) & (p1[:, 0] <= w)
                            & (0 <= p1[:, 1]) & (p1[:, 1] <= h))
            else:
                p1, keep_ref = np.zeros((0, 2), np.float32), np.zeros(0, bool)
            surv_ref = p1[keep_ref]
            mask = np.full_like(im1, 255)
            for x, y in [np.int32(p) for p in surv_ref]:
                cv2.circle(mask, (int(x), int(y)), 10, 0, -1)
            new_ref = cv2.goodFeaturesToTrack(im1, mask=mask, **det)
            new_ref = np.zeros((0, 2), np.float32) if new_ref is None else new_ref.reshape(-1, 2)
            s = int(keep[b].sum())
            assert not keep[b, cnt[b]:].any(), "sequence %d frame %d: keep past the count" % (b, t)
            assert np.array_equal(keep[b, :cnt[b]], keep_ref), "sequence %d frame %d: keep" % (b, t)
            assert np.array_equal(nxt_pts[b, :s].view(np.uint32), surv_ref.view(np.uint32)), "sequence %d frame %d" % (b, t)
            assert int(ncnt[b]) == s + int(n_new[b]) and np.array_equal(nxt_pts[b, s:int(ncnt[b])], new_ref), (b, t)
            nxt.append(np.concatenate([surv_ref, new_ref]))
        pts = nxt


# ---- d. the minEigThreshold gate ---------------------------------------------------------------
@pytest.mark.parametrize("win", [(15, 15), (21, 21), (31, 31), (63, 63)], ids=["15x15", "21x21", "31x31", "63x63"])
def test_min_eig_threshold_gate_at_its_float32_boundary(klt, oracle, cv2, b200, win):
    """The gate compares the float32 min eigenvalue m with (float)minEigThreshold.  Thresholds: m of a chosen point, the
    next float32 above it, a double between m and halfway to that float (rounds to m), 0, and one above every m."""
    h, w = 376, 1241
    a, b = S.frame_pair(h, w, seed=5)
    p = border_points(300, h, w, seed=11)
    lk = dict(maxLevel=0, criteria=(3, 30, 0.01))
    _, st, m = check_all(klt, oracle, cv2, a, b, p, win, "GET_MIN_EIGENVALS", flags=8, **lk)
    m, ok = m.reshape(-1), st.reshape(-1) == 1
    i = np.flatnonzero(ok)[np.argsort(m[ok])[ok.sum() // 2]]   # a tracked point with the median eigenvalue
    mi = m[i]
    up = np.nextafter(mi, np.float32(np.inf))
    thresholds = [float(mi), float(up), float(mi) + (float(up) - float(mi)) / 4, 0.0, float(m[ok].max()) * 2]
    assert np.float32(thresholds[2]) == mi and thresholds[2] > float(mi)
    status = []
    for thr in thresholds:
        _, st, _ = check_all(klt, oracle, cv2, a, b, p, win, "minEigThreshold %r" % thr, minEigThreshold=thr, **lk)
        status.append(int(st.reshape(-1)[i]))
    assert status == [1, 0, 1, 1, 0], status
