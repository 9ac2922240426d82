"""GPU tier: the small-batch pyramid build (pyr_build_cluster_kernel, one thread-block cluster per image) against cv2.pyrDown,
level by level and bit for bit, on both sides of its batch threshold, and the launch path it shares with LK (programmatic
dependent launch) under CUDA-graph capture.  Which kernel ran is read from torch.profiler."""
import ctypes

import numpy as np
import pytest

from conftest import assert_lk_equal
from visual_odom_pipeline_b200 import synth as S

pytestmark = pytest.mark.gpu

CLUSTER, FUSED = "pyr_build_cluster_kernel", "pyr_build_fused_kernel"


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tier needs a CUDA device"
    return torch


def kernels_of(torch, fn):
    """Names of the CUDA kernels fn launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " ".join(e.key for e in prof.key_averages())


def cv2_levels(cv2, img, top):
    out = [img]
    for _ in range(top):
        out.append(cv2.pyrDown(out[-1]))
    return out


def check_batch(torch, cv2, h, w, batch, max_level, expect, win=(5, 5), seed=0):
    from visual_odom_pipeline_b200 import tracker as T
    imgs = [S.texture(h, w, seed=seed + i).astype(np.uint8) for i in range(batch)]
    d = T.alloc_image_batch(batch, h, w)
    d.copy_(torch.from_numpy(np.stack(imgs)))
    pyr = T.DevicePyramid(d, win, max_level)
    names = kernels_of(torch, pyr.build)
    for k in (CLUSTER, FUSED):
        assert (k in names) == (k == expect), (h, w, batch, names)
    for b in range(batch):
        ref = cv2_levels(cv2, imgs[b], pyr.top)
        for l in range(1, pyr.top + 1):
            assert np.array_equal(pyr.level(l)[b].cpu().numpy(), ref[l]), (h, w, batch, b, l)
    return pyr.top


@pytest.fixture(scope="module")
def threshold(torch_cuda):
    """The largest batch the cluster build takes (KLT_PYR_CLUSTER_MAX_ITEMS in csrc/klt_pyramid.cu), found from which kernel
    builds a batch of small images.  A frame pair must take it."""
    torch = torch_cuda
    from visual_odom_pipeline_b200 import tracker as T

    def cluster_at(batch):
        pyr = T.DevicePyramid(T.alloc_image_batch(batch, 64, 96), (5, 5), 2)
        return CLUSTER in kernels_of(torch, pyr.build)
    lo, hi = 2, 64
    assert cluster_at(lo) and not cluster_at(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if cluster_at(mid) else (lo, mid)
    return lo


BATCHES = {"one": lambda t: 1, "pair": lambda t: 2, "threshold": lambda t: t, "above_threshold": lambda t: t + 1}


@pytest.mark.parametrize("which", sorted(BATCHES))
def test_cluster_build_bit_exact_on_both_sides_of_the_threshold(cv2, torch_cuda, threshold, which):
    batch = BATCHES[which](threshold)
    expect = CLUSTER if batch <= threshold else FUSED
    assert check_batch(torch_cuda, cv2, 376, 1241, batch, 3, expect, win=(21, 21), seed=10 * batch) == 3


@pytest.mark.parametrize("hw", [(3, 4), (5, 7), (9, 6), (17, 33), (47, 156), (61, 130), (94, 311), (200, 301), (240, 322), (480, 640)])
def test_cluster_build_odd_and_tiny_shapes(cv2, torch_cuda, hw):
    """Widths that are no multiple of 4 (or of the 16-byte granule), bands of one row or none, up to 6 levels.  Shapes the
    one-launch builds reject (a level narrower than 4 or lower than 3 pixels) take the per-level launches."""
    h, w = hw
    for batch in (1, 2):
        from visual_odom_pipeline_b200 import _lib
        lay = _lib.klt_pyr_layout()
        assert _lib.load().klt_pyr_plan(w, h, 3, 3, 6, batch, ctypes.byref(lay)) == 0
        takes = all(lay.level[l].w >= 4 and lay.level[l].h >= 3 for l in range(lay.top)) and lay.top >= 1
        check_batch(torch_cuda, cv2, h, w, batch, 6, CLUSTER if takes else None, win=(3, 3), seed=h + w)


def test_cluster_build_caller_pitches_leave_the_padding_alone(cv2, torch_cuda):
    """Level 0 with a caller pitch and batch stride, levels 1..3 with pitches larger than their width: only the w pixels of
    every row are written.  A level-0 pitch that is not a multiple of 16 is not for the cluster build (nor for the other
    one-launch build) and goes level by level."""
    torch = torch_cuda
    from visual_odom_pipeline_b200 import _lib
    L = _lib.load()
    ctx = _lib.default_context(0)
    B, H, W = 2, 120, 203
    imgs = [S.texture(H, W, seed=70 + i).astype(np.uint8) for i in range(B)]
    for pitch0, expect in ((272, CLUSTER), (216, None)):
        base = torch.zeros((B, H + 3, pitch0), dtype=torch.uint8, device="cuda")
        for b in range(B):
            base[b, :H, :W].copy_(torch.from_numpy(imgs[b]))
        lay = _lib.klt_pyr_layout()
        assert L.klt_pyr_plan(W, H, 5, 5, 3, B, ctypes.byref(lay)) == 0
        lay.level[0].pitch, lay.level[0].batch_stride = pitch0, base.stride(0)
        off = 0
        for l in range(1, lay.top + 1):
            lv = lay.level[l]
            lv.pitch = (lv.w + 7) // 8 * 8 + 24
            lv.batch_stride = lv.pitch * (lv.h + 1)
            lv.offset = off
            off += lv.batch_stride * B
        lay.bytes = off
        buf = torch.full((off,), 0xA5, dtype=torch.uint8, device="cuda")
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        names = kernels_of(torch, lambda: L.klt_pyr_build(ctx.handle, base.data_ptr(), ctypes.byref(lay), buf.data_ptr(), 0, B, st) == 0 or pytest.fail("build"))
        for k in (CLUSTER, FUSED):
            assert (k in names) == (k == expect), (pitch0, names)
        host = buf.cpu().numpy()
        for b in range(B):
            ref = cv2_levels(cv2, imgs[b], lay.top)
            for l in range(1, lay.top + 1):
                lv = lay.level[l]
                item = host[lv.offset + b * lv.batch_stride: lv.offset + (b + 1) * lv.batch_stride].reshape(lv.h + 1, lv.pitch)
                assert np.array_equal(item[:lv.h, :lv.w], ref[l]), (pitch0, b, l)
                assert (item[:, lv.w:] == 0xA5).all() and (item[lv.h:] == 0xA5).all(), ("padding written", pitch0, b, l)


def test_cluster_build_falls_back_when_a_band_does_not_fit(cv2, torch_cuda):
    """A 3840 x 2160 image: the staged level-0 rows of one band exceed the shared-memory budget."""
    check_batch(torch_cuda, cv2, 2160, 3840, 1, 3, FUSED, seed=3)


def test_cluster_build_pyramid_reuse_skips_and_rebuilds(cv2, torch_cuda):
    """The host entry point builds its pair (a batch of 2) with the cluster kernel, which honours the reuse hashes: the same
    arrays passed again skip both builds, an image edited in place is rebuilt."""
    from visual_odom_pipeline_b200 import _lib
    import visual_odom_pipeline_b200 as K
    L = _lib.load()
    ctx = K.default_context(0)
    L.klt_debug_pyr_reuse_count.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_ulonglong)]
    L.klt_debug_pyr_reuse_count.restype = ctypes.c_int

    def skipped():
        v = ctypes.c_ulonglong()
        assert L.klt_debug_pyr_reuse_count(ctx.handle, ctypes.byref(v)) == 0
        return v.value
    lk = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    a, b = S.frame_pair(376, 1241, seed=81)
    p = S.uniform_points(300, 376, 1241, seed=82)

    def call(what):
        assert_lk_equal(K.calcOpticalFlowPyrLK(a, b, p, None, **lk), cv2.calcOpticalFlowPyrLK(a, b, p, None, **lk), what)
    call("first call")
    names = kernels_of(torch_cuda, lambda: call("second call: hashes recorded"))
    assert CLUSTER in names and FUSED not in names, names
    s0 = skipped()
    call("third call: both skipped")
    assert skipped() == s0 + 2
    a[7, 9] ^= 0x10
    call("previous image edited in place")
    assert skipped() == s0 + 3
    call("unchanged again")
    assert skipped() == s0 + 5


@pytest.mark.parametrize("which", ["pair", "above_threshold"])
def test_pyramid_and_lk_graph_replay_equals_direct_launches(cv2, torch_cuda, threshold, which):
    """The pyramids of `batch` images, the two single-image pyramids of a pair and LK recorded into one CUDA graph: the replay
    (programmatic dependent launch edges) writes the same bytes as direct launches, for both one-launch builds."""
    torch = torch_cuda
    from visual_odom_pipeline_b200 import tracker as T
    batch = BATCHES[which](threshold)
    h, w, win, crit = 376, 1241, (21, 21), (3, 30, 0.01)
    frames = S.sequence(h, w, batch + 2, seed=30 + batch)
    d = T.alloc_image_batch(batch, h, w)
    pyr, P0, P1 = T.DevicePyramid(d, win, 3), T.DevicePyramid(d[0:1], win, 3), T.DevicePyramid(d[1:2], win, 3)
    pts = torch.from_numpy(S.uniform_points(2000, h, w, seed=31).reshape(1, -1, 2)).cuda()

    def step():
        pyr.build(); P0.build(); P1.build()
        return T.lk_track(P0, P1, pts, criteria=crit)

    def outputs(res):
        return [x.cpu().numpy().copy() for x in res] + [p.level(l).cpu().numpy().copy() for p in (pyr, P0, P1) for l in range(1, 4)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                        # scratch of the capture stream is allocated outside the capture
        for _ in range(2):
            step()
    side.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        res = step()
    for t in (1, 2):
        d.copy_(torch.from_numpy(np.stack(frames[t:t + batch])))
        torch.cuda.synchronize()
        g.replay()
        torch.cuda.synchronize()
        replay = outputs(res)
        direct = outputs(step())
        for i, (x, y) in enumerate(zip(replay, direct)):
            assert np.array_equal(x, y), (batch, t, i)
        ref = cv2.calcOpticalFlowPyrLK(frames[t], frames[t + 1], pts.cpu().numpy().reshape(-1, 1, 2), None, winSize=win, maxLevel=3,
                                       criteria=crit)
        assert_lk_equal(tuple(x.reshape(y.shape) for x, y in zip(replay[:3], ref)), ref, "replay of step %d, batch %d" % (t, batch))
