"""GPU tier (pytest -m gpu, B200) of the detection step at every regime of the eigenvalue-map kernels, not only at the
reference's blockSize 31 on frames of 33 rows and more (tests/test_gpu_corners.py).  The grid follows the kernels:
- col_scan_kernel works in chunks of 16 rows (6-stage operand ring, 4-chunk sum ring): heights of 1 to 9 chunks, on
  both sides of each chunk edge;
- row_scan_kernel works in chunks of 64 columns and fetches interior chunks without reflection: widths of 1 to 6
  chunks, on both sides of the 64-px edges, and blocks so large that no chunk is interior;
- cov_kernel switches the y-derivative's row filter to the scalar tail at 32 * (W / 32): W % 32 in {0, 1, 31} and
  W < 32;
- row_sum_small_kernel serves blocks up to 5 and row_scan_kernel 6 and up: blocks 1-8, 15, 16, 31, 63, 64, 65, 127.
Every map is compared with live cv2.cornerMinEigenVal and with the C oracle as uint32, corners with live
cv2.goodFeaturesToTrack in value and order.  Then the batched device API (per-item strides in blockIdx.z, an all-zero
mask, the masked maximum), the block sizes the library refuses, and KLTSequenceBatch at small block sizes."""
import numpy as np
import pytest

from test_corners_blocks_cpu import accepted, eig_mismatch, image, same_corners

pytestmark = pytest.mark.gpu

HEIGHTS = [1, 2, 15, 16, 17, 32, 33, 48, 49, 64, 65, 80, 81, 96, 97, 112, 113, 128, 129]
WIDTHS = [1, 2, 5, 31, 32, 33, 63, 64, 65, 127, 128, 129, 256, 257, 320, 321]
BLOCKS = [1, 2, 3, 4, 5, 6, 7, 8, 15, 16, 31, 63, 64, 65, 127]
# heights at a one-chunk and a three-chunk width, widths at a two-chunk and an eight-chunk height
SHAPES = sorted({(h, w) for h in HEIGHTS for w in (33, 129)} | {(h, w) for w in WIDTHS for h in (17, 128)})
GFTT_PARAMS = [(0, 0.01, 0.0), (40, 0.03, 3.5)]   # (maxCorners, qualityLevel, minDistance)


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def random_mask(h, w, seed):
    """About half the pixels zero, so that the masked maximum and the candidates depend on the mask of every row."""
    return (np.random.default_rng(seed).random((h, w)) < 0.5).astype(np.uint8) * 255


@pytest.mark.parametrize("block", BLOCKS)
def test_eigenvalues_and_corners_equal_cv2_and_oracle(klt, oracle, cv2, block):
    """Noise and 0/255 noise (where the box sums' rounding shows) on every accepted shape of the grid.  Every call
    follows one on another image of the same shape, so a stage that leaves part of the context's workspace unwritten
    shows up as the previous image's values."""
    shapes = [s for s in SHAPES if accepted(block, *s)]
    assert shapes
    failures = []
    for (h, w) in shapes:
        for kind in ("noise", "binary"):
            img = image(kind, h, w, block)
            what = "block %d, %dx%d %s" % (block, h, w, kind)
            got = klt.cornerMinEigenVal(img, block)
            for name, want in (("cv2", cv2.cornerMinEigenVal(img, block, ksize=3)), ("the oracle", oracle.corner_min_eigen_val(img, block))):
                msg = eig_mismatch(got, want)
                if msg:
                    failures.append("%s: eigenvalues vs %s: %s" % (what, name, msg))
            for mask in (None, random_mask(h, w, block)):
                for (mc, ql, md) in GFTT_PARAMS:
                    c = klt.goodFeaturesToTrack(img, mc, ql, md, mask=mask, blockSize=block)
                    k = cv2.goodFeaturesToTrack(img, mc, ql, md, mask=mask, blockSize=block)
                    if not same_corners(c, k):
                        failures.append("%s: corners differ for maxCorners=%d quality=%g minDistance=%g masked=%s"
                                        % (what, mc, ql, md, mask is not None))
    assert not failures, "%d cases differ:\n%s" % (len(failures), "\n".join(failures[:30]))


@pytest.mark.parametrize("block", [1, 2, 3, 4, 5, 6, 7, 8])
def test_kitti_size_noise_equals_cv2(klt, oracle, cv2, block):
    """At blocks 2 and 4 a fresh and a running row sum differ on a few pixels of a KITTI-size noise frame only."""
    for seed in range(2):
        img = image("noise", 376, 1241, seed)
        got = klt.cornerMinEigenVal(img, block)
        assert eig_mismatch(got, cv2.cornerMinEigenVal(img, block, ksize=3)) is None, (block, seed)
        assert eig_mismatch(got, oracle.corner_min_eigen_val(img, block)) is None, (block, seed)
        c = klt.goodFeaturesToTrack(img, 0, 0.01, 0, blockSize=block)
        assert same_corners(c, cv2.goodFeaturesToTrack(img, 0, 0.01, 0, blockSize=block)), (block, seed)


@pytest.mark.parametrize("hw", [(1, 1), (1, 40), (2, 70), (5, 2), (16, 5), (17, 33), (33, 65), (64, 129), (129, 321)])
def test_largest_accepted_block_and_refusal(klt, cv2, hw):
    """block / 2 = min(h, w) - 1 is the largest the library takes (both parities), and equals cv2 there;
    block / 2 = min(h, w) is refused with the library's unsupported error, raised as cv2.error (cv2 itself takes it)."""
    h, w = hw
    m = min(hw)
    for kind in ("noise", "binary"):
        img = image(kind, h, w, m)
        for block in (2 * m - 2, 2 * m - 1):
            if block < 1:
                continue
            assert eig_mismatch(klt.cornerMinEigenVal(img, block), cv2.cornerMinEigenVal(img, block, ksize=3)) is None, (hw, block)
            assert same_corners(klt.goodFeaturesToTrack(img, 0, 0.01, 0, blockSize=block),
                                cv2.goodFeaturesToTrack(img, 0, 0.01, 0, blockSize=block)), (hw, block)
        for block in (2 * m, 2 * m + 1):
            with pytest.raises(cv2.error, match="outside libklt_b200 limits"):
                klt.cornerMinEigenVal(img, block)
            with pytest.raises(cv2.error, match="outside libklt_b200 limits"):
                klt.goodFeaturesToTrack(img, 0, 0.01, 0, blockSize=block)


def _ordered(v):
    """The order-preserving uint32 encoding of a float32 that the device keeps the masked maximum in."""
    b = int(np.float32(v).view(np.uint32))
    return (~b & 0xffffffff) if b & 0x80000000 else b | 0x80000000


@pytest.mark.parametrize("w", [33, 129])
@pytest.mark.parametrize("block", [2, 4, 7])
def test_batched_device_api_per_item(klt, cv2, w, block):
    """detector.py at B = 3 over every height of the grid: maps, masked maxima and corners of each item equal cv2 on
    that item alone.  The masks take the first chunk of 16 rows only, nothing, and everything but the first chunk, then
    a random half, everything and another random half, so that each item's maximum depends on which rows its mask
    covers."""
    import torch
    from visual_odom_pipeline_b200 import detector as D, tracker as T
    for h in HEIGHTS:
        if not accepted(block, h, w):
            continue
        frames = [image(kind, h, w, 7 * h + i) for i, kind in enumerate(("noise", "binary", "noise"))]
        top = np.zeros((h, w), np.uint8)
        top[:16] = 255
        for masks in ([top, np.zeros((h, w), np.uint8), 255 - top],
                      [random_mask(h, w, h), np.full((h, w), 255, np.uint8), random_mask(h, w, h + 1)]):
            dev = T.alloc_image_batch(3, h, w)
            dev.copy_(torch.from_numpy(np.stack(frames)))
            dmask = torch.from_numpy(np.stack(masks)).cuda()
            eig, mx, _ = D.corner_min_eigen_val(dev, block, mask=dmask, return_max=True)
            res = D.good_features_to_track(dev, 0, 0.01, 1.5, mask=dmask, blockSize=block)
            eig, mx = eig.cpu().numpy(), mx.cpu().numpy().view(np.uint32)
            for b in range(3):
                what = "block %d, %dx%d item %d" % (block, h, w, b)
                want = cv2.cornerMinEigenVal(frames[b], block, ksize=3)
                msg = eig_mismatch(eig[b], want)
                assert msg is None, "%s: eigenvalues: %s" % (what, msg)
                sel = masks[b] != 0
                assert int(mx[b]) == (_ordered(want[sel].max()) if sel.any() else 0), what + ": masked maximum"
                k = cv2.goodFeaturesToTrack(frames[b], 0, 0.01, 1.5, mask=masks[b], blockSize=block)
                assert same_corners(res[b], k), what + ": corners"


@pytest.mark.parametrize("block", [2, 4])
def test_sequence_batch_at_small_blocks(klt, cv2, block):
    """KLTSequenceBatch reaches the same launcher through the batched frame step: two KITTI-size noise sequences over
    four frames equal the capped cv2 loop at detection blockSize 2 and 4."""
    from test_gpu_frame_step_async import DET, KITTI, check_against_cv2, noise_sequence
    det = dict(DET, blockSize=block)
    seqs = [noise_sequence(KITTI[0], KITTI[1], 4, seed=900 + 10 * block + b) for b in range(2)]
    init = [cv2.goodFeaturesToTrack(s[0], **det).reshape(-1, 2)[:400 + 200 * b] for b, s in enumerate(seqs)]
    check_against_cv2(cv2, seqs, init, 1500, det=det)
