"""One-off fuzzing of the drop-ins against live cv2 on a GPU box (many more cases than tests/test_gpu_random.py keeps in the
suite): random shapes, windows, levels, criteria, flags, image kinds (noise, smooth, steps, 0/255 checkerboards, constant),
point sets reaching outside the image.  usage: python scripts/fuzz_gpu.py [cases] [seed]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__)))); sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np, cv2
import visual_odom_pipeline_b200 as K
from test_random_cpu import _image

cases = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 1)
mode = sys.argv[3] if len(sys.argv) > 3 else "lk"
bad = 0


def same(x, y):
    return (x is None and y is None) or (x is not None and y is not None and x.shape == y.shape and np.array_equal(x, y))


if mode == "other":
    # detection, pre-filter, pyramids, and call sequences through the host entry point (pyramid reuse): same bar
    from oracle import klt_oracle as O
    prev_pair = None
    for c in range(cases):
        h, w = int(rng.integers(36, 260)), int(rng.integers(36, 420))
        a = _image(h, w, int(rng.integers(0, 10 ** 6)), int(rng.integers(0, 5)))
        bs = [3, 5, 7, 15, 31][int(rng.integers(0, 5))]
        if bs // 2 < min(h, w):
            md = [0.0, 1.0, 4.5, 10.0][int(rng.integers(0, 4))]
            mc = [0, 25, 1000][int(rng.integers(0, 3))]
            m = None
            if rng.integers(0, 2):
                m = (rng.integers(0, 4, (h, w)) > 0).astype(np.uint8) * 255
            if not same(K.goodFeaturesToTrack(a, mc, 0.03, md, mask=m, blockSize=bs), cv2.goodFeaturesToTrack(a, mc, 0.03, md, mask=m, blockSize=bs)):
                bad += 1; print("MISMATCH gftt case", c, (h, w, bs, md, mc, m is not None), flush=True)
        d, sc, ss = [(5, 1.5, 1.5), (3, 12.0, 1.0), (9, 30.0, 4.0), (15, 50.0, 6.0)][int(rng.integers(0, 4))]
        if not np.array_equal(K.bilateralFilter(a, d, sc, ss), O.bilateral_filter(a, d, sc, ss)):
            bad += 1; print("MISMATCH bilateral case", c, (h, w, d, sc, ss), flush=True)
        top, lv = K.buildOpticalFlowPyramid(a, (5, 5), 4)
        ref = a
        for l in range(1, top + 1):
            ref = cv2.pyrDown(ref)
            if not np.array_equal(lv[l], ref):
                bad += 1; print("MISMATCH pyramid case", c, (h, w, l), flush=True); break
        # call sequence: sometimes the same pair again (other points), sometimes an edit in place, sometimes a new pair
        r = int(rng.integers(0, 4))
        if prev_pair is None or r == 0 or prev_pair[0].shape != a.shape:
            prev_pair = [a, np.roll(a, (int(rng.integers(-4, 5)), int(rng.integers(-4, 5))), axis=(0, 1)).copy()]
        elif r == 1:
            prev_pair[int(rng.integers(0, 2))][int(rng.integers(0, prev_pair[0].shape[0])), int(rng.integers(0, prev_pair[0].shape[1]))] ^= 0x55
        elif r == 2:
            prev_pair = [prev_pair[1], _image(prev_pair[1].shape[0], prev_pair[1].shape[1], int(rng.integers(0, 10 ** 6)), 1)]
        hh, ww = prev_pair[0].shape
        n = int(rng.integers(1, 300))
        p = np.stack([rng.uniform(0, ww, n), rng.uniform(0, hh, n)], -1).astype(np.float32).reshape(-1, 1, 2)
        kw = dict(winSize=[(21, 21), (31, 31)][int(rng.integers(0, 2))], maxLevel=3, criteria=(3, 30, 0.03))
        g, rf = K.calcOpticalFlowPyrLK(prev_pair[0], prev_pair[1], p, None, **kw), cv2.calcOpticalFlowPyrLK(prev_pair[0], prev_pair[1], p, None, **kw)
        if not (np.array_equal(g[0].view(np.uint32), rf[0].view(np.uint32)) and np.array_equal(g[1], rf[1])):
            bad += 1; print("MISMATCH sequence case", c, (hh, ww, r, n, kw["winSize"]), flush=True)
    print("fuzz other: %d cases, %d mismatches" % (cases, bad))
    sys.exit(1 if bad else 0)

crits = [(3, 30, 0.01), (3, 30, 0.03), (3, 5, 0.03), (1, 7, 0.0), (2, 0, 0.05), (3, 100, 1e-4)]
for c in range(cases):
    h, w = int(rng.integers(8, 220)), int(rng.integers(8, 300))
    kind, seed = int(rng.integers(0, 5)), int(rng.integers(0, 10 ** 6))
    win = [(21, 21), (31, 31), (int(rng.integers(3, 45)), int(rng.integers(3, 45)))][int(rng.integers(0, 3))]
    lvl, n = int(rng.integers(0, 6)), int(rng.integers(1, 400))
    crit, flags = crits[int(rng.integers(0, len(crits)))], [0, 0, 8, 4][int(rng.integers(0, 4))]
    a = _image(h, w, seed, kind)
    if rng.integers(0, 4) == 0:
        b = _image(h, w, seed + 1, kind)                                   # unrelated second frame: diverging points
    else:
        b = np.roll(a, (int(rng.integers(-7, 8)), int(rng.integers(-7, 8))), axis=(0, 1))
    p = np.stack([rng.uniform(-10, w + 10, n), rng.uniform(-10, h + 10, n)], -1).astype(np.float32).reshape(-1, 1, 2)
    init = (p + rng.normal(0, 2.0, p.shape)).astype(np.float32) if flags == 4 else None
    kw = dict(winSize=win, maxLevel=lvl, criteria=crit, flags=flags)
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None if init is None else init.copy(), **kw)
    got = K.calcOpticalFlowPyrLK(a, b, p, init, **kw)
    m = (ref[1].ravel() == 1) & (got[1].ravel() == 1)
    ok = (np.array_equal(got[0].view(np.uint32), ref[0].view(np.uint32)) and np.array_equal(got[1], ref[1])
          and (flags == 8 or np.array_equal(got[2].ravel()[m].view(np.uint32), ref[2].ravel()[m].view(np.uint32))))
    if not ok:
        bad += 1
        d = np.nonzero((got[0].view(np.uint32) != ref[0].view(np.uint32)).any(-1).ravel() | (got[1].ravel() != ref[1].ravel()))[0]
        print("MISMATCH case %d: h=%d w=%d kind=%d seed=%d win=%s lvl=%d n=%d crit=%s flags=%d: %d points differ, first %s" % (c, h, w, kind, seed, win, lvl, n, crit, flags, len(d), d[:5]), flush=True)
print("fuzz: %d cases, %d mismatches" % (cases, bad))
sys.exit(1 if bad else 0)
