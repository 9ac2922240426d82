"""The exactness decisions of the generic LK kernel (csrc/klt_lk.cu), restated in numpy and checked against cv2 and the
CPU oracle without a GPU.

The kernel sums G, b and err as exact integers per accumulation class (4 SIMD lanes by x % 4 for x < 8 * (win_w // 8),
then the scalar tail) and converts the class totals to float32.  That shortcut equals OpenCV's float32 running sums only
while no partial sum can pass 2^24; past the kernel's bound for a sum it replays that sum serially in OpenCV's order.
`ClassSums` computes the same class totals in exact int64 and the outputs the shortcut would give.  These tests show that
the helper reproduces cv2 wherever the totals are within the bounds, and that the inputs of the replay cases (shared with
tests/test_gpu_lk_windows.py) put points past each bound where the shortcut would change an output bit, so a kernel that
skipped a replay would fail there."""
import numpy as np
import pytest

from conftest import assert_lk_equal

F = np.float32
EXACT = 1 << 24               # kExact (klt_lk_point.cuh)
B_EXACT = EXACT >> 4          # the b bound: sum of ceil(|d| (|gx| + |gy|) / 16) per class


def q14_weights(fx, fy):
    """A.4 step 3 on float32 arrays of fractional parts -> int64 Q14 weights."""
    ox, oy = F(1) - fx, F(1) - fy
    w00 = np.rint((ox * oy) * F(16384)).astype(np.int64)
    w01 = np.rint((fx * oy) * F(16384)).astype(np.int64)
    w10 = np.rint((ox * fy) * F(16384)).astype(np.int64)
    return w00, w01, w10, 16384 - w00 - w01 - w10


def combine5(t):
    """OpenCV's final combine of the 5 class accumulators, t + ((q0 + q2) + (q1 + q3)), then * 2^-20, on the
    float32-converted class totals t (n, 5)."""
    t = t.astype(F)
    return (t[:, 4] + ((t[:, 0] + t[:, 2]) + (t[:, 1] + t[:, 3]))) * F(2.0 ** -20)


class ClassSums:
    """Exact int64 class totals of the level-0 LK window of each point, as the generic kernel forms them.

    prev, nxt: u8 images; pts: (n, 2) window centres, whose windows (and the J windows passed to `mismatch`) must stay
    within `pad` pixels of the image (`fits`).  The intensity patch is Q5 bilinear of prev (REFLECT_101 outside), the derivative
    patch Q14 bilinear of cv2.Scharr(CV_16S) of prev (zero outside), as in OpenCV (SURVEY.md A.3-A.5)."""

    def __init__(self, prev, nxt, pts, win):
        import cv2
        self.ww, self.wh = win
        self.hw = (F((self.ww - 1) * 0.5), F((self.wh - 1) * 0.5))
        self.pad = pad = max(self.ww, self.wh) + 2
        self.I = cv2.copyMakeBorder(prev, pad, pad, pad, pad, cv2.BORDER_REFLECT_101).astype(np.int64)
        self.J = cv2.copyMakeBorder(nxt, pad, pad, pad, pad, cv2.BORDER_REFLECT_101).astype(np.int64)
        self.GX = np.pad(cv2.Scharr(prev, cv2.CV_16S, 1, 0).astype(np.int64), pad)
        self.GY = np.pad(cv2.Scharr(prev, cv2.CV_16S, 0, 1).astype(np.int64), pad)
        nv = 8 * (self.ww // 8)
        x = np.arange(self.ww)
        self.cls = np.where(x < nv, x % 4, 4)
        x0, y0, wts = self._corner(pts)
        self.iv = self._bilinear(self.I, x0, y0, wts, 9)
        self.gx = self._bilinear(self.GX, x0, y0, wts, 14)
        self.gy = self._bilinear(self.GY, x0, y0, wts, 14)
        self.s11 = self._classes(self.gx * self.gx)
        self.s12 = self._classes(self.gx * self.gy)
        self.s22 = self._classes(self.gy * self.gy)
        self.corner = (np.asarray(pts, F).reshape(-1, 2)[:, 0] - self.hw[0], np.asarray(pts, F).reshape(-1, 2)[:, 1] - self.hw[1])

    def _corner(self, pts):
        p = np.asarray(pts, F).reshape(-1, 2)
        cx, cy = p[:, 0] - self.hw[0], p[:, 1] - self.hw[1]
        ix, iy = np.floor(cx), np.floor(cy)
        return ix.astype(np.int64), iy.astype(np.int64), q14_weights(cx - ix, cy - iy)

    def _bilinear(self, plane, x0, y0, wts, shift):
        ys = y0[:, None] + self.pad + np.arange(self.wh + 1)
        xs = x0[:, None] + self.pad + np.arange(self.ww + 1)
        ys, xs = np.clip(ys, 0, plane.shape[0] - 1), np.clip(xs, 0, plane.shape[1] - 1)   # see fits()
        P = plane[ys[:, :, None], xs[:, None, :]]
        w00, w01, w10, w11 = (w[:, None, None] for w in wts)
        v = P[:, :-1, :-1] * w00 + P[:, :-1, 1:] * w01 + P[:, 1:, :-1] * w10 + P[:, 1:, 1:] * w11
        return (v + (1 << (shift - 1))) >> shift

    def fits(self, jpts):
        """Points whose window lies within the padded planes; the sums of the others are meaningless."""
        x0, y0, _ = self._corner(jpts)
        lim_y, lim_x = self.I.shape[0] - 2 * self.pad, self.I.shape[1] - 2 * self.pad
        return (x0 >= -self.pad) & (y0 >= -self.pad) & (x0 + self.ww + 1 <= lim_x + self.pad) & (y0 + self.wh + 1 <= lim_y + self.pad)

    def _classes(self, v):
        return np.stack([v[:, :, self.cls == k].sum((1, 2)) for k in range(5)], -1)

    # ---- G -------------------------------------------------------------------------------------
    def g_replayed(self):
        """The kernel replays G when some class has sum gx^2 + sum gy^2 > 2^24."""
        return (self.s11 + self.s22 > EXACT).any(-1)

    def shortcut_G(self):
        """-> A11, A12, A22, min_eig, det from the float-converted class totals (A.4 step 5)."""
        A11, A12, A22 = combine5(self.s11), combine5(self.s12), combine5(self.s22)
        D = A11 * A22 - A12 * A12
        dA = A11 - A22
        rad = np.sqrt(dA * dA + (F(4) * A12) * A12)
        min_eig = ((A22 + A11) - rad) / F(2 * self.ww * self.wh)
        return A11, A12, A22, min_eig, D

    # ---- b and err -----------------------------------------------------------------------------
    def mismatch(self, jpts):
        """Q5 difference patch bilinear(J) - Ipatch with the J window centred at jpts (n, 2)."""
        x0, y0, wts = self._corner(jpts)
        return self._bilinear(self.J, x0, y0, wts, 9) - self.iv

    def b_sums(self, jpts):
        """-> class totals of d*gx, d*gy and the kernel's bound sum ceil(|d| (|gx| + |gy|) / 16), each (n, 5)."""
        d = self.mismatch(jpts)
        bound = (np.abs(d) * (np.abs(self.gx) + np.abs(self.gy)) + 15) >> 4
        return self._classes(d * self.gx), self._classes(d * self.gy), self._classes(bound)

    def b_replayed(self, jpts):
        return (self.b_sums(jpts)[2] > B_EXACT).any(-1)

    def shortcut_first_step(self):
        """nextPts after one Newton step from the initial guess (no initial flow, maxLevel 0), with G and b taken from
        the float-converted class totals (A.4 step 6)."""
        A11, A12, A22, _, D = self.shortcut_G()
        cx, cy = self.corner
        s1, s2, _ = self.b_sums(np.stack([cx + self.hw[0], cy + self.hw[1]], -1))
        b1, b2 = combine5(s1), combine5(s2)
        inv = F(1) / D
        dx = (A12 * b2 - A22 * b1) * inv
        dy = (A12 * b1 - A11 * b2) * inv
        return np.stack([(cx + dx) + self.hw[0], (cy + dy) + self.hw[1]], -1)

    def err_total(self, jpts):
        """sum |d| over the window at jpts: the kernel replays err when it exceeds 2^24."""
        return np.abs(self.mismatch(jpts)).sum((1, 2))

    def shortcut_err(self, jpts):
        return (self.err_total(jpts).astype(F) * F(1)) / F(32 * self.ww * self.wh)


# ---- the replay cases ----------------------------------------------------------------------------
# Each builds (prev, next, points, window, lk kwargs); H x W leaves room for a 504-px side.  Points are fractional and keep
# their windows (and the first iterate's) inside the image, so every output the tests compare is defined.
H, W = 160, 640
REPLAY_MIN = 8                # reach and relevance: at least this many points per case


def _checker(cell):
    yy, xx = np.mgrid[0:H, 0:W]
    return ((((xx // cell) + (yy // cell)) % 2) * 255).astype(np.uint8)


def _inner_points(n, win, seed, slack=4):
    rng = np.random.default_rng(seed)
    hx, hy = (win[0] - 1) / 2 + slack, (win[1] - 1) / 2 + slack
    return np.stack([rng.uniform(hx, W - 1 - hx, n), rng.uniform(hy, H - 1 - hy, n)], -1).astype(np.float32).reshape(-1, 1, 2)


def g_case(win, image, seed=0, n=160):
    """G past its bound: 0/255 checkerboards and white noise give gx^2 + gy^2 up to ~2^23 per pixel."""
    rng = np.random.default_rng(seed)
    prev = _checker(image) if isinstance(image, int) else rng.integers(0, 256, (H, W), dtype=np.uint8)
    return prev, prev.copy(), _inner_points(n, win, seed + 1), win, dict(maxLevel=0, flags=8, criteria=(3, 30, 0.01))


def b_case(win, seed=0, n=160):
    """b past its bound, G exact: a smooth low-gradient prev and an unrelated next (large residual), one iteration."""
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    rng = np.random.default_rng(seed)
    prev = 128 + 60 * np.sin(xx / 23.0 + seed) * np.cos(yy / 17.0) + 40 * np.sin((xx + yy) / 31.0)
    nxt = rng.integers(0, 256, (H, W))
    return (np.clip(prev, 0, 255).astype(np.uint8), nxt.astype(np.uint8), _inner_points(n, win, seed + 1, slack=12), win,
            dict(maxLevel=0, criteria=(1, 1, 0.0)))


def err_case(win, seed=0, n=160):
    """err past its bound, G exact: sparse faint dots on black (enough gradient for the gate, |d| near 8160 everywhere)
    and next = 255 - prev."""
    rng = np.random.default_rng(seed)
    prev = np.zeros((H, W), np.uint8)
    ys, xs = rng.integers(0, H, H * W // 150), rng.integers(0, W, H * W // 150)
    prev[ys, xs] = 20
    return prev, 255 - prev, _inner_points(n, win, seed + 1, slack=12), win, dict(maxLevel=0, criteria=(3, 30, 0.01))


REPLAY_CASES = [
    ("G_63x63_cell2", "G", lambda: g_case((63, 63), 2)),
    ("G_63x63_cell3", "G", lambda: g_case((63, 63), 3)),
    ("G_63x63_noise", "G", lambda: g_case((63, 63), None)),
    ("G_504x7_cell2", "G", lambda: g_case((504, 7), 2)),
    ("G_504x7_noise", "G", lambda: g_case((504, 7), None)),
    ("b_63x63", "b", lambda: b_case((63, 63))),
    ("b_504x7", "b", lambda: b_case((504, 7))),
    ("err_46x46", "err", lambda: err_case((46, 46))),
    ("err_63x63", "err", lambda: err_case((63, 63))),
    ("err_504x8", "err", lambda: err_case((504, 8))),
]


def shortcut_vs_cv2(kind, prev, nxt, pts, win, ref):
    """Compares the integer shortcut for one sum (kind "G", "b" or "err") with cv2's result `ref` of the case's call.
    -> (reached, relevant, within, wrong): the points past the kernel's bound for that sum, those of them where the
    shortcut gives another output bit than cv2, the points within every bound that decides the output, and those of
    them where the shortcut differs from cv2 (the helper's self-check: must be none).  Only points with status 1 count.
      G: err is the min eigenvalue (flags OPTFLOW_LK_GET_MIN_EIGENVALS);
      b: nextPts after one iteration from the initial guess (criteria (TERM_COUNT, 1, *));
      err: err at cv2's returned point."""
    q, st, er = (np.asarray(a) for a in ref)
    q, st, er = q.reshape(-1, 2).astype(F), st.reshape(-1), er.reshape(-1).astype(F)
    cs = ClassSums(prev, nxt, pts, win)
    p = np.asarray(pts, F).reshape(-1, 2)
    ok = st == 1
    g_rep = cs.g_replayed()
    if kind == "G":
        reached, within = g_rep, ~g_rep
        diff = cs.shortcut_G()[3].view(np.uint32) != er.view(np.uint32)
    elif kind == "b":
        b_rep = cs.b_replayed(p)
        reached, within = b_rep & ~g_rep, ~b_rep & ~g_rep
        diff = (cs.shortcut_first_step().view(np.uint32) != q.view(np.uint32)).any(-1)
    else:
        ok &= cs.fits(q)
        e_rep = cs.err_total(q) > EXACT
        reached, within = e_rep & ~g_rep, ~e_rep & ~g_rep
        diff = cs.shortcut_err(q).view(np.uint32) != er.view(np.uint32)
    reached, within = reached & ok, within & ok
    return int(reached.sum()), int((reached & diff).sum()), int(within.sum()), int((within & diff).sum())


def run_cv2_and_oracle(oracle, prev, nxt, pts, win, lk):
    import cv2
    ref = cv2.calcOpticalFlowPyrLK(prev, nxt, pts, None, winSize=win, **lk)
    want = oracle.calc_optical_flow_pyr_lk(prev, nxt, pts, None, win, lk["maxLevel"], lk["criteria"], flags=lk.get("flags", 0))
    assert_lk_equal(want, ref, "oracle vs cv2")
    return ref


@pytest.mark.parametrize("case", REPLAY_CASES, ids=[c[0] for c in REPLAY_CASES])
def test_replay_cases_pass_each_bound_where_the_shortcut_is_wrong(oracle, case):
    """cv2 and the oracle agree on the case, at least REPLAY_MIN points pass the kernel's bound for the sum and get
    another output bit from the integer shortcut, and the points within the bounds get cv2's bits from it."""
    _, kind, make = case
    prev, nxt, pts, win, lk = make()
    ref = run_cv2_and_oracle(oracle, prev, nxt, pts, win, lk)
    reached, relevant, within, wrong = shortcut_vs_cv2(kind, prev, nxt, pts, win, ref)
    assert wrong == 0, "shortcut differs from cv2 at %d of %d points within the bounds" % (wrong, within)
    assert reached >= REPLAY_MIN and relevant >= REPLAY_MIN, (reached, relevant)


SELF_CHECK = [(46, 46), (63, 63), (63, 65), (504, 8), (8, 504), (50, 81), (21, 21), (13, 29)]
LK_OF_KIND = {"G": dict(maxLevel=0, flags=8, criteria=(3, 30, 0.01)), "b": dict(maxLevel=0, criteria=(1, 1, 0.0)),
              "err": dict(maxLevel=0, criteria=(3, 30, 0.01))}


@pytest.mark.parametrize("win", SELF_CHECK, ids=["%dx%d" % w for w in SELF_CHECK])
@pytest.mark.parametrize("kind", ["G", "b", "err"])
def test_shortcut_helper_equals_cv2_within_the_bounds(oracle, kind, win):
    """The helper itself, at the windows of the GPU window sweep: on smooth textured frames moved by one pixel, where
    most sums stay within the bounds, the shortcut gives cv2's bits for every such point.  (Unblurred textures push G
    past its bound at nearly every point of a window of 46x46 or more.)"""
    import cv2
    from visual_odom_pipeline_b200 import synth as S
    h, w = 600, 640
    tested = 0
    for seed, motion in ((7, S.BENIGN), (8, S.HARD)):
        prev = cv2.GaussianBlur(S.frame_pair(h, w, seed=seed, motion=motion)[0], (0, 0), 3)
        nxt = np.roll(prev, (1, -1), (0, 1))
        rng = np.random.default_rng(seed)
        mx, my = win[0] / 2 + 20, win[1] / 2 + 20
        pts = np.stack([rng.uniform(mx, w - mx, 120), rng.uniform(my, h - my, 120)], -1).astype(np.float32).reshape(-1, 1, 2)
        ref = run_cv2_and_oracle(oracle, prev, nxt, pts, win, LK_OF_KIND[kind])
        _, _, within, wrong = shortcut_vs_cv2(kind, prev, nxt, pts, win, ref)
        assert wrong == 0, "%s: shortcut differs from cv2 at %d of %d points within the bounds" % (kind, wrong, within)
        tested += within
    assert tested >= 150, tested
