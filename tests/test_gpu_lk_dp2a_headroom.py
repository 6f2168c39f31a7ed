"""LK Newton sums on dp2a: the int32 headroom of the byte-split accumulators, driven near their reachable maximum.

newton_sums (lk.cu) splits each bilinear J sample j (0 <= j <= 8160) into its low byte (<= 255) and high byte (<= 31) and
accumulates sum(lo * Ix) and sum(hi * Ix) (and the same with Iy) per lane in int32, flushed every 16 rows with one plain REDUX
each.  A lane owns 4 adjacent columns, so at a flush it has summed at most 64 pixels:
    loose bound   per lane 64 * 4080 * 255 = 66 585 600,   32 lanes 2 130 739 200 < 2^31 - 1.
No scene reaches the loose bound: over 4 adjacent columns the positive Ix telescope to at most 2 * 16 * 255 = 8160 per row, and
negative Ix only subtract (lo >= 0), so
    reachable     per lane 16 * 8160 * 255 = 33 292 800,   32 lanes 1 065 369 600.
The scene below reaches >= 90 % of the reachable bounds (asserted from a numpy restatement of the lane mapping): I is a column
pattern 0, 0, 255, 255 (|Ix| = 4080 in every column, signs + + - -), and J is the pattern 0, 1, 224, 223 sampled 1/32 px to the
right (weights 31/32, 1/32), so the first Newton step sees lo = 255 where Ix > 0 and lo = 1 where Ix < 0.  From row FLIP down
both patterns are shifted by two columns: the step gives I a well-conditioned structure tensor, and in the 63-row window it
falls into the second flush, which leaves the first flush at the full pattern.  The transposed scene drives the Iy sums the
same way.  One Newton step (maxCount 1) from that guess makes the position a direct function of the sums; results must equal
the CPU oracle's bit for bit, after one step and after convergence.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

INIT = 4                                 # OPTFLOW_USE_INITIAL_FLOW
LANE_REACH = 16 * 8160 * 255
WARP_REACH = 32 * LANE_REACH
LANE_LOOSE = 64 * 4080 * 255
I32_MAX = 2 ** 31 - 1
SIZE, Y0, FLIP = 192, 80, 73             # window rows centred on Y0; rows >= FLIP have both patterns shifted by 2
XS = (84, 88, 92)                        # multiples of 4: the same stripe phase under every window
WINDOWS = [(21, 21), (31, 31), (35, 35), (63, 63)]      # the compiled-in windows and the largest runtime one
I_PAT = np.array([0, 0, 255, 255], np.uint8)
J_PAT = np.array([0, 1, 224, 223], np.uint8)


def _scene(transpose):
    x = np.arange(SIZE)
    I = np.tile(I_PAT[x % 4], (SIZE, 1))
    I[FLIP:] = I_PAT[(x + 2) % 4]
    J = np.tile(J_PAT[x % 4], (SIZE, 1))
    J[FLIP:] = J_PAT[(x + 2) % 4]
    pts = np.array([(X, Y0) for X in XS], np.float32)
    guess = pts + np.float32([1 / 32, 0])
    if transpose:
        I, J, pts, guess = I.T.copy(), J.T.copy(), pts[:, ::-1].copy(), guess[:, ::-1].copy()
    return I, J, pts, guess


def _newton_lane_sums(I, D, J, pt, guess, win):
    """First Newton step at level 0, restated: per (lane, 16-row flush) sums of lo(j) * Ix and lo(j) * Iy under newton_sums'
    lane mapping (NL lanes of 4 columns per row group, NG groups of RG rows)."""
    f32 = np.float32
    w, h = win

    def weights(px, py):
        ix, iy = int(np.floor(px)), int(np.floor(py))
        a, b = f32(px - f32(ix)), f32(py - f32(iy))
        iw00 = int(np.rint(f32(f32(f32(1) - a) * f32(f32(1) - b)) * f32(16384)))
        iw01 = int(np.rint(f32(a * f32(f32(1) - b)) * f32(16384)))
        iw10 = int(np.rint(f32(f32(f32(1) - a) * b) * f32(16384)))
        return ix, iy, (iw00, iw01, iw10, 16384 - iw00 - iw01 - iw10)

    def bil(P, ix, iy, wt):
        P = P.astype(np.int64)
        ys, xs, ys1, xs1 = slice(iy, iy + h), slice(ix, ix + w), slice(iy + 1, iy + h + 1), slice(ix + 1, ix + w + 1)
        return P[ys, xs] * wt[0] + P[ys, xs1] * wt[1] + P[ys1, xs] * wt[2] + P[ys1, xs1] * wt[3]

    hx, hy = f32((w - 1) * 0.5), f32((h - 1) * 0.5)
    ix, iy, wt = weights(f32(pt[0]) - hx, f32(pt[1]) - hy)
    Ix, Iy = (bil(D[..., 0], ix, iy, wt) + 8192) >> 14, (bil(D[..., 1], ix, iy, wt) + 8192) >> 14
    jx, jy, wj = weights(f32(guess[0]) - hx, f32(guess[1]) - hy)
    lo = ((bil(J, jx, jy, wj) + 256) >> 9) & 255
    assert np.abs(Ix).max() <= 4080 and np.abs(Iy).max() <= 4080
    nl = (w + 3) // 4
    ng0 = min(32 // nl, h)
    rg = -(-h // ng0)
    ng = -(-h // rg)
    s1, s2 = {}, {}
    for lane in range(32):
        grp, cq = divmod(lane, nl)
        if grp >= ng:
            continue
        for f, r0 in enumerate(range(0, rg, 16)):
            rows = slice(grp * rg + r0, min(grp * rg + min(rg, r0 + 16), h))
            cols = slice(4 * cq, min(4 * cq + 4, w))
            s1[lane, f] = int((lo[rows, cols] * Ix[rows, cols]).sum())
            s2[lane, f] = int((lo[rows, cols] * Iy[rows, cols]).sum())
    warp = lambda s, f: sum(v for (ln, g), v in s.items() if g == f)
    nflush = -(-rg // 16)
    return (max(max(abs(v) for v in s.values()) for s in (s1, s2)),
            max(abs(warp(s, f)) for s in (s1, s2) for f in range(nflush)))


def _same(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _check(ibt, oracle, I, J, pts, guess, win, criteria, what):
    lp = dict(winSize=win, maxLevel=0, criteria=criteria)
    p1, st, _, it = ibt.calcOpticalFlowPyrLK(I, J, pts, guess.copy(), flags=INIT, return_iters=True, **lp)
    po, so, _, ito = oracle.calcOpticalFlowPyrLK(I, J, pts, guess.copy(), flags=INIT, return_iters=True, **lp)
    assert so.all(), what
    assert _same(p1, po) and _same(st, so), (what, p1, po)
    assert np.array_equal(it, ito.sum(1)), (what, it, ito)
    return it


@pytest.mark.parametrize("transpose", [False, True], ids=["Ix", "Iy"])
def test_lk_dp2a_newton_headroom(ibt, oracle, transpose):
    I, J, pts, guess = _scene(transpose)
    D = oracle.scharr_deriv(I)
    lane_peak = warp_peak = 0
    for win in WINDOWS:
        for pt, g in zip(pts, guess):
            lp, wp = _newton_lane_sums(I, D, J, pt, g, win)
            assert lp <= LANE_LOOSE and wp <= I32_MAX, (win, lp, wp)
            lane_peak, warp_peak = max(lane_peak, lp), max(warp_peak, wp)
        it = _check(ibt, oracle, I, J, pts, guess, win, (1, 1, 0.0), "one step %s" % (win,))
        assert (it == 1).all(), (win, it)
        _check(ibt, oracle, I, J, pts, guess, win, (3, 30, 0.01), "converged %s" % (win,))
    assert lane_peak >= 0.9 * LANE_REACH, (lane_peak, LANE_REACH)
    assert warp_peak >= 0.9 * WARP_REACH, (warp_peak, WARP_REACH)


def test_lk_dp2a_newton_headroom_multichannel(ibt, oracle):
    I, J, pts, guess = _scene(False)
    I3, J3 = np.stack([I, I, I], -1), np.stack([J, J, J], -1)
    it = _check(ibt, oracle, I3, J3, pts, guess, (63, 63), (1, 1, 0.0), "3 channels, one step")
    assert (it == 1).all(), it
