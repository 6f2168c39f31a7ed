"""GPU: the CUDA Lucas-Kanade solver against the CPU oracle, bit for bit.

The kernel and oracle/ibt_oracle.c (orc_lk_cn) compute the same thing: every window sum is an exact integer, and the
float steps are the same unfused IEEE operations.  So nextPts, status, err and the iteration counts must agree exactly,
with no tolerance.  BASELINE's cv2 tolerances in parity.py would hide a bug that moves a fraction of a percent of the
points, or moves positions by less than 0.01 px.

A seeded generator draws frames, windows, criteria, flags, points and initial guesses.  It reaches the paths that few
points take: border bands at every level (the TMA patch mirrored in shared memory, the REFLECT_101 gather far outside), J
patch re-staging after drifts of more than 3 px, the generic and split-template kernels, flat windows, min-eigenvalue
rejections, and non-finite points.  The committed seeds run in about a minute on one B200; IBT_LK_EXACT_SEEDS=N runs
seeds 0..N-1 for a soak.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from parity import _f32_same, assert_lk_exact

pytestmark = pytest.mark.gpu

INIT, MINEIG = 4, 8                     # cv2.OPTFLOW_USE_INITIAL_FLOW, cv2.OPTFLOW_LK_GET_MIN_EIGENVALS
SEEDS = range(int(os.environ.get("IBT_LK_EXACT_SEEDS", "8")))
NONFINITE = [(np.nan, 40.0), (40.0, np.nan), (np.nan, np.nan), (np.inf, 40.0), (40.0, -np.inf), (3e9, 40.0),
             (40.0, -3e9), (1e30, 1e30), (-np.inf, np.inf)]


# ---- scenes -------------------------------------------------------------------------------------------------------------
def _texture(rng, h, w):
    """band-limited random texture with block corners (u8): what LK locks on"""
    a = rng.random((h + 8, w + 8)).astype(np.float32)
    for _ in range(2):
        a = (a + np.roll(a, 1, 0) + np.roll(a, 1, 1) + np.roll(np.roll(a, 1, 0), 1, 1)) * 0.25
    a = a[4:4 + h, 4:4 + w]
    a = (a - a.min()) / max(float(a.max() - a.min()), 1e-9)
    blocks = np.kron((rng.random((h // 7 + 2, w // 7 + 2)) > 0.5).astype(np.float32), np.ones((7, 7), np.float32))[:h, :w]
    return np.clip(a * 170 + blocks * 70 + rng.normal(0, 2, (h, w)), 0, 255).astype(np.float32)


def _flat(rng, h, w):
    """texture with a flat plateau over its middle third (windows there have D < FLT_EPSILON)"""
    a = _texture(rng, h, w)
    a[h // 3:max(h // 3 + 1, 2 * h // 3), w // 3:max(w // 3 + 1, 2 * w // 3)] = 128
    return a


def _steps(rng, h, w):
    """0 / 255 rectangles: step edges, the largest Scharr responses"""
    a = np.zeros((h, w), np.float32)
    for _ in range(max(3, h * w // 900)):
        y, x = rng.integers(0, h), rng.integers(0, w)
        a[y:y + rng.integers(3, 40), x:x + rng.integers(3, 40)] = 255 * rng.integers(0, 2)
    return a


SCENES = {"tex": _texture, "flat": _flat, "steps": _steps}


def _shift(a, dx, dy):
    """a displaced by (dx, dy) px, bilinear, borders replicated, rounded to u8"""
    h, w = a.shape
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float64)
    x, y = xs - dx, ys - dy
    x0, y0 = np.floor(x), np.floor(y)
    fx, fy = x - x0, y - y0
    xi = lambda v: np.clip(v, 0, w - 1).astype(np.int64)
    yi = lambda v: np.clip(v, 0, h - 1).astype(np.int64)
    v = ((1 - fx) * (1 - fy) * a[yi(y0), xi(x0)] + fx * (1 - fy) * a[yi(y0), xi(x0 + 1)] +
         (1 - fx) * fy * a[yi(y0 + 1), xi(x0)] + fx * fy * a[yi(y0 + 1), xi(x0 + 1)])
    return np.clip(np.rint(v), 0, 255).astype(np.uint8)


def _frames(rng, scene, h, w, cn, shift):
    I, J = [], []
    for _ in range(cn):
        a = SCENES[scene](rng, h, w)
        I.append(np.clip(np.rint(a), 0, 255).astype(np.uint8))
        J.append(_shift(a, *shift))
    if cn == 1:
        return I[0], J[0]
    return np.stack(I, -1), np.stack(J, -1)


# ---- points -------------------------------------------------------------------------------------------------------------
def _points(rng, h, w, win, sizes, n_in):
    """-> (pts (N,2) f32, band (N,) bool: the point lies in a level-0 border band).  Interior points, integer and
    half-integer positions, border bands x = (e + o) * 2^l (e in {0, cols_l - 1}, o in [-winW - 2, 2], half a pixel on or
    not) at every level, the same in y, corners, the exact bounds of the window test (ipx = -winW is in, -winW - 1 is out;
    ipx = cols - 1 is in, cols is out) at every level, and non-finite coordinates."""
    hx, hy = (win[0] - 1) * 0.5, (win[1] - 1) * 0.5
    P = [rng.uniform([0, 0], [w, h], (n_in, 2))]
    q = rng.integers([0, 0], [w, h], (max(8, n_in // 8), 2)).astype(np.float64)
    P += [q, q + 0.5]
    nb = len(np.concatenate(P))
    for l, (hl, wl) in enumerate(sizes):
        s = float(2 ** l)
        for axis, (n_l, other) in enumerate(((wl, h), (hl, w))):
            e = np.array([(e + o) for e in (0, n_l - 1) for o in range(-win[axis] - 2, 3)], np.float64)
            e = np.concatenate([e, e + 0.5])
            half = hx if axis == 0 else hy
            exact = np.array([-win[axis] + half, -win[axis] + half - 0.25, n_l - 1 + half + 0.5, n_l + half], np.float64)
            c = np.concatenate([e, exact]) * s
            o = rng.uniform(0, other, len(c))
            P.append(np.c_[c, o] if axis == 0 else np.c_[o, c])
        cx = np.array([-2, -0.5, 0, 1, wl - 2, wl - 1, wl - 0.5, wl + 1], np.float64) * s
        cy = np.array([-2, -0.5, 0, 1, hl - 2, hl - 1, hl - 0.5, hl + 1], np.float64) * s
        P.append(np.stack(np.meshgrid(cx, cy), -1).reshape(-1, 2))
        if l == 0:
            band_end = len(np.concatenate(P))
    P.append(np.array(NONFINITE))
    pts = np.concatenate(P).astype(np.float32)
    band = np.zeros(len(pts), bool)
    band[nb:band_end] = True
    return pts, band


def _guesses(rng, pts, shift, h, w):
    """initial flow: exact, +-0.5 px off, 4-10 px off, outside the image, NaN (one kind per point, cycling)"""
    n = len(pts)
    g = pts.astype(np.float64) + shift
    kind = np.arange(n) % 6
    g[kind == 1] += rng.choice([-0.5, 0.5], (int((kind == 1).sum()), 2))
    off = rng.uniform(4, 10, (int((kind == 2).sum()), 2)) * rng.choice([-1, 1], (int((kind == 2).sum()), 2))
    g[kind == 2] += off
    g[kind == 3] = rng.uniform([-3 * w, -3 * h], [-w, -h], (int((kind == 3).sum()), 2)) * rng.choice([-1, 1], (int((kind == 3).sum()), 1))
    g[kind == 4, rng.integers(0, 2)] = np.nan
    return g.astype(np.float32)


# ---- cases --------------------------------------------------------------------------------------------------------------
# (entry, (h, w), cn, scene, shift, winSize, maxLevel, criteria, minEigThreshold, flags, interior points)
# entry: "np" = numpy frames, "pyr" = FramePyramid objects, "fb" = calcOpticalFlowPyrLK_FB
FIXED = [
    ("np", (240, 321), 1, "tex", (0.3, -0.7), (21, 21), 3, (3, 30, 0.01), 1e-4, 0, 600),
    ("pyr", (240, 321), 1, "tex", (25.0, -12.5), (21, 21), 4, (3, 30, 0.01), 1e-4, INIT, 400),
    ("np", (257, 383), 1, "tex", (6.0, -5.0), (31, 31), 0, (3, 30, 0.01), 1e-4, 0, 400),
    ("pyr", (257, 383), 1, "steps", (4.5, 7.25), (35, 35), 0, (1, 100, 0.0), 1e-4, INIT, 300),
    ("np", (97, 131), 1, "tex", (0.6, 0.2), (35, 35), 7, (2, 0, 1e-3), 0.0, MINEIG, 300),
    ("np", (97, 131), 1, "flat", (0.25, -0.5), (3, 3), 2, (3, 2, 0.3), 1e-2, INIT | MINEIG, 300),
    ("np", (5, 7), 1, "tex", (0.5, 0.25), (21, 21), 3, (3, 30, 0.01), 1e-4, 0, 40),
    ("np", (9, 130), 1, "tex", (1.5, 0.5), (4, 4), 5, (3, 150, 20.0), 0.0, INIT, 100),
    ("np", (130, 9), 1, "steps", (0.5, 1.5), (5, 61), 1, (1, 0, 0.01), 1e-4, MINEIG, 100),
    ("np", (24, 24), 1, "tex", (0.75, -0.25), (61, 5), 2, (3, 1, 0.0), 1e-4, INIT, 100),
    ("np", (40, 37), 1, "flat", (0.4, 0.4), (33, 32), 3, (3, 30, 0.01), 1.0, 0, 100),
    ("pyr", (240, 321), 1, "steps", (7.5, -4.0), (63, 63), 2, (3, 30, 0.01), 1e-4, INIT, 200),
    ("pyr", (240, 321), 1, "flat", (30.0, 17.0), (31, 31), 4, (3, 100, 1e-3), 1e-4, 0, 400),
    ("np", (97, 131), 1, "tex", (2.0, 1.0), (21, 21), 0, (3, 2, 0.0), 1e-4, 0, 200),
    ("np", (1080, 1920), 1, "tex", (12.0, -30.0), (21, 21), 3, (3, 30, 0.01), 1e-4, 0, 1500),
    ("np", (240, 321), 3, "tex", (15.0, 8.0), (21, 21), 3, (3, 30, 0.01), 1e-4, 0, 300),
    ("np", (97, 131), 2, "steps", (6.0, -4.0), (9, 15), 0, (3, 30, 0.01), 1e-4, INIT, 200),
    ("pyr", (257, 383), 4, "flat", (0.3, 0.6), (31, 31), 7, (3, 30, 0.01), 1e-4, INIT | MINEIG, 150),
    ("np", (24, 24), 3, "tex", (0.5, 0.5), (35, 35), 1, (3, 100, 0.0), 1e-2, 0, 60),
    ("fb", (240, 321), 1, "tex", (20.0, -10.0), (31, 31), 4, (3, 30, 0.01), 1e-4, 0, 400),
    ("fb", (130, 9), 1, "tex", (0.5, 2.0), (5, 5), 2, (3, 30, 0.01), 1e-4, 0, 100),
    ("fb", (257, 383), 3, "steps", (3.0, -2.5), (35, 35), 3, (3, 30, 0.01), 1e-4, 0, 150),
    ("fb", (97, 131), 4, "tex", (5.0, 6.0), (63, 63), 0, (3, 30, 0.01), 1e-4, 0, 60),
    ("fb", (257, 383), 1, "flat", (4.0, 5.0), (21, 21), 0, (3, 30, 0.01), 1e-4, 0, 300),
]


def _random_cases(rng, k):
    """k cases with a random window (3..63)^2 and random parameters from the issue's lists"""
    out = []
    for i in range(k):
        entry = ["np", "pyr", "fb", "np"][i % 4]
        cn = int(rng.choice([1, 1, 2, 3, 4]))
        hw = [(97, 131), (240, 321), (257, 383), (40, 37)][int(rng.integers(0, 4))]
        win = (int(rng.integers(3, 64)), int(rng.integers(3, 64)))
        shift = tuple(float(v) for v in rng.choice([rng.uniform(-1, 1, 2), rng.uniform(-8, 8, 2), rng.uniform(-40, 40, 2)]))
        crit = (int(rng.integers(1, 4)), int(rng.choice([0, 1, 2, 30, 100, 150])), float(rng.choice([0, 1e-3, 0.01, 0.3, 20])))
        flags = 0 if entry == "fb" else int(rng.choice([0, INIT, MINEIG, INIT | MINEIG]))
        out.append((entry, hw, cn, str(rng.choice(list(SCENES))), shift, win, int(rng.integers(0, 8)), crit,
                    float(rng.choice([0, 1e-4, 1e-2, 1])), flags, 150))
    return out


def _criteria_count(crit):
    return min(max(crit[1], 0), 100) if crit[0] & 1 else 30


def _run_case(ibt, oracle, rng, case, stats):
    entry, (h, w), cn, scene, shift, win, maxLevel, crit, mineig, flags, n_in = case
    I, J = _frames(rng, scene, h, w, cn, shift)
    ml, sizes = oracle.pyramid_sizes(h, w, win, maxLevel)
    pts, band = _points(rng, h, w, win, sizes, n_in)
    guess = _guesses(rng, pts, shift, h, w) if flags & INIT else None
    lp = dict(winSize=win, maxLevel=maxLevel, criteria=crit, minEigThreshold=mineig)
    what = "%s %dx%d cn %d %s shift %s win %s maxLevel %d (levels %s) criteria %s minEig %g flags %d" % (
        entry, h, w, cn, scene, shift, win, maxLevel, sizes, crit, mineig, flags)
    po, so, eo, io = oracle.calcOpticalFlowPyrLK(I, J, pts, None if guess is None else guess.copy(), flags=flags,
                                                return_iters=True, **lp)
    ref = dict(p1=po, st=so, err=eo, iters=io)
    if entry == "fb":
        r = ibt.calcOpticalFlowPyrLK_FB(I, J, pts, fb_threshold=1.0, return_iters=True, **lp)
        pr, sr, er, ir = oracle.calcOpticalFlowPyrLK(J, I, po, None, return_iters=True, **lp)
        assert_lk_exact(dict(p1=r["p1"], st=r["st1"], err=r["err1"], iters=r["iters"][:, 0]), ref, what + " forward", pts)
        assert_lk_exact(dict(p1=r["p0r"], st=r["st0"], err=r["err0"], iters=r["iters"][:, 1]),
                        dict(p1=pr, st=sr, err=er, iters=ir), what + " backward", po)
        _check_fb(r, pts, pr, what)
        got = dict(p1=r["p1"], st=r["st1"], iters=r["iters"][:, 0])
    else:
        a, b = (I, J) if entry == "np" else (ibt.FramePyramid(I, win, maxLevel, True), ibt.FramePyramid(J, win, maxLevel, False))
        p1, st, err, it = ibt.calcOpticalFlowPyrLK(a, b, pts, guess, winSize=win, maxLevel=maxLevel, criteria=crit,
                                                   flags=flags, minEigThreshold=mineig, return_iters=True)
        got = dict(p1=p1, st=st, err=err, iters=it)
        assert_lk_exact(got, ref, what, pts, guess)
    # what the case reached
    st = np.asarray(got["st"]).reshape(-1)
    stats["st0"] += int((st == 0).sum())
    stats["st1"] += int((st == 1).sum())
    stats["band_st0"] += int((st[band] == 0).sum())
    stats["band_st1"] += int((st[band] == 1).sum())
    if ml == 0:
        start = pts if guess is None else guess
        moved = np.abs(np.asarray(got["p1"]).reshape(-1, 2) - start).max(1)
        stats["restaged"] += int(((st == 1) & (moved > 3)).sum())
        mc, it = _criteria_count(crit), np.asarray(got["iters"]).reshape(-1)
        if mc >= 2:
            stats["at_max"] += int(((st == 1) & (it == mc)).sum())
            stats["early"] += int(((st == 1) & (it > 0) & (it < mc)).sum())


def _check_fb(r, pts, p0r_o, what):
    """dist = hypot(|p0 - p0r|) is numpy's float32 hypot bit for bit (the kernel restates glibc's hypotf), NaN included, and
    valid = dist < 1 on every point"""
    d = np.abs(pts - p0r_o.reshape(-1, 2)).astype(np.float32)
    d_o = np.hypot(d[:, 0], d[:, 1]).astype(np.float32)
    dist, valid = np.asarray(r["dist"]).reshape(-1), np.asarray(r["valid"]).reshape(-1)
    bad = np.flatnonzero(~_f32_same(dist, d_o))
    assert not len(bad), "%s: FB distance differs from numpy's hypot at %s (gpu %s, numpy %s)" % (
        what, bad[:6].tolist(), dist[bad[:6]].tolist(), d_o[bad[:6]].tolist())
    bad = np.flatnonzero(valid != (d_o < 1))
    assert not len(bad), "%s: FB valid differs at %s (dist %s)" % (what, bad[:6].tolist(), d_o[bad[:6]].tolist())


@pytest.mark.parametrize("seed", SEEDS)
def test_lk_exact_fuzz(ibt, oracle, seed):
    rng = np.random.default_rng(7000 + seed)
    stats = dict(st0=0, st1=0, band_st0=0, band_st1=0, restaged=0, at_max=0, early=0)
    for case in FIXED + _random_cases(rng, 6):
        _run_case(ibt, oracle, rng, case, stats)
    # the generator reaches what it is written for
    assert stats["st0"] > 0 and stats["st1"] > 0, stats
    assert stats["band_st0"] > 0 and stats["band_st1"] > 0, stats
    assert stats["restaged"] > 0, stats
    assert stats["at_max"] > 0 and stats["early"] > 0, stats


# ---- non-finite points: cv2 gives status 0, err 0 and the propagated input ------------------------------------------------
@pytest.mark.parametrize("cn", [1, 3])
def test_lk_non_finite_points(ibt, oracle, cn):
    """NaN, +-inf, +-3e9 and 1e30 coordinates (and NaN initial guesses): the window is out of bounds at every level, as with
    cv2 (its cvFloor gives INT_MIN for NaN), so status is 0, err 0 and nextPts the input, or the guess, scaled down and back up."""
    rng = np.random.default_rng(5)
    I, J = _frames(rng, "tex", 97, 131, cn, (0.5, 0.25))
    good = np.array([[60.25, 50.5], [30.0, 70.0]], np.float32)
    pts = np.concatenate([np.array(NONFINITE, np.float32), good])
    nf = len(NONFINITE)
    for maxLevel in (0, 3):
        for flags in (0, MINEIG, INIT, INIT | MINEIG):
            lp = dict(winSize=(21, 21), maxLevel=maxLevel, criteria=(3, 30, 0.01))
            guess = np.concatenate([good[:1].repeat(nf, 0), np.array([[np.nan, 50.0], [30.5, np.nan]], np.float32)]) if flags & INIT else None
            what = "cn %d maxLevel %d flags %d" % (cn, maxLevel, flags)
            p1, st, err, it = ibt.calcOpticalFlowPyrLK(I, J, pts, guess, flags=flags, return_iters=True, **lp)
            po, so, eo, io = oracle.calcOpticalFlowPyrLK(I, J, pts, None if guess is None else guess.copy(), flags=flags,
                                                        return_iters=True, **lp)
            assert_lk_exact(dict(p1=p1, st=st, err=err, iters=it), dict(p1=po, st=so, err=eo, iters=io), what, pts, guess)
            assert not st.any() if flags & INIT else not st[:nf].any(), (what, st.ravel().tolist())
            assert (err[:nf] == 0).all() and (it[:nf] == 0).all(), what
            assert _f32_same(p1, guess).all() if flags & INIT else _f32_same(p1[:nf], pts[:nf]).all(), (what, p1.tolist())
        if cn == 1:
            r = ibt.calcOpticalFlowPyrLK_FB(I, J, pts, return_iters=True, **lp)
            assert not r["st1"][:nf].any() and (r["err1"][:nf] == 0).all()
            # p0r = p1 = p0: the FB distance is 0 for the finite ones (3e9, 1e30), NaN for the others
            assert np.array_equal(r["valid"][:nf], np.isfinite(pts[:nf]).all(1))
            assert _f32_same(r["p1"][:nf], pts[:nf]).all()


# ---- status / err buffers left out -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("win", [(21, 21), (17, 23)])
def test_lk_null_status_err(ibt, oracle, win):
    """ibt_lk with err = NULL (the err stage is skipped, the final bounds test still sets status), and with status and err
    NULL (the whole final stage is skipped): p1 and status equal the full call's."""
    from iceberg_tracking_code_b200 import _native as N
    rng = np.random.default_rng(9)
    I, J = _frames(rng, "tex", 240, 321, 1, (6.5, -3.25))
    ml, sizes = oracle.pyramid_sizes(240, 321, win, 2)
    pts, _ = _points(rng, 240, 321, win, sizes, 400)
    pa, pb = ibt.FramePyramid(I, win, 2, True), ibt.FramePyramid(J, win, 2, False)
    p1, st, _ = ibt.calcOpticalFlowPyrLK(pa, pb, pts, None, winSize=win, maxLevel=2)
    st = st.reshape(-1)
    assert 0 < int(st.sum()) < len(st)
    d = torch.from_numpy(pts).cuda()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for with_status in (True, False):
        q = torch.empty((len(pts), 2), dtype=torch.float32, device="cuda")
        qs = torch.full((len(pts),), 0xEE, dtype=torch.uint8, device="cuda")
        rc = N.lib().ibt_lk(C.byref(pa.c), C.byref(pb.c), d.data_ptr(), q.data_ptr(), len(pts), win[0], win[1], 30, 0.01, 1e-4,
                            0, qs.data_ptr() if with_status else None, None, None, s)
        assert rc == 0
        assert _f32_same(q.cpu().numpy(), p1).all(), with_status
        if with_status:
            qs = qs.cpu().numpy()
            assert np.array_equal(qs, st), int((qs != st).sum())
