"""GPU: pyramids of 2- to 4-channel frames (ibt_pyramid_build_multichannel), colour FramePyramids reused by
calcOpticalFlowPyrLK, and forward-backward tracking of colour frames in one launch (ibt_lk_fb_multichannel).

cv2 builds a multi-channel frame's pyramid channel by channel: level l of channel c is the gray pyramid of plane c, and
derivative channels 2c, 2c+1 are that plane's Scharr (dx, dy) (pinned without a GPU in test_multichannel_host.py).  Where
cv2 does not import, the CPU oracle's gray pyramid of each plane is the reference."""
import ctypes as C

import numpy as np
import pytest
import torch

import multichannel_cases as MC
from parity import ERR_TOL, LK_SETS, _f32_same, assert_lk_parity
from test_gpu_layouts import Placed, _ok, _ru, _same, _stream

pytestmark = pytest.mark.gpu

SIZES = [(1, 37), (29, 1), (2, 9), (63, 127), (64, 128), (65, 129), (64, 129), (65, 127), (257, 383)]


def _reference_pyramid(oracle, f, win, maxLevel, derivs):
    """cv2.buildOpticalFlowPyramid(f) where cv2 imports, else the oracle's gray pyramid of every plane, interleaved like cv2"""
    try:
        import cv2
        ml, p = cv2.buildOpticalFlowPyramid(f, win, maxLevel, withDerivatives=derivs)
        return ml, [np.ascontiguousarray(a) for a in p]
    except ImportError:
        pass
    per = [oracle.buildOpticalFlowPyramid(np.ascontiguousarray(f[..., c]), win, maxLevel, derivs) for c in range(f.shape[2])]
    ml, k = per[0][0], 2 if derivs else 1
    out = []
    for l in range(ml + 1):
        out.append(np.stack([p[1][k * l] for p in per], -1))
        if derivs:
            out.append(np.concatenate([p[1][k * l + 1] for p in per], -1))
    return ml, out


def _check(ibt, oracle, f, win, maxLevel, derivs, what):
    ml_r, ref = _reference_pyramid(oracle, f, win, maxLevel, derivs)
    ml, out = ibt.buildOpticalFlowPyramid(f, win, maxLevel, derivs)
    assert ml == ml_r and len(out) == len(ref), what
    for i, (a, b) in enumerate(zip(out, ref)):
        assert a.shape == b.shape and a.dtype == b.dtype, (what, i, a.shape, b.shape)
        assert np.array_equal(a, b), (what, i)


@pytest.mark.parametrize("cn", [2, 3, 4])
def test_pyramid_vs_cv2(ibt, oracle, cn):
    """every level, every derivative array and the returned maxLevel, with and without derivatives: thin frames, tile edges"""
    rng = np.random.default_rng(40 + cn)
    for h, w in SIZES:
        f = rng.integers(0, 256, (h, w, cn), dtype=np.uint8)
        for derivs in (True, False):
            _check(ibt, oracle, f, (3, 3), 5, derivs, (cn, h, w, derivs))
        _check(ibt, oracle, f, (21, 21), 3, True, (cn, h, w, "win 21"))


def test_pyramid_24mp_vs_cv2(ibt, oracle):
    rng = np.random.default_rng(24)
    base = rng.integers(0, 256, (500, 750, 3), dtype=np.uint8)
    f = np.ascontiguousarray(np.kron(base, np.ones((8, 8, 1), np.uint8)) ^ rng.integers(0, 32, (4000, 6000, 3), dtype=np.uint8))
    _check(ibt, oracle, f, (31, 31), 4, True, "24 MP")


# ---- layouts through ctypes ------------------------------------------------------------------------------------------
def _mc_build(N, frame, cn, h, w, win, maxLevel, plane_off, plane_extra, derivs=True):
    """pyramid of `frame` (a Placed) in Placed planes: level pitches round_up(w, 16) + plane_extra, derivative pitches
    round_up(4w, 16) + 4 * plane_extra, every buffer at byte offset plane_off"""
    sizes = (C.c_int * (2 * N.IBT_MAX_LEVELS))()
    ml = N.lib().ibt_pyramid_levels(h, w, win[0], win[1], maxLevel, sizes)
    shapes = [(sizes[2 * l], sizes[2 * l + 1]) for l in range(ml + 1)]
    planes = [[Placed((lh, lw), torch.uint8, plane_off, _ru(lw, 16) + plane_extra) for lh, lw in shapes] for _ in range(cn)]
    ders = [[Placed((lh, lw, 2), torch.int16, 4 * plane_off, _ru(4 * lw, 16) + 4 * plane_extra) for lh, lw in shapes]
            for _ in range(cn)] if derivs else None
    structs = []
    for c in range(cn):
        st = N.ibt_pyramid_t()
        st.nlevels = ml + 1
        for l, (lh, lw) in enumerate(shapes):
            st.rows[l], st.cols[l] = lh, lw
            st.img[l], st.img_pitch[l] = planes[c][l].ptr, planes[c][l].pitch
            if derivs:
                st.deriv[l], st.deriv_pitch[l] = ders[c][l].ptr, ders[c][l].pitch
        structs.append(st)
    PP = C.POINTER(N.ibt_pyramid_t)
    arr = (PP * cn)(*[C.pointer(s) for s in structs])
    _ok(N.lib().ibt_pyramid_build_multichannel(C.c_void_p(frame.ptr), frame.pitch, cn, arr, int(derivs), _stream()),
        "ibt_pyramid_build_multichannel")
    torch.cuda.synchronize()
    return planes, ders


@pytest.mark.parametrize("cn", [3, 4])
def test_frame_any_layout(ibt, cn, monkeypatch):
    """frame views at byte offsets 0..15 and pitches that are not multiples of 16 (byte path), planes at odd offsets and
    pitches (byte / scalar paths at every level), the 16-byte paths with and without tensor maps: identical outputs, and no
    byte outside the logical rows of any buffer changes (the frame's included)"""
    from iceberg_tracking_code_b200 import _native as N
    rng = np.random.default_rng(7 + cn)
    h, w, win = 70, 301, (5, 5)
    img = rng.integers(0, 256, (h, w, cn), dtype=np.uint8)
    canon_f = Placed((h, w, cn), torch.uint8, 0, _ru(w * cn, 16), img)
    canon, canon_d = _mc_build(N, canon_f, cn, h, w, win, 3, 0, 0)
    ref = [[p.np() for p in ch] for ch in canon] + [[d.np() for d in ch] for ch in canon_d]
    cases = [(off, w * cn + extra, 0, 0) for off in range(16) for extra in (0, 5)]
    cases += [(16, _ru(w * cn, 16) + 32, 0, 0), (0, _ru(w * cn, 16), 3, 7), (5, w * cn + 1, 1, 3)]
    for tma in (True, False):
        if not tma:
            monkeypatch.setenv("IBT_NO_TMA", "1")        # levels >= 1 of the aligned cases: cp.async instead of tensor maps
        for foff, fpitch, poff, pextra in cases:
            fr = Placed((h, w, cn), torch.uint8, foff, fpitch, img)
            planes, ders = _mc_build(N, fr, cn, h, w, win, 3, poff, pextra)
            got = [[p.np() for p in ch] for ch in planes] + [[d.np() for d in ch] for ch in ders]
            assert all(_same(a, b) for ga, ra in zip(got, ref) for a, b in zip(ga, ra)), (foff, fpitch, poff, pextra)
            assert fr.intact() and np.array_equal(fr.np(), img), (foff, fpitch)
            assert all(p.intact() for ch in planes + ders for p in ch), (foff, fpitch, poff, pextra)


# ---- pyramid reuse and forward-backward ------------------------------------------------------------------------------
class _ViaPyramids:
    """calcOpticalFlowPyrLK with multi-channel frames turned into FramePyramids first (cv2's other input form)"""

    def __init__(self, ibt):
        self.ibt = ibt

    def calcOpticalFlowPyrLK(self, f0, f1, pts, nxt=None, **kw):
        if f0.ndim == 3 and f0.shape[2] > 1:
            f0 = self.ibt.FramePyramid(f0, kw["winSize"], kw["maxLevel"], True)
            f1 = self.ibt.FramePyramid(f1, kw["winSize"], kw["maxLevel"], False)
        return self.ibt.calcOpticalFlowPyrLK(f0, f1, pts, nxt, **kw)


def test_lk_on_colour_pyramids_golden(ibt, golden):
    """calcOpticalFlowPyrLK on colour FramePyramids == cv2's recorded answers (the multi-channel golden checks), and bit for
    bit == the same call on the colour arrays"""
    g = golden("kat_multichannel.npz")
    MC.check_multichannel_golden(_ViaPyramids(ibt), g)
    f0, f1, pts = g["f0"], g["f1"], g["pts"]
    for lp in MC.MC_SETS:
        a = ibt.calcOpticalFlowPyrLK(f0, f1, pts, None, return_iters=True, **lp)
        b = _ViaPyramids(ibt).calcOpticalFlowPyrLK(f0, f1, pts, None, return_iters=True, **lp)
        assert all(_same(x, y) for x, y in zip(a, b)), lp


def _fb_reference(ibt, f0, f1, pts, lp):
    p1, st1, err1 = ibt.calcOpticalFlowPyrLK(f0, f1, pts, None, **lp)
    p0r, st0, err0 = ibt.calcOpticalFlowPyrLK(f1, f0, p1, None, **lp)
    d = (pts - p0r).reshape(-1, 2)
    return p1, st1, err1, p0r, st0, err0, np.hypot(np.abs(d[:, 0]), np.abs(d[:, 1])).astype(np.float32)


@pytest.mark.parametrize("cn", [2, 3, 4])
def test_fb_one_launch_equals_two_calls(ibt, golden, cn):
    g = golden("kat_multichannel.npz")
    f0, f1, pts = g["f0"], g["f1"], g["pts"]
    if cn != 3:
        f0, f1 = np.ascontiguousarray(np.dstack([f0, f0[..., 0]])[..., :cn]), np.ascontiguousarray(np.dstack([f1, f1[..., 1]])[..., :cn])
    for lp in MC.MC_SETS:
        p1, st1, err1, p0r, st0, err0, dist = _fb_reference(ibt, f0, f1, pts, lp)
        r = ibt.calcOpticalFlowPyrLK_FB(f0, f1, pts, **lp)
        for k, v in dict(p1=p1, st1=st1, err1=err1, p0r=p0r, st0=st0, err0=err0).items():
            assert _same(r[k], v), (cn, lp, k)
        assert _f32_same(r["dist"], dist).all() and np.array_equal(r["valid"], dist < 1), (cn, lp)
        # FramePyramids of the frames give the same launch
        pa, pb = (ibt.FramePyramid(f, lp["winSize"], lp["maxLevel"], True) for f in (f0, f1))
        q = ibt.calcOpticalFlowPyrLK_FB(pa, pb, pts, **lp)
        assert all(_same(q[k], r[k]) for k in r), (cn, lp)


def test_fb_alive_and_cv2(ibt, golden):
    """alive in/out as in the gray path (dead points are skipped, their outputs untouched); cv2's two calls + numpy FB within
    the suite's LK tolerances"""
    g = golden("kat_multichannel.npz")
    f0, f1, pts = (torch.from_numpy(g[k]).cuda() for k in ("f0", "f1", "pts"))
    lp = MC.MC_SETS[0]
    n = pts.shape[0]
    alive = torch.ones(n, dtype=torch.uint8, device="cuda")
    alive[::3] = 0
    dead = alive == 0
    full = ibt.calcOpticalFlowPyrLK_FB(f0, f1, pts, **lp)
    pa, pb = (ibt.FramePyramid(f, lp["winSize"], lp["maxLevel"], True) for f in (f0, f1))
    from iceberg_tracking_code_b200 import _native as N
    p1 = torch.full((n, 2), -7.0, device="cuda")
    dist = torch.full((n,), -7.0, device="cuda")
    total = torch.zeros(1, dtype=torch.int64, device="cuda")
    tail = (C.c_void_p(pts.data_ptr()), n, lp["winSize"][0], lp["winSize"][1], 30, 0.01, 1e-4, 1.0, C.c_void_p(p1.data_ptr()),
            None, None, None, None, None, C.c_void_p(dist.data_ptr()), C.c_void_p(alive.data_ptr()), None,
            C.c_void_p(total.data_ptr()), _stream())
    a0 = alive.clone()
    _ok(N.lib().ibt_lk_fb_multichannel(pa.chan_ptrs, pb.chan_ptrs, 3, *tail), "ibt_lk_fb_multichannel")
    torch.cuda.synchronize()
    assert bool((p1[dead] == -7.0).all()) and bool((dist[dead] == -7.0).all()) and bool((alive[dead] == 0).all())
    live = ~dead
    assert torch.equal(p1[live], full["p1"].reshape(n, 2)[live]) and torch.equal(dist[live], full["dist"][live])
    assert torch.equal(alive[live].bool(), full["valid"][live] & a0[live].bool())
    assert int(total.item()) > 0
    cv2 = pytest.importorskip("cv2")
    a, b, p = g["f0"], g["f1"], g["pts"]
    for lp in MC.MC_SETS:
        c1, s1, _ = cv2.calcOpticalFlowPyrLK(a, b, p, None, **lp)
        c0, s0, _ = cv2.calcOpticalFlowPyrLK(b, a, c1, None, **lp)
        r = ibt.calcOpticalFlowPyrLK_FB(a, b, p, **lp)
        assert_lk_parity(r["p1"], r["st1"], c1, s1, "fwd %s" % (lp,))
        assert_lk_parity(r["p0r"], r["st0"], c0, s0, "bwd %s" % (lp,))


def test_rebuild_equals_fresh_build(ibt):
    rng = np.random.default_rng(5)
    win, ml = (21, 21), 3
    a, b = (rng.integers(0, 256, (301, 517, 3), dtype=np.uint8) for _ in range(2))
    p = ibt.FramePyramid(a, win, ml, True)
    bufs = [t.data_ptr() for t in p._img_buf + p._deriv_buf]
    p.rebuild(torch.from_numpy(b).cuda()[:, :, :])
    q = ibt.FramePyramid(b, win, ml, True)
    assert [t.data_ptr() for t in p._img_buf + p._deriv_buf] == bufs          # nothing reallocated
    for l in range(ml + 1):
        assert torch.equal(p.level(l), q.level(l)) and torch.equal(p.deriv(l), q.deriv(l)), l
    # a crop view of a larger device frame (row pitch, unaligned base) is used in place
    big = torch.from_numpy(rng.integers(0, 256, (320, 540, 3), dtype=np.uint8)).cuda()
    view = big[7:308, 3:520]
    p.rebuild(view)
    q = ibt.FramePyramid(view.contiguous(), win, ml, True)
    for l in range(ml + 1):
        assert torch.equal(p.level(l), q.level(l)) and torch.equal(p.deriv(l), q.deriv(l)), l
    with pytest.raises(ibt.error):
        p.rebuild(a[:, :, :2].copy())
