"""GPU: the C ABI's layout promise -- any pitch, any base alignment -- on every staging path of every entry point, and the
int32 headroom of the LK window sums.

Each kernel picks its staging path from the layout it is handed (16-byte vector loads, TMA tensor maps, 4-byte cp.async,
byte gathers; see include/ibt.h).  cv.py always hands over the same layouts, so here every entry point is called through
ctypes with buffers placed at chosen byte offsets and row pitches inside sentinel-filled allocations.  Every case is checked
against (a) the canonical aligned layout, bit for bit -- every path computes the same exact integer arithmetic -- and (b) the
CPU oracle; and no byte outside the logical rows of any buffer may change.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from parity import CORNER_OVERLAP, as_corners, assert_lk_exact, assert_lk_parity, corner_overlap

pytestmark = pytest.mark.gpu

SENT = 0xA5
INIT, MINEIG = 4, 8                     # IBT_LK_USE_INITIAL_FLOW, IBT_LK_GET_MIN_EIGENVALS
I32_MAX = 2 ** 31 - 1


def _N():
    from iceberg_tracking_code_b200 import _native
    return _native


def _lib():
    return _N().lib()


def _stream(s=None):
    return C.c_void_p((s or torch.cuda.current_stream()).cuda_stream)


def _ok(rc, what):
    assert rc == 0, "%s returned %d" % (what, rc)


def _ru(v, m):
    return (v + m - 1) // m * m


def _same(a, b):
    """bit-for-bit equality (NaN-safe)"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


class Placed:
    """An (h, w[, c]) array of `dtype` in a fresh device buffer: the logical data starts `off` bytes into the buffer, rows are
    `pitch` bytes apart, and every other byte of the buffer (before, between and after the rows) holds SENT."""

    def __init__(self, shape, dtype, off, pitch, data=None):
        item = torch.empty((), dtype=dtype).element_size()
        h = shape[0]
        rowbytes = int(np.prod(shape[1:])) * item
        assert pitch >= rowbytes and off % item == 0 and pitch % item == 0
        nbytes = _ru(off + (h - 1) * pitch + rowbytes + 64, 16)
        self.buf = torch.full((nbytes,), SENT, dtype=torch.uint8, device="cuda")
        logical = torch.zeros(nbytes, dtype=torch.bool, device="cuda")
        logical.as_strided((h, rowbytes), (pitch, 1), off).fill_(True)
        self.pad = ~logical
        inner = [int(np.prod(shape[i + 1:])) for i in range(1, len(shape))]
        self.view = self.buf.view(dtype).as_strided(tuple(shape), (pitch // item,) + tuple(inner), off // item)
        self.ptr = self.buf.data_ptr() + off
        self.pitch = pitch
        if data is not None:
            self.view.copy_(torch.as_tensor(np.ascontiguousarray(data)).to("cuda"))

    def np(self):
        return self.view.cpu().numpy()

    def intact(self):
        return bool((self.buf[self.pad] == SENT).all())


# ---- ibt_gray_u8 -----------------------------------------------------------------------------------------------------
GRAY_W = [1, 2, 15, 16, 17, 31, 33, 1920, 1921, 1935]


def _gray_layouts(W, cn):
    """(src off, src pitch, dst off, dst pitch): vector only / vector + scalar tail when W % 16 == 0 / != 0 (cn 3, all
    16-byte aligned), scalar only (odd offset or pitch), and the plain contiguous layout."""
    a16 = _ru(W * cn, 16)
    return [(0, a16, 0, _ru(W, 16)),                  # vector (+ tail)
            (16, a16 + 32, 32, _ru(W, 16) + 16),     # vector (+ tail), non-zero aligned offsets
            (0, a16, 3, W + 5),                      # destination unaligned -> scalar
            (1, W * cn + 3, 0, _ru(W, 16)),          # source unaligned -> scalar
            (0, W * cn, 0, W)]                       # contiguous


@pytest.mark.parametrize("cn", [3, 4])
def test_gray_any_layout(ibt, oracle, cn):
    rng = np.random.default_rng(cn)
    for W in GRAY_W:
        for H in (1, 5):
            rgb = rng.integers(0, 256, (H, W, cn), dtype=np.uint8)
            for cs in (0, 1):
                ref = oracle.cvtColor(rgb, coeffset=cs)
                for (so, sp, do, dp) in _gray_layouts(W, cn):
                    src = Placed((H, W, cn), torch.uint8, so, sp, rgb)
                    dst = Placed((H, W), torch.uint8, do, dp)
                    _ok(_lib().ibt_gray_u8(src.ptr, H, W, cn, sp, dst.ptr, dp, cs, _stream()), "ibt_gray_u8")
                    what = (W, H, cs, so, sp, do, dp)
                    assert np.array_equal(dst.np(), ref), what
                    assert dst.intact() and src.intact(), what


# ---- ibt_pyr_level_u8 ------------------------------------------------------------------------------------------------
# (1080, 1921): 16 x 17 = 272 tiles of 128 x 64, just below the big-tile switch at 2 * 148; (1200, 2049): 17 x 19 = 323, above
PYR_SIZES = [(1, 1), (2, 3), (7, 15), (8, 16), (9, 17), (64, 48), (333, 641), (1080, 1921), (1200, 2049)]


def _src_layout(w, aligned):
    return (0, _ru(w, 16) + 16) if aligned else (1, w + 2 if w % 2 else w + 1)          # odd offset and odd pitch


def _deriv_layout(w, aligned):
    return (0, _ru(4 * w, 16)) if aligned else (4, _ru(4 * w, 16) + 4)                  # pitch a multiple of 4, not of 16


def _down_layout(w, aligned):
    ow = (w + 1) // 2
    return (0, _ru(ow, 16)) if aligned else (1, ow + 1 if ow % 2 == 0 else ow + 2)     # odd offset and odd pitch


@pytest.mark.parametrize("hw", PYR_SIZES)
def test_pyr_level_any_layout(ibt, oracle, hw):
    h, w = hw
    rng = np.random.default_rng(h * 7919 + w)
    a = rng.integers(0, 256, hw, dtype=np.uint8)
    ref_d, ref_n = oracle.scharr_deriv(a), oracle.pyrDown(a)
    oh, ow = ref_n.shape
    for sa in (True, False):
        for da in (True, False):
            for na in (True, False):
                for outs in ("deriv", "down", "both"):
                    if (outs == "deriv" and not na) or (outs == "down" and not da):
                        continue                       # the absent output's layout does not matter
                    so, sp = _src_layout(w, sa)
                    src = Placed(hw, torch.uint8, so, sp, a)
                    der = dn = None
                    if outs != "down":
                        do, dp = _deriv_layout(w, da)
                        der = Placed((h, w, 2), torch.int16, do, dp)
                    if outs != "deriv":
                        no, npch = _down_layout(w, na)
                        dn = Placed((oh, ow), torch.uint8, no, npch)
                    _ok(_lib().ibt_pyr_level_u8(src.ptr, h, w, sp, der.ptr if der else None, der.pitch if der else 0,
                                                dn.ptr if dn else None, dn.pitch if dn else 0, _stream()), "ibt_pyr_level_u8")
                    what = (hw, sa, da, na, outs)
                    assert src.intact(), what
                    if der is not None:
                        assert np.array_equal(der.np(), ref_d), what
                        assert der.intact(), what
                    if dn is not None:
                        assert np.array_equal(dn.np(), ref_n), what
                        assert dn.intact(), what


# ---- ibt_pyramid_build -----------------------------------------------------------------------------------------------
def _pyr_struct(imgs, ders):
    st = _N().ibt_pyramid_t()
    st.nlevels = len(imgs)
    for l, im in enumerate(imgs):
        st.rows[l], st.cols[l] = im.view.shape[0], im.view.shape[1]
        st.img[l], st.img_pitch[l] = im.ptr, im.pitch
        if ders is not None and ders[l] is not None:
            st.deriv[l], st.deriv_pitch[l] = ders[l].ptr, ders[l].pitch
    return st


def test_pyramid_build_mixed_levels(ibt, oracle):
    """One hand-filled ibt_pyramid_t whose levels all take different staging paths."""
    h, w = 333, 1150                                     # level widths 1150, 575, 288, 144, 72
    a = np.random.default_rng(5).integers(0, 256, (h, w), dtype=np.uint8)
    ml, ref = oracle.buildOpticalFlowPyramid(a, (5, 5), 4, True)
    assert ml == 4
    img_lay = [lambda w: (1, w + 2 if w % 2 else w + 1),   # offset 1, odd pitch: byte path, no TMA
               lambda w: (0, _ru(w, 128)),                 # aligned: TMA
               lambda w: (0, _ru(w, 16) + 4),              # pitch = 4 (mod 16): word loads, no TMA
               lambda w: (2, _ru(w, 16) + 2),              # offset 2
               lambda w: (16, _ru(w, 16) + 16)]            # aligned, offset 16
    der_lay = [lambda w: (4, 4 * w + 4), lambda w: (0, _ru(4 * w, 128)), lambda w: (0, _ru(4 * w, 16) + 4),
               lambda w: (16, _ru(4 * w, 16)), lambda w: (4, _ru(4 * w, 16) + 12)]
    for with_derivs in (1, 0):
        imgs, ders = [], []
        for l in range(ml + 1):
            lh, lw = ref[2 * l].shape
            o, p = img_lay[l](lw)
            imgs.append(Placed((lh, lw), torch.uint8, o, p, a if l == 0 else None))
            o, p = der_lay[l](lw)
            ders.append(Placed((lh, lw, 2), torch.int16, o, p))
        st = _pyr_struct(imgs, ders)
        _ok(_lib().ibt_pyramid_build(C.byref(st), with_derivs, _stream()), "ibt_pyramid_build")
        for l in range(ml + 1):
            assert np.array_equal(imgs[l].np(), ref[2 * l]), (with_derivs, l)
            assert imgs[l].intact(), (with_derivs, l)
            if with_derivs:
                assert np.array_equal(ders[l].np(), ref[2 * l + 1]), l
            else:
                assert bool((ders[l].buf == SENT).all()), l            # nothing written at all
            assert ders[l].intact(), (with_derivs, l)


# ---- LK: one pyramid pair, five layouts --------------------------------------------------------------------------------
LK_H, LK_W = 360, 550                  # level widths 550, 275 (odd), 138, 69
LK_SHIFT = (5.25, -4.5)                # px: at maxLevel 0 Newton walks out of the staged patch (restage_sync)
LK_WINDOWS = [(21, 21), (31, 31), (35, 35), (9, 15), (33, 32), (5, 61), (63, 63)]
LK_CN = 4


def _lay_canon(w):
    return (0, _ru(w, 128), 0, _ru(4 * w, 128))          # TMA image + TMA Scharr (what FramePyramid allocates)


def _lay_i_tma(w):
    return (0, _ru(w, 16), 0, _ru(4 * w, 16) + 4)        # tensor maps for the image only: Scharr by cp.async (stage_deriv)


def _lay_d_tma(w):
    return (0, _ru(w, 16) + 4, 0, _ru(4 * w, 16))        # image pitch = 4 (mod 16): 4-byte cp.async; Scharr by TMA


def _lay_bytes(w):
    return (1, _ru(w, 16) + 16, 4, _ru(4 * w, 16) + 4)   # image at offset 1 (word_ok = 0): byte gather; no Scharr map


LK_LAYOUTS = {"canon": _lay_canon, "i_tma": _lay_i_tma, "d_tma": _lay_d_tma, "bytes": _lay_bytes,
              "mix": lambda w, l: [_lay_bytes, _lay_canon, _lay_i_tma, _lay_d_tma][l % 4](w)}


@pytest.fixture(scope="module")
def lk_scene(oracle):
    """cn channel planes of a frame pair (channel 0 is the gray pair), their oracle pyramids (maxLevel 3, every level
    kept), and points inside, near every border (reflectable windows) and beyond it."""
    from iceberg_tracking_code_b200 import synthetic as syn
    planes = []
    for c in range(LK_CN):
        base = syn.base_texture(LK_H, LK_W, 40 + c)
        planes.append((syn.frame_gray(base, 0).numpy(), syn.frame_gray(base, 1, *LK_SHIFT).numpy()))
    pyrs = []
    for a, b in planes:
        ml, pa = oracle.buildOpticalFlowPyramid(a, (3, 3), 3, True)
        _, pb = oracle.buildOpticalFlowPyramid(b, (3, 3), 3, True)
        assert ml == 3
        pyrs.append((pa, pb))
    rng = np.random.default_rng(11)
    h, w = LK_H, LK_W
    pts = [rng.uniform([40, 40], [w - 40, h - 40], (200, 2))]
    for lo, hi in ((-8, 40), (-70, -12)):                 # near (reflectable), beyond (gather / out of bounds)
        pts += [np.c_[rng.uniform(lo, hi, 40), rng.uniform(0, h, 40)], np.c_[w - 1 - rng.uniform(lo, hi, 40), rng.uniform(0, h, 40)],
                np.c_[rng.uniform(0, w, 40), rng.uniform(lo, hi, 40)], np.c_[rng.uniform(0, w, 40), h - 1 - rng.uniform(lo, hi, 40)]]
    pts = np.concatenate(pts).astype(np.float32)
    guess = (pts + np.float32(LK_SHIFT) + rng.normal(0, 0.7, pts.shape)).astype(np.float32)
    return dict(planes=planes, pyrs=pyrs, pts=pts, guess=guess)


def _placed_pyramids(scene, layout, nlev, cn):
    """[(I struct, J struct)] per channel for `layout`; the Placed buffers are kept alive in the returned list."""
    out = []
    for c in range(cn):
        pair = []
        for pyr in scene["pyrs"][c]:
            imgs, ders = [], []
            for l in range(nlev):
                im, dv = pyr[2 * l], pyr[2 * l + 1]
                f = LK_LAYOUTS[layout]
                io, ip, do, dp = f(im.shape[1], l) if layout == "mix" else f(im.shape[1])
                imgs.append(Placed(im.shape, torch.uint8, io, ip, im))
                ders.append(Placed(dv.shape, torch.int16, do, dp, dv))
            pair.append((_pyr_struct(imgs, ders), imgs + ders))
        out.append(pair)
    return out


def _lk_outputs(n, fb):
    f = lambda *s: torch.full(s, float("nan"), dtype=torch.float32, device="cuda")
    u = lambda: torch.full((n,), 0xEE, dtype=torch.uint8, device="cuda")
    i = lambda *s: torch.full(s, -7, dtype=torch.int32, device="cuda")
    if fb:
        return dict(p1=f(n, 2), st1=u(), err1=f(n), p0r=f(n, 2), st0=u(), err0=f(n), fbdist=f(n),
                    alive=torch.ones(n, dtype=torch.uint8, device="cuda"), iters=i(n, 2))
    return dict(p1=f(n, 2), st=u(), err=f(n), iters=i(n))


def _p(t):
    return t.data_ptr() if t is not None else None


def _run_lk(pyrs, pts, guess, win, flags, cn=1):
    n = pts.shape[0]
    o = _lk_outputs(n, False)
    if flags & INIT:
        o["p1"].copy_(guess)
    tail = (_p(pts), _p(o["p1"]), n, win[0], win[1], 30, 0.01, 1e-4, flags, _p(o["st"]), _p(o["err"]), _p(o["iters"]), _stream())
    if cn == 1:
        _ok(_lib().ibt_lk(C.byref(pyrs[0][0][0]), C.byref(pyrs[0][1][0]), *tail), "ibt_lk")
    else:
        PP = C.POINTER(_N().ibt_pyramid_t)
        arrI = (PP * cn)(*[C.pointer(pyrs[c][0][0]) for c in range(cn)])
        arrJ = (PP * cn)(*[C.pointer(pyrs[c][1][0]) for c in range(cn)])
        _ok(_lib().ibt_lk_multichannel(arrI, arrJ, cn, *tail), "ibt_lk_multichannel")
    return {k: v.cpu().numpy() for k, v in o.items()}


def _run_lk_fb(pyrs, pts, win):
    n = pts.shape[0]
    o = _lk_outputs(n, True)
    tot = torch.zeros(1, dtype=torch.int64, device="cuda")
    _ok(_lib().ibt_lk_fb(C.byref(pyrs[0][0][0]), C.byref(pyrs[0][1][0]), _p(pts), n, win[0], win[1], 30, 0.01, 1e-4, 1.0,
                         _p(o["p1"]), _p(o["st1"]), _p(o["err1"]), _p(o["p0r"]), _p(o["st0"]), _p(o["err0"]), _p(o["fbdist"]),
                         _p(o["alive"]), _p(o["iters"]), _p(tot), _stream()), "ibt_lk_fb")
    r = {k: v.cpu().numpy() for k, v in o.items()}
    r["iter_total"] = int(tot.item())
    return r


def _all_intact(pyrs):
    return all(b.intact() for ch in pyrs for (_, bufs) in ch for b in bufs)


@pytest.mark.parametrize("win", LK_WINDOWS)
def test_lk_layout_invariance(ibt, oracle, lk_scene, win):
    """ibt_lk, ibt_lk_fb and ibt_lk_multichannel on the same pyramids in five layouts: canonical (TMA image + Scharr), TMA
    image only, TMA Scharr only, byte gather (image at offset 1), and a per-level mix -- identical outputs, and the canonical
    ones against the oracle."""
    S = lk_scene
    pts, guess = torch.from_numpy(S["pts"]).cuda(), torch.from_numpy(S["guess"]).cuda()
    for maxLevel in (0, 3):
        ml, _ = oracle.pyramid_sizes(LK_H, LK_W, win, maxLevel)
        nlev = ml + 1
        res = {}
        for name in LK_LAYOUTS:
            pyrs = _placed_pyramids(S, name, nlev, LK_CN)
            r = {}
            for flags in (0, INIT, MINEIG):
                r["lk", flags] = _run_lk(pyrs, pts, guess, win, flags)
            r["fb"] = _run_lk_fb(pyrs, pts, win)
            for cn in (2, 4):
                r["mc%d" % cn] = _run_lk(pyrs, pts, guess, win, 0, cn)
            r["mc2", INIT] = _run_lk(pyrs, pts, guess, win, INIT, 2)
            assert _all_intact(pyrs), (win, maxLevel, name)
            res[name] = r
        canon = res["canon"]
        for name, r in res.items():
            for key, out in r.items():
                if key == "fb":
                    assert out["iter_total"] == canon[key]["iter_total"] == int(canon[key]["iters"].sum())
                    out = {k: v for k, v in out.items() if k != "iter_total"}
                for k, v in out.items():
                    ref = canon[key][k]
                    assert _same(v, ref), (win, maxLevel, name, key, k, int((v != ref).sum()))
        # (b) the oracle, on the canonical outputs
        lv = [S["planes"][c] for c in range(LK_CN)]
        crit = dict(winSize=win, maxLevel=maxLevel, criteria=(3, 30, 0.01))
        for flags in (0, INIT, MINEIG):
            po, so, eo, io = oracle.calcOpticalFlowPyrLK(lv[0][0], lv[0][1], S["pts"], S["guess"], flags=flags, return_iters=True,
                                                        **crit)
            assert_lk_exact(canon["lk", flags], dict(p1=po, st=so, err=eo, iters=io), "%s ml %d flags %d" % (win, maxLevel, flags),
                            S["pts"], S["guess"] if flags & INIT else None)
        fb = canon["fb"]
        assert _same(fb["p1"], canon["lk", 0]["p1"]) and _same(fb["st1"], canon["lk", 0]["st"])
        stack = lambda k: np.stack([lv[c][k] for c in range(2)], -1)
        po, so, eo, io = oracle.calcOpticalFlowPyrLK(stack(0), stack(1), S["pts"], None, return_iters=True, **crit)
        assert_lk_exact(canon["mc2"], dict(p1=po, st=so, err=eo, iters=io), "%s ml %d cn 2" % (win, maxLevel), S["pts"])
        st = canon["lk", 0]["st"]
        assert 0 < st.sum() < len(st), (win, maxLevel)          # both outcomes occur: the border cases are exercised


# ---- the persistent LK launch --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lk_frames(ibt):
    from iceberg_tracking_code_b200 import synthetic as syn
    h, w = 720, 1150
    base = syn.base_texture(h, w, 3)
    f0, f1 = syn.frame_gray(base, 0).cuda(), syn.frame_gray(base, 1).cuda()
    rng = np.random.default_rng(4)
    pts = np.concatenate([rng.uniform([20, 20], [w - 20, h - 20], (4800, 2)), rng.uniform([-30, -30], [w + 30, h + 30], (200, 2))])
    return f0, f1, torch.from_numpy(pts.astype(np.float32)).cuda()


@pytest.mark.parametrize("win", [(21, 21), (9, 15)])
def test_lk_launch_independent_of_grid_and_history(ibt, lk_frames, win):
    f0, f1, pts = lk_frames
    pa, pb = ibt.FramePyramid(f0, win, 3, True), ibt.FramePyramid(f1, win, 3, True)
    one = [[(pa.c, []), (pb.c, [])]]
    ref = _run_lk(one, pts, None, win, 0)
    # occupancy cap (process-wide: restored whatever happens)
    try:
        for ctas in (1, 2, 0):
            _ok(_lib().ibt_lk_set_max_ctas_per_sm(ctas), "ibt_lk_set_max_ctas_per_sm")
            r = _run_lk(one, pts, None, win, 0)
            for k in ref:
                assert _same(r[k], ref[k]), (win, ctas, k)
    finally:
        _lib().ibt_lk_set_max_ctas_per_sm(0)
    # back-to-back launches on one stream, nothing read back in between: the work queue re-arms itself
    def launch(n, s, o):
        _ok(_lib().ibt_lk(C.byref(pa.c), C.byref(pb.c), _p(pts), _p(o["p1"]), n, win[0], win[1], 30, 0.01, 1e-4, 0,
                          _p(o["st"]), _p(o["err"]), _p(o["iters"]), _stream(s)), "ibt_lk")
    torch.cuda.synchronize()
    cur = torch.cuda.current_stream()
    s2 = torch.cuda.Stream()
    plan = [(n, cur) for n in (1, 7, 5000, 1)] + [(n, s) for n in (3000, 5000, 1, 7) for s in (cur, s2)]
    outs = [_lk_outputs(n, False) for n, _ in plan]
    torch.cuda.synchronize()
    for (n, s), o in zip(plan, outs):
        launch(n, s, o)
    torch.cuda.synchronize()
    for i, ((n, s), o) in enumerate(zip(plan, outs)):
        for k in ref:
            assert _same(o[k].cpu().numpy(), ref[k][:n]), (win, i, n, k)


def test_lk_fb_alive_null_buffers_and_iter_total(ibt, lk_frames):
    f0, f1, pts = lk_frames
    win = (21, 21)
    pa, pb = ibt.FramePyramid(f0, win, 3, True), ibt.FramePyramid(f1, win, 3, True)
    one = [[(pa.c, []), (pb.c, [])]]
    full = _run_lk_fb(one, pts, win)
    assert full["iter_total"] == int(full["iters"].astype(np.int64).sum())
    n = pts.shape[0]
    # alive partly 0: dead points are skipped and their outputs left as they were
    alive0 = (np.random.default_rng(9).random(n) < 0.6).astype(np.uint8)
    o = _lk_outputs(n, True)
    o["alive"].copy_(torch.from_numpy(alive0))
    before = {k: v.cpu().numpy() for k, v in o.items()}
    tot = torch.zeros(1, dtype=torch.int64, device="cuda")
    _ok(_lib().ibt_lk_fb(C.byref(pa.c), C.byref(pb.c), _p(pts), n, 21, 21, 30, 0.01, 1e-4, 1.0, _p(o["p1"]), _p(o["st1"]),
                         _p(o["err1"]), _p(o["p0r"]), _p(o["st0"]), _p(o["err0"]), _p(o["fbdist"]), _p(o["alive"]),
                         _p(o["iters"]), _p(tot), _stream()), "ibt_lk_fb")
    got = {k: v.cpu().numpy() for k, v in o.items()}
    live = alive0 == 1
    for k, v in got.items():
        if k == "alive":
            assert np.array_equal(v[~live], before[k][~live])
            assert np.array_equal(v[live], full[k][live])
        else:
            assert _same(v[~live], before[k][~live]), k
            assert _same(v[live], full[k][live]), k
    assert int(tot.item()) == int(full["iters"][live].astype(np.int64).sum())
    # NULL for any subset of st1 / err1 / st0 / err0: p1, p0r and fbdist do not change
    fresh = {k: v.cpu().numpy() for k, v in _lk_outputs(n, True).items()}
    for mask in range(16):
        o = _lk_outputs(n, True)
        nul = lambda k, bit: None if (mask >> bit) & 1 else _p(o[k])
        _ok(_lib().ibt_lk_fb(C.byref(pa.c), C.byref(pb.c), _p(pts), n, 21, 21, 30, 0.01, 1e-4, 1.0, _p(o["p1"]), nul("st1", 0),
                             nul("err1", 1), _p(o["p0r"]), nul("st0", 2), nul("err0", 3), _p(o["fbdist"]), _p(o["alive"]),
                             None, None, _stream()), "ibt_lk_fb")
        for k in ("p1", "p0r", "fbdist", "alive"):
            assert _same(o[k].cpu().numpy(), full[k]), (mask, k)
        for bit, k in enumerate(("st1", "err1", "st0", "err0")):
            assert _same(o[k].cpu().numpy(), fresh[k] if (mask >> bit) & 1 else full[k]), (mask, k)


# ---- GFTT --------------------------------------------------------------------------------------------------------------
GFTT_H, GFTT_W = 300, 457


@pytest.fixture(scope="module")
def gftt_scene(ibt):
    from iceberg_tracking_code_b200 import synthetic as syn
    img = syn.frame_gray(syn.base_texture(GFTT_H, GFTT_W, 8), 0).numpy()
    mask = np.zeros_like(img)
    mask[20:280, 30:400] = 1
    mask[100:150, 200:260] = 0
    return img, mask


def _gftt(img_pl, mask_pl, bs, harris, use_async=False):
    H, W = GFTT_H, GFTT_W
    nb = _lib().ibt_gftt_workspace_bytes(H, W)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    cap = H * W // 4
    out = torch.full((cap, 2), -1.0, dtype=torch.float32, device="cuda")
    args = (img_pl.ptr, img_pl.pitch, mask_pl.ptr if mask_pl else None, mask_pl.pitch if mask_pl else 0, H, W, 0, 0.01, 5.0,
            bs, harris, 0.04, _p(ws), nb, _p(out), cap)
    if use_async:
        cnt = torch.full((1,), -1, dtype=torch.int32, device="cuda")
        _ok(_lib().ibt_gftt_async(*args, _p(cnt), _stream()), "ibt_gftt_async")
        n = int(cnt.item())
    else:
        c = C.c_int(0)
        _ok(_lib().ibt_gftt(*args, C.byref(c), _stream()), "ibt_gftt")
        n = c.value
    return out[:n].cpu().numpy()


def test_gftt_any_layout(ibt, oracle, gftt_scene):
    """Pitches W, W+1, W+3, round_up(W, 128) at base offsets 0..3 (word loads only where both are 4-byte aligned; every
    strip takes the border path otherwise); a mask with its own pitch and offset; blockSize 3 and 10 (compiled in) and 5."""
    img, mask = gftt_scene
    H, W = img.shape
    canon_img = Placed(img.shape, torch.uint8, 0, W, img)
    canon_mask = Placed(img.shape, torch.uint8, 0, W, mask)
    for bs in (3, 10, 5):
        for harris in (0, 1):
            for m in (False, True):
                ref = _gftt(canon_img, canon_mask if m else None, bs, harris)
                assert len(ref) > 100
                orc = as_corners(oracle.goodFeaturesToTrack(img, 0, 0.01, 5.0, mask=mask if m else None, blockSize=bs,
                                                            useHarrisDetector=bool(harris)))
                assert corner_overlap(ref, orc) >= CORNER_OVERLAP, (bs, harris, m)
                for off in range(4):
                    for pitch in (W, W + 1, W + 3, _ru(W, 128)):
                        ip = Placed(img.shape, torch.uint8, off, pitch, img)
                        mp = Placed(img.shape, torch.uint8, (off + 1) % 4, W + 7 + off, mask) if m else None
                        for use_async in ((False, True) if off in (0, 1) and pitch == W + 3 else (False,)):
                            got = _gftt(ip, mp, bs, harris, use_async)
                            assert _same(got, ref), (bs, harris, m, off, pitch, use_async, len(got), len(ref))
                        assert ip.intact() and (mp is None or mp.intact())
    # the padded level 0 of a FramePyramid with a contiguous mask: SequenceTracker.gftt_prefetch's call
    ip = Placed(img.shape, torch.uint8, 0, _ru(W, 128), img)
    assert _same(_gftt(ip, canon_mask, 10, 0, True), _gftt(canon_img, canon_mask, 10, 0))


def test_eig_maps_any_layout(ibt, gftt_scene):
    img, _ = gftt_scene
    H, W = img.shape
    for fn in ("ibt_min_eigen_f32", "ibt_corner_harris_f32"):
        for bs in (3, 5, 10, 31):
            ref = None
            for off, pitch, eoff, epitch in ((0, W, 0, 4 * W), (1, W + 3, 4, 4 * W + 4), (3, _ru(W, 128), 0, 4 * W + 4),
                                             (2, W + 1, 16, _ru(4 * W, 128))):
                ip = Placed(img.shape, torch.uint8, off, pitch, img)
                ep = Placed(img.shape, torch.float32, eoff, epitch)
                extra = (0.04,) if fn == "ibt_corner_harris_f32" else ()
                _ok(getattr(_lib(), fn)(ip.ptr, H, W, pitch, bs, *extra, ep.ptr, epitch, _stream()), fn)
                got = ep.np()
                if ref is None:
                    ref = got
                assert _same(got, ref), (fn, bs, off, pitch, epitch)
                assert ip.intact() and ep.intact(), (fn, bs, off, pitch, epitch)


# ---- ibt_polygon_mask ----------------------------------------------------------------------------------------------------
def test_polygon_mask_any_layout(ibt):
    H, W = 97, 301
    poly = torch.tensor([[10.5, 3.0], [290.0, 20.25], [250.0, 90.0], [150.0, 40.0], [12.0, 80.0]], dtype=torch.float64,
                        device="cuda")
    ref = None
    for off, pitch in ((0, W), (1, W + 6), (3, _ru(W, 128) + 1), (16, W + 16)):
        out = Placed((H, W), torch.uint8, off, pitch)
        _ok(_lib().ibt_polygon_mask(_p(poly), 5, H, W, out.ptr, pitch, 7, _stream()), "ibt_polygon_mask")
        got = out.np()
        ref = got if ref is None else ref
        assert np.array_equal(got, ref) and set(np.unique(got)) == {0, 7}, (off, pitch)
        assert out.intact(), (off, pitch)


# ---- INTEGRATION.md, Level 3: contiguous caller-allocated buffers --------------------------------------------------------
@pytest.mark.parametrize("hw", [(720, 1150), (3600, 5750)])
def test_integration_level3_recipe(ibt, hw):
    """ibt_gray_u8 -> ibt_pyramid_build -> ibt_lk_fb on plain contiguous tensors per level (level 1 of 1150 / 5750 is odd:
    no tensor maps, byte gathers, the pyramid's unaligned source path) == the same frames through FramePyramid /
    calcOpticalFlowPyrLK_FB."""
    from iceberg_tracking_code_b200 import synthetic as syn
    H, W = hw
    win, maxLevel = (35, 35), 4
    base = syn.base_texture(H, W, 17, device="cuda")
    rgb = [syn.frame_rgb(base, t) for t in (0, 1)]
    rng = np.random.default_rng(H)
    n = 20000 if H > 1000 else 5000
    p0 = torch.from_numpy(np.concatenate([rng.uniform([0, 0], [W, H], (n - 200, 2)),
                                          rng.uniform([-20, -20], [W + 20, H + 20], (200, 2))]).astype(np.float32)).cuda()
    lib, s = _lib(), _stream()
    sizes = (C.c_int * 16)()
    ml = lib.ibt_pyramid_levels(H, W, win[0], win[1], maxLevel, sizes)
    assert ml == maxLevel
    pyr = []
    keep = []
    for f in rgb:
        gray = torch.empty((H, W), dtype=torch.uint8, device="cuda")
        _ok(lib.ibt_gray_u8(f.data_ptr(), H, W, 3, 3 * W, gray.data_ptr(), W, 0, s), "ibt_gray_u8")
        st = _N().ibt_pyramid_t()
        st.nlevels = ml + 1
        for l in range(ml + 1):
            h, w = sizes[2 * l], sizes[2 * l + 1]
            img = gray if l == 0 else torch.empty((h, w), dtype=torch.uint8, device="cuda")
            der = torch.empty((h, w, 2), dtype=torch.int16, device="cuda")
            keep += [img, der]
            st.rows[l], st.cols[l] = h, w
            st.img[l], st.img_pitch[l] = img.data_ptr(), w
            st.deriv[l], st.deriv_pitch[l] = der.data_ptr(), 4 * w
        _ok(lib.ibt_pyramid_build(C.byref(st), 1, s), "ibt_pyramid_build")
        pyr.append(st)
    assert sizes[3] % 2 == 1                                             # level 1 is odd: no level gets a tensor map
    p1 = torch.empty((n, 2), dtype=torch.float32, device="cuda")
    fbdist = torch.empty(n, dtype=torch.float32, device="cuda")
    alive = torch.ones(n, dtype=torch.uint8, device="cuda")
    _ok(lib.ibt_lk_fb(C.byref(pyr[0]), C.byref(pyr[1]), p0.data_ptr(), n, 35, 35, 25, 0.03, 1e-4, 1.0, p1.data_ptr(), None,
                      None, None, None, None, fbdist.data_ptr(), alive.data_ptr(), None, None, s), "ibt_lk_fb")
    fp = [ibt.FramePyramid(ibt.cvtColor(f), win, maxLevel, True) for f in rgb]
    r = ibt.calcOpticalFlowPyrLK_FB(fp[0], fp[1], p0, winSize=win, maxLevel=maxLevel, criteria=(3, 25, 0.03))
    assert torch.equal(p1, r["p1"]) and torch.equal(fbdist, r["dist"]) and torch.equal(alive.bool(), r["valid"])
    assert float(r["valid"].float().mean()) > 0.5


# ---- worst-case magnitudes: the int32 headroom of the exact window sums -----------------------------------------------------
# Per lane, LK keeps its window sums as exact int32 and flushes them to int64 (warp_sum_wide):
#   template (build_template*): one lane owns one window column over up to 63 rows; Iw <= 255 * 32 = 8160, |Ix| <= 16 * 255 = 4080,
#     so |c1| = |sum Iw * Ix| <= 63 * 8160 * 4080 = 2 097 446 400 = 97.7 % of 2^31 - 1.  A vertical 0 -> 255 step edge under a
#     63-row window, sampled at an integer position, reaches exactly that.
#   Newton (newton_sums): a lane owns 4 adjacent columns and flushes every 16 rows.  The loose bound 64 * 8160 * 4080 is above
#     2^31; what a scene can reach is about half of it, because positive Ix over four adjacent columns telescopes to at most
#     2 * 255 * 16 = 8160 per row: 16 * 8160 * 8160 = 1 065 369 600.
# The cases below must reach >= 95 % of 2^31 - 1 in the template (asserted from a numpy restatement); a change to the lane mapping
# or to the flush interval that overflows shows up as wrong positions / eigenvalues here.
HR_WINDOWS = [(63, 63), (61, 63), (33, 63), (35, 35)]
HR_EDGE = 100                            # first bright column


def _headroom_scene():
    h, w = 200, 220
    I = np.zeros((h, w), np.uint8)
    I[:, HR_EDGE:] = 255
    I[90:100, HR_EDGE + 12:HR_EDGE + 30] = 0                        # dark bar away from the edge: a well-conditioned tensor
    # J = I shifted by (0.25, 0.375) px (bilinear, rounded)
    ax, ay = 0.25, 0.375
    If = np.pad(I.astype(np.float64), ((1, 0), (1, 0)), mode="edge")
    J = ((1 - ax) * (1 - ay) * If[1:, 1:] + ax * (1 - ay) * If[1:, :-1] + (1 - ax) * ay * If[:-1, 1:] + ax * ay * If[:-1, :-1])
    return I, np.clip(np.rint(J), 0, 255).astype(np.uint8)


def _hr_points(win):
    xs = [HR_EDGE + win[0] // 2 - k for k in (0, 5, 12)]
    return np.array([(x + fx, 95 + fy) for x in xs for fx in (0.0, 0.5) for fy in (0.0, 0.5)], np.float32)


def _structure_restated(I, D, pt, win):
    """OpenCV's fixed point at level 0 (14-bit bilinear weights, Iw with 5 fractional bits): per-column partials of
    c1 = sum Iw * Ix, and (A11, A12, A22) as int64."""
    f32 = np.float32
    ppx, ppy = f32(pt[0]) - f32((win[0] - 1) * 0.5), f32(pt[1]) - f32((win[1] - 1) * 0.5)
    ix, iy = int(np.floor(ppx)), int(np.floor(ppy))
    a, b = f32(ppx - f32(ix)), f32(ppy - f32(iy))
    iw00 = int(np.rint(f32(f32(f32(1) - a) * f32(f32(1) - b)) * f32(16384)))
    iw01 = int(np.rint(f32(a * f32(f32(1) - b)) * f32(16384)))
    iw10 = int(np.rint(f32(f32(f32(1) - a) * b) * f32(16384)))
    iw11 = 16384 - iw00 - iw01 - iw10
    ys, xs = slice(iy, iy + win[1]), slice(ix, ix + win[0])
    ys1, xs1 = slice(iy + 1, iy + win[1] + 1), slice(ix + 1, ix + win[0] + 1)
    bil = lambda P: (P[ys, xs] * iw00 + P[ys, xs1] * iw01 + P[ys1, xs] * iw10 + P[ys1, xs1] * iw11)
    I, D = I.astype(np.int64), D.astype(np.int64)
    Iw = (bil(I) + 256) >> 9
    Ix = (bil(D[..., 0]) + 8192) >> 14
    Iy = (bil(D[..., 1]) + 8192) >> 14
    return (Iw * Ix).sum(0), (Ix * Ix).sum(), (Ix * Iy).sum(), (Iy * Iy).sum()


def test_lk_int32_headroom(ibt, oracle):
    I, J = _headroom_scene()
    D = oracle.scharr_deriv(I)
    peak = 0
    for win in HR_WINDOWS:
        pts = _hr_points(win)
        for pt in pts:
            c1cols, _, _, _ = _structure_restated(I, D, pt, win)
            peak = max(peak, int(np.abs(c1cols).max()))
    assert peak == 63 * 8160 * 4080 and peak >= 0.95 * I32_MAX, peak
    try:
        import cv2
    except ImportError:
        cv2 = None
    for win in HR_WINDOWS:
        pts = _hr_points(win)
        for maxLevel in (0, 2):
            lp = dict(winSize=win, maxLevel=maxLevel, criteria=(3, 30, 0.01))
            p1, st, err, it = ibt.calcOpticalFlowPyrLK(I, J, pts, None, return_iters=True, **lp)
            po, so, eo, io = oracle.calcOpticalFlowPyrLK(I, J, pts, None, return_iters=True, **lp)
            assert_lk_exact(dict(p1=p1, st=st, err=err, iters=it), dict(p1=po, st=so, err=eo, iters=io),
                            "headroom %s ml %d" % (win, maxLevel), pts)
            assert st.all(), (win, maxLevel)
            if cv2 is not None:
                pc, sc, _ = cv2.calcOpticalFlowPyrLK(I, J, pts.reshape(-1, 1, 2), None, **lp)
                assert_lk_parity(p1, st, pc, sc, "headroom vs cv2 %s ml %d" % (win, maxLevel))
            # the same scene as 4 identical channel planes
            I4, J4 = np.repeat(I[..., None], 4, -1), np.repeat(J[..., None], 4, -1)
            q1, qs, qe, qi = ibt.calcOpticalFlowPyrLK(I4, J4, pts, None, return_iters=True, **lp)
            qo, qso, qeo, qio = oracle.calcOpticalFlowPyrLK(I4, J4, pts, None, return_iters=True, **lp)
            assert_lk_exact(dict(p1=q1, st=qs, err=qe, iters=qi), dict(p1=qo, st=qso, err=qeo, iters=qio),
                            "headroom 4 channels %s ml %d" % (win, maxLevel), pts)
        # min eigenvalue at level 0: err with GET_MIN_EIGENVALS, against the int64 restatement
        _, _, err = ibt.calcOpticalFlowPyrLK(I, J, pts, None, winSize=win, maxLevel=0, flags=MINEIG)
        for k, pt in enumerate(pts):
            _, a11, a12, a22 = _structure_restated(I, D, pt, win)
            A11, A12, A22 = a11 / 2.0 ** 20, a12 / 2.0 ** 20, a22 / 2.0 ** 20
            lam = (A11 + A22 - np.sqrt((A11 - A22) ** 2 + 4 * A12 * A12)) / (2 * win[0] * win[1])
            assert lam > 0 and abs(float(err[k, 0]) - lam) <= 1e-6 * lam, (win, pt, float(err[k, 0]), lam)


def test_gftt_saturated_scenes(ibt, oracle):
    """blockSize 31 on 0/255 checkerboards and step edges: the largest products and box sums the Sobel stage can produce.
    Periodic checkerboards have plateaus of exactly equal responses whose raw 3x3 maxima outnumber the workspace's candidate
    capacity (H*W/4 + 4096): ibt_gftt reports IBT_E_CAPACITY there (include/ibt.h)."""
    yy, xx = np.mgrid[0:160, 0:203]
    scenes = [((yy // 8 + xx // 8) % 2 * 255).astype(np.uint8), ((yy // 13 + xx // 5) % 2 * 255).astype(np.uint8),
              np.where(xx >= 101, 255, 0).astype(np.uint8), np.where((xx >= 90) & (yy >= 70), 255, 0).astype(np.uint8)]
    H, W = yy.shape
    for i, img in enumerate(scenes):
        e, eo = ibt.cornerMinEigenVal(img, 31), oracle.cornerMinEigenVal(img, 31)
        assert np.abs(e - eo).max() <= 2e-4 * np.abs(eo).max(), i
        pad = np.pad(eo, 1, constant_values=-np.inf)
        raw = (eo == np.max([pad[dy:dy + H, dx:dx + W] for dy in range(3) for dx in range(3)], 0)) & (eo > 0.01 * eo.max())
        nraw = int(raw[1:-1, 1:-1].sum())
        if nraw > H * W // 4 + 4096:
            with pytest.raises(ibt.N.IbtError) as ex:
                ibt.goodFeaturesToTrack(img, 0, 0.01, 3, blockSize=31)
            assert ex.value.code == ibt.N.IBT_E_CAPACITY, i
            continue
        got = as_corners(ibt.goodFeaturesToTrack(img, 0, 0.01, 3, blockSize=31))
        ref = as_corners(oracle.goodFeaturesToTrack(img, 0, 0.01, 3, blockSize=31))
        assert corner_overlap(got, ref) >= CORNER_OVERLAP, (i, len(got), len(ref))
        assert (len(ref) > 0) == (i != 2), (i, len(ref))              # a straight edge has no corner (rank-1 tensor)
