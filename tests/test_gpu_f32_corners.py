"""cornerMinEigenVal / cornerHarris / goodFeaturesToTrack on float32 images on the GPU: against cv2's answers (golden file and
a live fuzz), the CPU reference of tests/f32_cases.py at 1080p and 24 MP, exact scale invariance, the u8 path on
integer-valued images, other memory layouts, non-finite pixels and repeatability."""
import ctypes as C

import numpy as np
import pytest
import torch

import f32_cases as FC
from parity import as_corners

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scenes(golden):
    return {name: golden("kat_%s.npz" % name) for name in ("texture", "iceberg")}


def _frame(h, w, seed):
    from iceberg_tracking_code_b200 import synthetic as syn
    base = syn.base_texture(h, w, seed, device="cuda")
    return syn.frame_gray(base, 0).cpu().numpy()


def _gamma(u8):
    return np.power(u8.astype(np.float32) / np.float32(255.0), np.float32(1.8)).astype(np.float32)


def test_cuda_golden(ibt, golden, scenes):
    FC.check_f32_golden(ibt, golden("kat_f32.npz"), scenes)


def test_cuda_live_cv2(ibt, oracle):
    """sizes 3x3 .. 240x321, windows wider than the image, every aperture, both responses, masks, value ranges from 1e-3 to
    1e4 with offsets of either sign: maps within the bound, lists by FC.check_lists on cv2's own map"""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(2024)
    sizes = [(3, 3), (3, 11), (9, 4), (17, 29), (64, 70), (131, 97), (240, 321)]
    for i, (h, w) in enumerate(sizes):
        a = rng.random((h + 2, w + 2))
        a = (a[1:, 1:] + a[:-1, :-1])[:h, :w] + (np.kron(rng.random((h // 4 + 2, w // 4 + 2)) > 0.5, np.ones((4, 4)))[:h, :w])
        lo, span = [(0.0, 1.0), (-3.5, 0.02), (1e4, 250.0), (-2e-3, 1e-3)][i % 4]
        img = (lo + span * a).astype(np.float32)
        mask = (rng.random((h, w)) > 0.2).astype(np.uint8) * 255
        for ks in FC.APERTURES:
            for bs in sorted({2, 3, min(min(h, w) + 2, 31), int(rng.integers(4, 32))}):   # (blockSize <= 31)
                what = (h, w, ks, bs)
                cm = cv2.cornerMinEigenVal(img, bs, ksize=ks)
                ch = cv2.cornerHarris(img, bs, ks, 0.04)
                FC.check_map(ibt.cornerMinEigenVal(img, bs, ksize=ks), cm, img, bs, ks, False, what)
                FC.check_map(ibt.cornerHarris(img, bs, ks, 0.04), ch, img, bs, ks, True, what)
                if h < 3 or w < 3:
                    continue
                for harris, cmap in ((False, cm), (True, ch)):
                    for m in (None, mask):
                        gp = dict(maxCorners=int(rng.integers(0, 300)), qualityLevel=0.01,
                                  minDistance=float(rng.integers(0, 9)), blockSize=bs)
                        want = cv2.goodFeaturesToTrack(img, mask=m, useHarrisDetector=harris, gradientSize=ks, **gp)
                        got = ibt.goodFeaturesToTrack(img, mask=m, useHarrisDetector=harris, gradientSize=ks, **gp)
                        FC.check_lists(got, want, harris, what + (harris, m is not None), cmap, oracle, m, gp)


def test_cuda_vs_reference_1080p(ibt, oracle):
    """every aperture, blockSize 3 / 10 / 31, both responses, with and without a mask: maps within the bound, lists by the
    rule on the reference's map"""
    img = _gamma(_frame(1080, 1920, 3))
    mask = np.zeros(img.shape, np.uint8); mask[100:1000, 150:1800] = 255
    for ks in FC.APERTURES:
        for bs in (3, 10, 31):
            for harris in (False, True):
                r = FC.corner_response(img, bs, ks, harris)
                g = ibt.cornerHarris(img, bs, ks, 0.04) if harris else ibt.cornerMinEigenVal(img, bs, ksize=ks)
                FC.check_map(g, r, img, bs, ks, harris, (ks, bs, harris))
                for m in (None, mask):
                    gp = dict(maxCorners=0, qualityLevel=0.007, minDistance=10, blockSize=bs)
                    sel = oracle.gftt_select(r, m, 0, 0.007, 10)
                    got = ibt.goodFeaturesToTrack(img, mask=m, useHarrisDetector=harris, gradientSize=ks, **gp)
                    FC.check_lists(got, sel, harris, (ks, bs, harris, m is not None), r, oracle, m, gp)


@pytest.mark.parametrize("ks", [-1, 3, 7])
def test_cuda_vs_reference_24mp(ibt, oracle, ks):
    """the ordered top-20 k corner list of a 24 MP float frame (config-2 parameters)"""
    img = _gamma(_frame(4000, 6000, 7))
    gp = dict(maxCorners=20000, qualityLevel=0.007, minDistance=10, blockSize=10, gradientSize=ks)
    got = ibt.goodFeaturesToTrack(img, **gp)
    r = FC.corner_response(img, 10, ks)
    ref = oracle.gftt_select(r, None, 20000, 0.007, 10)
    assert as_corners(ref).shape[0] == 20000
    FC.check_lists(got, ref, False, ks, r, oracle, None, dict(gp))


def test_scale_invariance(ibt):
    """I * 2^j scales the min-eig map by exactly 4^j and the Harris map by 16^j, and leaves every corner list identical"""
    img = _gamma(_frame(300, 500, 11))
    mask = np.zeros(img.shape, np.uint8); mask[20:280, 30:470] = 255
    for ks in FC.APERTURES:
        for bs in (3, 10):
            m0 = ibt.cornerMinEigenVal(img, bs, ksize=ks)
            h0 = ibt.cornerHarris(img, bs, ks, 0.04)
            for harris in (False, True):
                base = ibt.goodFeaturesToTrack(img, 0, 0.01, 5, mask=mask, blockSize=bs, useHarrisDetector=harris, gradientSize=ks)
                for j in (-6, 3, 10):
                    s = np.float32(2.0 ** j)
                    assert np.array_equal(ibt.cornerMinEigenVal(img * s, bs, ksize=ks), m0 * np.float32(4.0 ** j)), (ks, bs, j)
                    assert np.array_equal(ibt.cornerHarris(img * s, bs, ks, 0.04), h0 * np.float32(16.0 ** j)), (ks, bs, j)
                    got = ibt.goodFeaturesToTrack(img * s, 0, 0.01, 5, mask=mask, blockSize=bs, useHarrisDetector=harris,
                                                  gradientSize=ks)
                    assert np.array_equal(as_corners(got), as_corners(base)) and len(as_corners(base)) > 50, (ks, bs, j, harris)


def test_integer_valued_image_gives_the_u8_corners(ibt):
    """a float image holding the u8 frame's values: the same corners as the u8 path (the maps differ by the factor 255^2 of
    the u8 scale and by rounding)"""
    u8 = _frame(480, 640, 5)
    f = u8.astype(np.float32)
    for ks in FC.APERTURES:
        for bs in (3, 10):
            for harris in (False, True):
                gp = dict(maxCorners=500, qualityLevel=0.01, minDistance=10, blockSize=bs, useHarrisDetector=harris,
                          gradientSize=ks)
                FC.check_lists(ibt.goodFeaturesToTrack(f, **gp), ibt.goodFeaturesToTrack(u8, **gp), harris, (ks, bs, harris))


def _sentinel(shape_bytes, fill):
    return torch.full((shape_bytes,), fill, dtype=torch.uint8, device="cuda")


def test_layouts():
    """images at 4-byte (not 16-byte) offsets and odd pitches, masks at odd offsets, maps written at an offset and pitch into
    sentinel buffers: the contiguous layout's bytes, and no byte outside the output rows changed"""
    from iceberg_tracking_code_b200 import build, _native as N
    build.build()
    lib = N.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    img = _gamma(_frame(300, 700, 13))
    H, W = img.shape
    t = torch.from_numpy(img).cuda()
    m = torch.zeros((H, W), dtype=torch.uint8, device="cuda"); m[20:280, 30:650] = 255
    pitch = W * 4 + 12                                            # bytes: a multiple of 4, not of 16
    ibuf = _sentinel(4 + H * pitch, 0)
    ibuf[4:].view(H, pitch)[:, :W * 4].copy_(t.view(torch.uint8).view(H, W * 4))
    img_odd = ibuf.data_ptr() + 4
    mbuf = _sentinel(1 + H * (W + 5), 0)
    mbuf[1:].view(H, W + 5)[:, :W].copy_(m)

    def gftt(ptr, p, mptr, mp, bs, ks, harris):
        nbytes = lib.ibt_gftt_workspace_bytes(H, W)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device="cuda")
        out = torch.zeros((H * W // 4 + 4096, 2), dtype=torch.float32, device="cuda")
        cnt = C.c_int(0)
        N.check(lib.ibt_gftt_f32src(C.c_void_p(ptr), p, C.c_void_p(mptr), mp, H, W, 0, 0.01, 5.0, bs, ks, harris, 0.04,
                                    C.c_void_p(ws.data_ptr()), nbytes, C.c_void_p(out.data_ptr()), out.shape[0], C.byref(cnt),
                                    st), "ibt_gftt_f32src")
        return out[:cnt.value].cpu().numpy()

    def maps(ptr, p, bs, ks, harris, out_off, out_pitch):
        buf = _sentinel(out_off + (H + 2) * out_pitch, 0xA5)
        dst = buf.data_ptr() + out_off + out_pitch                # one sentinel row above, one below
        if harris:
            N.check(lib.ibt_corner_harris_f32src(C.c_void_p(ptr), H, W, p, bs, ks, 0.04, C.c_void_p(dst), out_pitch, st), "h")
        else:
            N.check(lib.ibt_min_eigen_f32src(C.c_void_p(ptr), H, W, p, bs, ks, C.c_void_p(dst), out_pitch, st), "m")
        b = buf.cpu().numpy()
        rows = b[out_off + out_pitch:out_off + (H + 1) * out_pitch].reshape(H, out_pitch)
        outside = np.concatenate([b[:out_off + out_pitch], b[out_off + (H + 1) * out_pitch:], rows[:, W * 4:].ravel()])
        assert np.all(outside == 0xA5), (bs, ks, harris)
        return rows[:, :W * 4].copy()

    for ks in FC.APERTURES:
        for bs in (3, 10, 31):
            for harris in (0, 1):
                a = gftt(t.data_ptr(), W * 4, m.data_ptr(), W, bs, ks, harris)
                b = gftt(img_odd, pitch, mbuf.data_ptr() + 1, W + 5, bs, ks, harris)
                assert a.tobytes() == b.tobytes() and len(a) > 50, (ks, bs, harris)
                assert maps(t.data_ptr(), W * 4, bs, ks, harris, 0, W * 4).tobytes() == \
                    maps(img_odd, pitch, bs, ks, harris, 8, W * 4 + 20).tobytes(), (ks, bs, harris)


def test_non_finite_and_repeatable(ibt):
    """a NaN or inf pixel: the maps carry NaN / inf around it (as cv2's do) and goodFeaturesToTrack raises rather than return
    corners derived from it; two calls on a finite image give identical bytes"""
    img = _gamma(_frame(200, 300, 21))
    for bad in (np.nan, np.inf, -np.inf):
        x = img.copy(); x[77, 123] = bad
        for ks in FC.APERTURES:
            mp = ibt.cornerMinEigenVal(x, 5, ksize=ks)
            assert not np.isfinite(mp[77, 123]) and np.isfinite(mp[0, 0]) and np.isfinite(mp[150, 250]), (bad, ks)
            for harris in (False, True):
                with pytest.raises(ibt.error, match="non-finite"):
                    ibt.goodFeaturesToTrack(x, 100, 0.01, 5, blockSize=5, useHarrisDetector=harris, gradientSize=ks)
    # the workspace is reusable after a refusal
    for ks in FC.APERTURES:
        for harris in (False, True):
            gp = dict(maxCorners=0, qualityLevel=0.01, minDistance=5, blockSize=7, useHarrisDetector=harris, gradientSize=ks)
            a = ibt.goodFeaturesToTrack(img, **gp)
            b = ibt.goodFeaturesToTrack(torch.from_numpy(img).cuda(), **gp).cpu().numpy()
            assert a.tobytes() == b.tobytes() and len(a) > 50, (ks, harris)
            assert ibt.cornerHarris(img, 7, ks, 0.04).tobytes() == ibt.cornerHarris(img, 7, ks, 0.04).tobytes()


def test_map_equals_the_list_producer(ibt, oracle):
    """the fused producer and the map hook compute the same bits: goodFeaturesToTrack is exactly the selection on the map,
    tiny images and windows wider than the image included"""
    rng = np.random.default_rng(5)
    for h, w in [(3, 3), (3, 8), (8, 3), (5, 7), (4, 40), (37, 6), (130, 270)]:
        img = (rng.random((h, w)) * 2.0 - 0.5).astype(np.float32)
        mask = (rng.random((h, w)) > 0.3).astype(np.uint8) * 255
        for ks in FC.APERTURES:
            for bs in sorted({2, min(min(h, w) + 1, 31), 31}):
                for harris in (False, True):
                    r = ibt.cornerHarris(img, bs, ks, 0.04) if harris else ibt.cornerMinEigenVal(img, bs, ksize=ks)
                    for m in (None, mask):
                        for mc, q, md in ((0, 0.007, 0), (300, 0.02, 5)):
                            got = ibt.goodFeaturesToTrack(img, mc, q, md, mask=m, blockSize=bs, useHarrisDetector=harris,
                                                          gradientSize=ks)
                            sel = oracle.gftt_select(r, m, mc, q, md)
                            assert np.array_equal(as_corners(got), as_corners(sel)), (h, w, ks, bs, harris, m is not None)
