"""cornerMinEigenVal / cornerHarris / goodFeaturesToTrack with the Sobel apertures other than 3 (ksize / gradientSize = -1
(Scharr), 1, 5, 7) on the GPU: against cv2's answers, the CPU reference of tests/ksize_cases.py, the exact int64 window sums,
other memory layouts, and through the sequence tracker's prefetch path."""
import ctypes as C

import numpy as np
import pytest
import torch

import ksize_cases as KC
from parity import as_corners

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scenes(golden):
    return {name: golden("kat_%s.npz" % name) for name in ("texture", "iceberg")}


def _frame(h, w, seed):
    from iceberg_tracking_code_b200 import synthetic as syn
    base = syn.base_texture(h, w, seed, device="cuda")
    return syn.frame_gray(base, 0).cpu().numpy()


def test_cuda_golden(ibt, golden, scenes):
    KC.check_ksize_golden(ibt, golden("kat_ksize.npz"), scenes)


def test_cuda_vs_reference_1080p(ibt, oracle):
    """every aperture, blockSize 3 / 10 / 31, min-eig and Harris, with and without a mask: maps and corner lists"""
    img = _frame(1080, 1920, 3)
    mask = np.zeros_like(img); mask[100:1000, 150:1800] = 255
    ref = KC.Reference(oracle)
    for ks in KC.OTHER_APERTURES:
        for bs in (3, 10, 31):
            for harris in (False, True):
                r = ref.cornerHarris(img, bs, ks, 0.04) if harris else ref.cornerMinEigenVal(img, bs, ks)
                g = ibt.cornerHarris(img, bs, ks, 0.04) if harris else ibt.cornerMinEigenVal(img, bs, ksize=ks)
                KC.check_map(g, r, (ks, bs, harris))
                for m in (None, mask):
                    gp = dict(maxCorners=0, qualityLevel=0.007, minDistance=10, blockSize=bs, useHarrisDetector=harris,
                              gradientSize=ks)
                    sel = oracle.gftt_select(r, m, 0, 0.007, 10)
                    KC.check_lists(ibt.goodFeaturesToTrack(img, mask=m, **gp), sel, harris, (ks, bs, harris, m is not None))


@pytest.mark.parametrize("ks", [5, 7])
def test_cuda_vs_reference_24mp(ibt, oracle, ks):
    """the whole ordered corner list of a 24 MP frame (config-2 parameters, top 20 k)"""
    img = _frame(4000, 6000, 7)
    gp = dict(maxCorners=20000, qualityLevel=0.007, minDistance=10, blockSize=10, gradientSize=ks)
    got = ibt.goodFeaturesToTrack(img, **gp)
    ref = KC.Reference(oracle).goodFeaturesToTrack(img, **gp)
    assert as_corners(ref).shape[0] == 20000
    KC.check_lists(got, ref, False, ks)


def test_cuda_live_cv2(ibt):
    cv2 = pytest.importorskip("cv2")
    img = _frame(480, 640, 5)
    mask = np.zeros_like(img); mask[40:440, 30:600] = 255
    for ks in KC.OTHER_APERTURES:
        for bs in (3, 10):
            KC.check_map(ibt.cornerMinEigenVal(img, bs, ksize=ks), cv2.cornerMinEigenVal(img, bs, ksize=ks), (ks, bs))
            KC.check_map(ibt.cornerHarris(img, bs, ks, 0.04), cv2.cornerHarris(img, bs, ks, 0.04), (ks, bs))
            for harris in (False, True):
                gp = dict(maxCorners=0, qualityLevel=0.007, minDistance=10, blockSize=bs, useHarrisDetector=harris,
                          gradientSize=ks)
                KC.check_lists(ibt.goodFeaturesToTrack(img, mask=mask, **gp), cv2.goodFeaturesToTrack(img, mask=mask, **gp),
                               harris, (ks, bs, harris))


def _gftt(fn, img_t, pitch, mask_t, mask_pitch, H, W, bs, *ks_harris):
    from iceberg_tracking_code_b200 import _native as N
    lib = N.lib()
    nbytes = lib.ibt_gftt_workspace_bytes(H, W)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device="cuda")
    out = torch.zeros((H * W // 4 + 4096, 2), dtype=torch.float32, device="cuda")
    cnt = C.c_int(0)
    mp = C.c_void_p(mask_t.data_ptr()) if mask_t is not None else None
    rc = getattr(lib, fn)(C.c_void_p(img_t.data_ptr()), pitch, mp, mask_pitch, H, W, 0, 0.01, 5.0, bs, *ks_harris, 0.04,
                          C.c_void_p(ws.data_ptr()), nbytes, C.c_void_p(out.data_ptr()), out.shape[0], C.byref(cnt),
                          C.c_void_p(torch.cuda.current_stream().cuda_stream))
    N.check(rc, fn)
    return out[:cnt.value].cpu().numpy()


def _map(fn, img_t, pitch, H, W, bs, args, out_pitch_f=None):
    from iceberg_tracking_code_b200 import _native as N
    pf = out_pitch_f or W
    out = torch.full((H, pf), -7.0, dtype=torch.float32, device="cuda")
    rc = getattr(N.lib(), fn)(C.c_void_p(img_t.data_ptr()), H, W, pitch, bs, *args, C.c_void_p(out.data_ptr()), pf * 4,
                              C.c_void_p(torch.cuda.current_stream().cuda_stream))
    N.check(rc, fn)
    return out[:, :W].cpu().numpy()


def test_aperture3_is_unchanged(ibt):
    """the aperture-taking entry points route ksize 3 to the aperture-3 kernels: their corner lists and maps equal the plain
    entry points' byte for byte (that aperture 3 computes what it did before rests on the unchanged SASS of those kernels and
    on bench.py --dump-outputs, not on this test)"""
    img = _frame(600, 900, 9)
    H, W = img.shape
    t = torch.from_numpy(img).cuda()
    m = torch.zeros_like(t); m[50:550, 60:850] = 255
    for bs in (3, 10, 7):
        for harris in (0, 1):
            for mask in (None, m):
                a = _gftt("ibt_gftt", t, W, mask, W, H, W, bs, harris)
                b = _gftt("ibt_gftt_ksize", t, W, mask, W, H, W, bs, 3, harris)
                assert a.tobytes() == b.tobytes() and len(a) > 100, (bs, harris)
        assert _map("ibt_min_eigen_f32", t, W, H, W, bs, ()).tobytes() == \
            _map("ibt_min_eigen_ksize_f32", t, W, H, W, bs, (3,)).tobytes()
        assert _map("ibt_corner_harris_f32", t, W, H, W, bs, (0.04,)).tobytes() == \
            _map("ibt_corner_harris_ksize_f32", t, W, H, W, bs, (3, 0.04)).tobytes()


@pytest.mark.parametrize("ks", [5, 7])
def test_layouts(ks):
    """odd byte offsets and pitches of image, mask and map give the contiguous layout's results byte for byte (the contiguous
    image takes the word-load strips, the odd one the byte-gather border strips everywhere)"""
    from iceberg_tracking_code_b200 import build
    build.build()
    img = _frame(300, 700, 13)
    H, W = img.shape
    t = torch.from_numpy(img).cuda()
    m = torch.zeros_like(t); m[20:280, 30:650] = 255
    buf = torch.zeros((H, W + 9), dtype=torch.uint8, device="cuda").view(-1)
    odd = buf[3:3 + H * (W + 9) - 9].as_strided((H, W), (W + 9, 1)); odd.copy_(t)
    mbuf = torch.zeros((H, W + 5), dtype=torch.uint8, device="cuda").view(-1)
    modd = mbuf[1:1 + H * (W + 5) - 5].as_strided((H, W), (W + 5, 1)); modd.copy_(m)
    for bs in (3, 10, 31):
        for harris in (0, 1):
            a = _gftt("ibt_gftt_ksize", t, W, m, W, H, W, bs, ks, harris)
            b = _gftt("ibt_gftt_ksize", odd, W + 9, modd, W + 5, H, W, bs, ks, harris)
            assert a.tobytes() == b.tobytes() and len(a) > 50, (bs, harris)
        for fn, args in (("ibt_min_eigen_ksize_f32", (ks,)), ("ibt_corner_harris_ksize_f32", (ks, 0.04))):
            assert _map(fn, t, W, H, W, bs, args).tobytes() == _map(fn, odd, W + 9, H, W, bs, args, W + 3).tobytes(), fn


def _exact_maps(img, bs, ks, k=0.04):
    """the maps restated from exact int64 window sums, in the CUDA path's float arithmetic"""
    sx, sy = KC.sobel_int(img, ks)
    h, w = img.shape
    a0 = -(bs // 2)
    rows = [KC.r101(np.arange(h) + a0 + i, h) for i in range(bs)]
    cols = [KC.r101(np.arange(w) + a0 + j, w) for j in range(bs)]
    sums = []
    for P in (sx * sx, sx * sy, sy * sy):
        V = sum(P[ri, :] for ri in rows)
        sums.append(sum(V[:, cj] for cj in cols))
    scale = np.float32(1.0 / (KC.TAPS[ks][2] * bs * 255.0))
    s2 = float(scale) * float(scale)
    a, b, c = (np.float32(S.astype(np.float64) * s2) for S in sums)
    tr = a + c
    harris = (a * c - b * b) - np.float32(k) * (tr * tr)
    ah, ch = a * np.float32(0.5), c * np.float32(0.5)
    mineig = (ah + ch) - np.sqrt((ah - ch) * (ah - ch) + b * b)
    return sums, mineig, harris


@pytest.mark.parametrize("ks,period,square", [(-1, 4, 2), (5, 6, 3), (7, 8, 4)])
def test_int64_headroom(ibt, ks, period, square):
    """blockSize-31 window sums far beyond int32: 0/255 stripes drive sum(sx^2) to 1.6e10 / 9.8e10 / 1.5e13 (Harris sees it; on
    pure stripes lambda_min is 0), checkerboards put sum(sx^2) and sum(sy^2) at 3x / 13x / 2300x 2^31 with lambda_min > 0"""
    x = np.arange(160)
    stripes = np.tile(np.where((x % period) < period // 2, 255, 0).astype(np.uint8), (96, 1))
    yy, xx = np.mgrid[0:96, 0:160]
    checker = np.where(((yy // square) + (xx // square)) % 2 == 0, 255, 0).astype(np.uint8)
    for img, what in ((stripes, "stripes"), (checker, "checker")):
        sums, mineig, harris = _exact_maps(img, 31, ks)
        if what == "stripes":
            assert sums[0].max() > 7 * 2 ** 31, (what, sums[0].max())
        else:
            assert min(sums[0].max(), sums[2].max()) > 3 * 2 ** 31 * 0.99 and mineig.max() > 0, (what, sums[0].max())
            got = ibt.cornerMinEigenVal(img, 31, ksize=ks)
            assert np.array_equal(got, mineig), (what, np.abs(got - mineig).max())
        got = ibt.cornerHarris(img, 31, ks, 0.04)
        assert np.array_equal(got, harris), (what, np.abs(got - harris).max())


def test_sequence_prefetch_honours_gradient_size(ibt):
    """SequenceTracker.gftt_prefetch + seed(prefetched=) computes the configured aperture, as goodFeaturesToTrack does, and
    both paths reject the same unsupported apertures"""
    from iceberg_tracking_code_b200.tracking import SequenceTracker
    img = torch.from_numpy(_frame(500, 700, 17)).cuda()
    gp = dict(maxCorners=3000, qualityLevel=0.007, minDistance=10, blockSize=10, gradientSize=5)
    lp = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.01))
    trk = SequenceTracker(gp, lp)
    pyr = trk.prepare(img)
    n = trk.seed(pyr, None, 2, prefetched=trk.gftt_prefetch(pyr, None))
    ref = ibt.goodFeaturesToTrack(img, **gp)
    assert n == ref.shape[0] and torch.equal(trk._tracks[0], ref.reshape(-1, 2))
    assert not torch.equal(ref, ibt.goodFeaturesToTrack(img, **dict(gp, gradientSize=3)))
    for g in KC.BAD_APERTURES:
        bad = SequenceTracker(dict(gp, gradientSize=g), lp)
        with pytest.raises(ibt.error):
            bad.gftt_prefetch(pyr, None)
        with pytest.raises(ibt.error):
            bad.seed(pyr, None, 2)


def test_tiny_images_and_wide_windows(ibt, oracle):
    """images of 3..8 rows or columns and windows wider than the image, every aperture: the all-reflection paths of
    eig_ap_kernel and eig_nms_ap_kernel (REFLECT_101 indices beyond one reflection, tap rows that never roll when the image has
    fewer rows than the aperture, border strips only).  Maps against the reference within check_map_cancel's bound; corner
    lists exactly the oracle's selection on the CUDA map itself (the producer computes the map's values bit for bit), so that
    ties between mathematically equal responses are decided the same way"""
    rng = np.random.default_rng(77)
    for h, w in KC.TINY_SIZES + [(3, 200), (200, 3), (6, 130)]:
        a = rng.random((h + 2, w + 2)).astype(np.float32)
        img = np.clip((a[1:, 1:] + a[:-1, :-1])[:h, :w] * 100 + (rng.random((h, w)) > 0.6) * 60, 0, 255).astype(np.uint8)
        mask = (rng.random((h, w)) > 0.3).astype(np.uint8) * 255
        for ks in KC.APERTURES:
            for bs in sorted({2, min(h, w), min(h, w) + 1, 31}):
                what = (h, w, ks, bs)
                gm = ibt.cornerMinEigenVal(img, bs, ksize=ks)
                gh = ibt.cornerHarris(img, bs, ks, 0.04)
                KC.check_map_cancel(gm, KC.corner_response(img, bs, ks), img, bs, ks, False, what)
                KC.check_map_cancel(gh, KC.corner_response(img, bs, ks, True, 0.04), img, bs, ks, True, what)
                for harris, r in ((False, gm), (True, gh)):
                    for m in (None, mask):
                        for mc, q, md in ((0, 0.007, 0), (300, 0.02, 5), (0, 0.007, 10)):
                            got = ibt.goodFeaturesToTrack(img, mc, q, md, mask=m, blockSize=bs, useHarrisDetector=harris,
                                                          gradientSize=ks)
                            sel = oracle.gftt_select(r, m, mc, q, md)
                            assert np.array_equal(as_corners(got), as_corners(sel)), (what, harris, m is not None, mc, q, md)
