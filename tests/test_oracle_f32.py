"""The CPU reference of cv2's corner maps on float32 images (tests/f32_cases.py) against cv2's answers, and the argument checks
of the float32 entry points that run without a GPU."""
import ctypes as C

import numpy as np
import pytest

import f32_cases as FC


@pytest.fixture(scope="module")
def scenes(golden):
    return {name: golden("kat_%s.npz" % name) for name in ("texture", "iceberg")}


def test_reference_golden(oracle, golden, scenes):
    """maps and corner lists of every aperture on the transformed scenes and tiny images against kat_f32.npz (cv2 4.13)"""
    FC.check_f32_golden(FC.Reference(oracle), golden("kat_f32.npz"), scenes)


def test_bound_is_not_vacuous(golden):
    """the bound sits far below the responses it guards: on the golden maps it is at most 1e-3 of the map's range (measured
    1e-4 .. 5.6e-4: it grows with |I| / |grad I|, as the float Sobel's rounding does)"""
    g = golden("kat_f32.npz")
    for tname, T in FC.TRANSFORMS.items():
        crop = np.ascontiguousarray(T(golden("kat_texture.npz")["f0"])[FC.MAP_CROP])
        for ks in FC.APERTURES:
            ref = g["map_%s_mineig_g%d_bs10" % (tname, ks)]
            assert FC.bound(crop, 10, ks, False).max() < 1e-3 * np.abs(ref).max(), (tname, ks)


def _scene(rng, h, w):
    a = rng.random((h + 2, w + 2))
    a = (a[1:, 1:] + a[:-1, :-1])[:h, :w] + (np.kron(rng.random((h // 4 + 2, w // 4 + 2)) > 0.5, np.ones((4, 4)))[:h, :w])
    lo, span = rng.choice([(0.0, 1.0), (-3.5, 0.02), (1e4, 250.0), (-2e-3, 1e-3)])
    return (lo + span * a).astype(np.float32)


@pytest.mark.parametrize("seed", range(4))
def test_reference_live_cv2(oracle, seed):
    """random float images (value ranges from 1e-3 to 1e4, offsets of either sign), every aperture: maps within the bound,
    lists by the rule of FC.check_lists"""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(400 + seed)
    ref = FC.Reference(oracle)
    for ks in FC.APERTURES:
        h, w = int(rng.integers(3, 120)), int(rng.integers(3, 160))
        img = _scene(rng, h, w)
        mask = (rng.random((h, w)) > 0.2).astype(np.uint8) * 255
        for bs in (2, 5, int(rng.integers(2, 32))):      # (blockSize 1: lambda_min is 0 up to rounding)
            FC.check_map(ref.cornerMinEigenVal(img, bs, ks), cv2.cornerMinEigenVal(img, bs, ksize=ks), img, bs, ks, False,
                         (seed, ks, bs))
            FC.check_map(ref.cornerHarris(img, bs, ks, 0.04), cv2.cornerHarris(img, bs, ks, 0.04), img, bs, ks, True,
                         (seed, ks, bs))
            for harris in (False, True):
                gp = dict(maxCorners=int(rng.integers(0, 200)), qualityLevel=0.01, minDistance=float(rng.integers(0, 8)),
                          blockSize=bs)
                want = cv2.goodFeaturesToTrack(img, mask=mask, useHarrisDetector=harris, gradientSize=ks, **gp)
                cmap = cv2.cornerHarris(img, bs, ks, 0.04) if harris else cv2.cornerMinEigenVal(img, bs, ksize=ks)
                got = ref.goodFeaturesToTrack(img, mask=mask, useHarrisDetector=harris, gradientSize=ks, **gp)
                FC.check_lists(got, want, harris, (seed, ks, bs, harris), cmap, oracle, mask, gp)


def test_dtypes_rejected_like_cv2():
    """every dtype but u8 and float32 raises cv.error before any device work, worded like cv2's assertion"""
    from iceberg_tracking_code_b200 import cv
    for dt in (np.float64, np.float16, np.int16, np.uint16, np.int32):
        img = np.zeros((16, 16), dt)
        for call in (lambda: cv.goodFeaturesToTrack(img, 10, 0.01, 1), lambda: cv.cornerMinEigenVal(img, 3),
                     lambda: cv.cornerHarris(img, 3, 3, 0.04)):
            with pytest.raises(cv.error, match=r"CV_8UC1 \|\| src.type\(\) == CV_32FC1"):
                call()


def test_f32_entry_points_reject_without_cuda():
    """invalid arguments of ibt_gftt_f32src / ibt_min_eigen_f32src / ibt_corner_harris_f32src return IBT_E_INVALID before any
    CUDA call (the pointers below are never dereferenced): null or misaligned image, pitch not a multiple of 4 or below 4 W,
    bad aperture or blockSize"""
    from iceberg_tracking_code_b200 import build
    build.build()
    from iceberg_tracking_code_b200 import _native as N
    lib = N.lib()
    assert lib.ibt_version() == 104
    E = N.IBT_E_INVALID
    good, odd = C.c_void_p(0x10000), C.c_void_p(0x10002)
    dst = C.c_void_p(0x20000)
    H, W = 64, 64
    cases = [(good, W * 4, 3, 3), (None, W * 4, 3, 3), (odd, W * 4, 3, 3), (good, W * 4 + 2, 3, 3), (good, W * 4 - 4, 3, 3),
             (good, W * 4, 2, 3), (good, W * 4, 9, 3), (good, W * 4, 3, 0), (good, W * 4, 3, 32)]
    for img, pitch, ks, bs in cases:
        valid = img is good and pitch % 4 == 0 and pitch >= W * 4 and ks in FC.APERTURES and 1 <= bs <= 31
        if valid:
            continue
        assert lib.ibt_min_eigen_f32src(img, H, W, pitch, bs, ks, dst, W * 4, None) == E, (img, pitch, ks, bs)
        assert lib.ibt_corner_harris_f32src(img, H, W, pitch, bs, ks, 0.04, dst, W * 4, None) == E, (img, pitch, ks, bs)
        cnt = C.c_int(-1)
        assert lib.ibt_gftt_f32src(img, pitch, None, 0, H, W, 0, 0.01, 1.0, bs, ks, 0, 0.04, good, 1 << 30, dst, 100,
                                   C.byref(cnt), None) == E, (img, pitch, ks, bs)
        assert cnt.value == 0
    # map pitch, NaN k, null output
    assert lib.ibt_min_eigen_f32src(good, H, W, W * 4, 3, 3, dst, W * 4 - 4, None) == E
    assert lib.ibt_min_eigen_f32src(good, H, W, W * 4, 3, 3, None, W * 4, None) == E
    assert lib.ibt_corner_harris_f32src(good, H, W, W * 4, 3, 3, float("nan"), dst, W * 4, None) == E
    assert lib.ibt_gftt_f32src(good, W * 4, None, 0, 2, W, 0, 0.01, 1.0, 3, 3, 0, 0.04, good, 1 << 30, dst, 100, None,
                               None) == E
