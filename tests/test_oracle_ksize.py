"""The CPU reference of the Sobel apertures other than 3 (tests/ksize_cases.py) against cv2's answers, and the argument checks
of the aperture-taking API that run without a GPU."""
import ctypes as C

import numpy as np
import pytest

import ksize_cases as KC


@pytest.fixture(scope="module")
def scenes(golden):
    return {name: golden("kat_%s.npz" % name) for name in ("texture", "iceberg")}


def test_reference_golden(oracle, golden, scenes):
    """maps and corner lists of every aperture other than 3 against kat_ksize.npz (cv2 4.13)"""
    KC.check_ksize_golden(KC.Reference(oracle), golden("kat_ksize.npz"), scenes)


def test_aperture3_is_the_oracle(oracle):
    """aperture 3 through the aperture-taking reference is orc_mineig_f32 / orc_harris_f32 byte for byte"""
    rng = np.random.default_rng(31)
    ref = KC.Reference(oracle, oracle_order=True)
    for (h, w), bs in (((3, 3), 1), ((5, 8), 4), ((37, 29), 7), ((24, 40), 31)):
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        assert ref.cornerMinEigenVal(img, bs, 3).tobytes() == oracle.cornerMinEigenVal(img, bs).tobytes(), (h, w, bs)
        assert ref.cornerHarris(img, bs, 3, 0.04).tobytes() == oracle.cornerHarris(img, bs, 3, 0.04).tobytes(), (h, w, bs)


def _scene(rng, h, w):
    """blurred noise with blocks: corners of every strength"""
    a = rng.random((h + 4, w + 4)).astype(np.float32)
    a = (a + np.roll(a, 1, 0) + np.roll(a, 1, 1) + np.roll(np.roll(a, 1, 0), 1, 1))[2:2 + h, 2:2 + w]
    blocks = np.kron(rng.random((h // 5 + 2, w // 5 + 2)) > 0.5, np.ones((5, 5)))[:h, :w]
    return np.clip(a * 50 + blocks * 150, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("seed", range(6))
def test_reference_live_cv2(oracle, seed):
    """against the cv2 wheel on seeded scenes of 9x9 .. 240x321: every aperture, blockSize 1..31, masks, min-eig and Harris"""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(4100 + seed)
    sizes = [(240, 321), (61, 83), (int(rng.integers(9, 14)), int(rng.integers(9, 14))), (int(rng.integers(9, 14)), 97),
             (53, int(rng.integers(9, 14))), (int(rng.integers(20, 240)), int(rng.integers(20, 321)))]
    ref = KC.Reference(oracle)
    for h, w in sizes:
        img = _scene(rng, h, w)
        mask = (rng.random((h, w)) > 0.3).astype(np.uint8) * 255
        for ks in KC.APERTURES:
            bs = int(rng.choice([b for b in (1, 2, 3, 5, 10, 15, 31) if b <= min(h, w)]))
            what = (seed, h, w, ks, bs)
            # blockSize 1: the tensor of one pixel has rank 1, lambda_min is 0 up to rounding noise in cv2 as here
            # under 16 px on a side the windows are mostly reflections: lambda_min's cancellation, see check_map_cancel
            if bs > 1:
                if min(h, w) < 16:
                    KC.check_map_cancel(ref.cornerMinEigenVal(img, bs, ks), cv2.cornerMinEigenVal(img, bs, ksize=ks), img, bs,
                                        ks, False, what)
                else:
                    KC.check_map(ref.cornerMinEigenVal(img, bs, ks), cv2.cornerMinEigenVal(img, bs, ksize=ks), what)
            KC.check_map(ref.cornerHarris(img, bs, ks, 0.04), cv2.cornerHarris(img, bs, ks, 0.04), what)
            for harris in ((False, True) if bs > 1 else (True,)):
                gp = dict(maxCorners=int(rng.choice([0, 300])), qualityLevel=float(rng.choice([0.007, 0.02])),
                          minDistance=float(rng.choice([0, 5, 10])), blockSize=bs, useHarrisDetector=harris, k=0.04,
                          gradientSize=ks)
                m = mask if rng.random() < 0.5 else None
                KC.check_lists(ref.goodFeaturesToTrack(img, mask=m, **gp), cv2.goodFeaturesToTrack(img, mask=m, **gp),
                               harris, (what, gp, m is not None))


def test_reference_live_cv2_tiny(oracle):
    """images of 3..8 rows or columns (narrower or shorter than the aperture: REFLECT_101 repeats) and windows wider than the
    image, every aperture, min-eig and Harris, masks.  Nearly every pixel's window is made of reflections of a few pixels, so
    the responses are small differences of large terms (check_map_cancel bounds the maps by that scale), and many responses
    are mathematically equal, so rounding decides which of two equal neighbours is a raw 3x3 maximum.  The corner lists must
    pass check_lists in >= 99 % of the cases; where one does not, cv2's own list must be the oracle's selection run on cv2's
    own map -- the difference is then the map's rounding, which the map check bounds."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(4200)
    ref = KC.Reference(oracle)
    cases = passed = 0
    for h, w in KC.TINY_SIZES + [(int(rng.integers(3, 9)), int(rng.integers(3, 60))) for _ in range(12)] + \
            [(int(rng.integers(3, 60)), int(rng.integers(3, 9))) for _ in range(12)]:
        img = _scene(rng, h, w)
        mask = (rng.random((h, w)) > 0.3).astype(np.uint8) * 255
        for ks in KC.APERTURES:
            for bs in (int(rng.integers(2, min(h, w) + 1)), int(rng.integers(min(h, w) + 1, 32))):
                what = (h, w, ks, bs)
                cm, ch = cv2.cornerMinEigenVal(img, bs, ksize=ks), cv2.cornerHarris(img, bs, ks, 0.04)
                KC.check_map_cancel(ref.cornerMinEigenVal(img, bs, ks), cm, img, bs, ks, False, what)
                KC.check_map_cancel(ref.cornerHarris(img, bs, ks, 0.04), ch, img, bs, ks, True, what)
                for harris in (False, True):
                    gp = dict(maxCorners=int(rng.choice([0, 300])), qualityLevel=float(rng.choice([0.007, 0.02])),
                              minDistance=float(rng.choice([0, 5, 10])), blockSize=bs, useHarrisDetector=harris, k=0.04,
                              gradientSize=ks)
                    m = mask if rng.random() < 0.5 else None
                    want = cv2.goodFeaturesToTrack(img, mask=m, **gp)
                    cases += 1
                    try:
                        KC.check_lists(ref.goodFeaturesToTrack(img, mask=m, **gp), want, harris, (what, gp))
                        passed += 1
                    except AssertionError:
                        sel = oracle.gftt_select(ch if harris else cm, m, gp["maxCorners"], gp["qualityLevel"], gp["minDistance"])
                        assert np.array_equal(KC.as_corners(sel), KC.as_corners(want)), (what, gp)
    assert passed >= 0.99 * cases, (passed, cases)


def test_unsupported_apertures_are_rejected_without_a_gpu():
    """cv.py raises cv.error naming the supported set; every aperture-taking entry point returns IBT_E_INVALID before any CUDA
    call (the valid-looking arguments would otherwise reach the device)"""
    from iceberg_tracking_code_b200 import build
    build.build()
    from iceberg_tracking_code_b200 import _native as N, cv
    img = np.zeros((32, 32), np.uint8)
    for g in KC.BAD_APERTURES:
        with pytest.raises(cv.error, match=r"-1 \(Scharr\), 1, 3, 5, 7"):
            cv.cornerMinEigenVal(img, 3, ksize=g)
        with pytest.raises(cv.error, match=r"-1 \(Scharr\), 1, 3, 5, 7"):
            cv.cornerHarris(img, 3, g, 0.04)
        with pytest.raises(cv.error, match=r"-1 \(Scharr\), 1, 3, 5, 7"):
            cv.goodFeaturesToTrack(img, 10, 0.01, 5, gradientSize=g)
    lib = N.lib()
    assert lib.ibt_version() >= 102
    fake = C.c_void_p(1 << 20)                   # never dereferenced: validation returns first
    for g in KC.BAD_APERTURES:
        assert lib.ibt_min_eigen_ksize_f32(fake, 32, 32, 32, 3, g, fake, 128, None) == N.IBT_E_INVALID, g
        assert lib.ibt_corner_harris_ksize_f32(fake, 32, 32, 32, 3, g, 0.04, fake, 128, None) == N.IBT_E_INVALID, g
        cnt = C.c_int(7)
        assert lib.ibt_gftt_ksize(fake, 32, None, 0, 32, 32, 10, 0.01, 5.0, 3, g, 0, 0.04, fake, 1 << 30, fake, 100,
                                  C.byref(cnt), None) == N.IBT_E_INVALID, g
        assert cnt.value == 0
        assert lib.ibt_gftt_async_ksize(fake, 32, None, 0, 32, 32, 10, 0.01, 5.0, 3, g, 0, 0.04, fake, 1 << 30, fake, 100,
                                        fake, None) == N.IBT_E_INVALID, g
