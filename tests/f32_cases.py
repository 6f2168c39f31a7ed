"""CPU reference of cv2's corner maps on float32 images (cv2 takes CV_8UC1 and CV_32FC1) and the shared body of the float32
checks.  OpenCV's CV_32F front end of cornerEigenValsVecs: Sobel / Scharr of the float image with the scale
1 / (sden * blockSize) (no factor 255, which only the u8 path has) on the smoothing taps, float products, double window sums
(REFLECT_101 on the product image), then the float response.

The Sobel here is taken in float64 from the float image with float64 taps (the smoothing taps times the scale rounded to float,
as OpenCV's float kernels hold them) and rounded to float once.  OpenCV computes it in float: no operation order tried -- row
taps then column taps, with and without FMA, folded symmetric pairs in either order -- reproduces the 4.13 wheel bit for bit
at every aperture (aperture 1 does; Scharr matches under none), so the maps are compared within a bound, not bit for bit.

Bound, per pixel: with g = sum |tap| * |I| (the derivative taps times the scaled smoothing taps over the aperture: the size
of every partial sum of the float Sobel), each of dx, dy is off by at most ~2 KT float epsilons of g, a product by ~4 KT of
g^2, and a window sum of products by that much of M = sum over the window of (gx^2 + gy^2).  min-eig moves by at most the sum
of the three entries' errors, Harris by ~(4 + 4k) M times it.  F32_ULPS float epsilons of M (min-eig) or of M^2 (Harris)
covers both with a margin; measured against the wheel, the largest difference is a few epsilons of M."""
import numpy as np

import ksize_cases as KC
from parity import as_corners

APERTURES = KC.APERTURES
F32_ULPS = 16
EPS = float(np.finfo(np.float32).eps)
MAP_BLOCKS = (3, 10, 31)
MAP_CROP = (slice(40, 80), slice(60, 108))      # the maps of kat_f32.npz cover this crop of the texture scene (file size)
TINY_SIZES = KC.TINY_SIZES + [(1, 1), (2, 2), (1, 9), (9, 2)]

# non-integer transforms of the golden scenes' u8 frames (kat_texture.npz / kat_iceberg.npz)
TRANSFORMS = {
    "div255": lambda f: f.astype(np.float32) / np.float32(255.0),
    "gamma": lambda f: np.power(f.astype(np.float32) / np.float32(255.0), np.float32(2.2)).astype(np.float32),
    "negaff": lambda f: (f.astype(np.float32) * np.float32(-0.37) + np.float32(12.5)).astype(np.float32),
    "large": lambda f: (f.astype(np.float32) * np.float32(4099.7) - np.float32(3.0e5)).astype(np.float32),
}
# goodFeaturesToTrack sets of kat_f32.npz (bounded maxCorners keep the file small); scene / transform / aperture rotate over them
F32_SETS = [
    dict(maxCorners=300, qualityLevel=0.01, minDistance=10, blockSize=10),
    dict(maxCorners=200, qualityLevel=0.02, minDistance=5, blockSize=3),
    dict(maxCorners=150, qualityLevel=0.01, minDistance=8, blockSize=31),
]


def set_index(ti, ks):
    return (ti + APERTURES.index(ks)) % len(F32_SETS)


def scaled_taps(ks, blockSize):
    """(derivative taps, smoothing taps * scale rounded to float) as float64"""
    d, s, sden = KC.TAPS[ks]
    scale = 1.0 / (sden * blockSize)
    return np.array(d, np.float64), np.array([np.float32(v * scale) for v in s], np.float64)


def _sep(img, kx, ky):
    """correlate kx along x then ky along y, REFLECT_101 at every border (repeated for images smaller than the aperture)"""
    h, w = img.shape
    R = len(kx) // 2
    T = sum(kx[j] * img[:, KC.r101(np.arange(w) + j - R, w)] for j in range(len(kx)) if kx[j] != 0)
    return sum(ky[i] * T[KC.r101(np.arange(h) + i - R, h), :] for i in range(len(ky)) if ky[i] != 0)


def sobel_f32(img, ks, blockSize):
    """(dx, dy) float32: the scaled Sobel / Scharr in float64, rounded once"""
    d, s = scaled_taps(ks, blockSize)
    I = np.asarray(img, np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        return _sep(I, d, s).astype(np.float32), _sep(I, s, d).astype(np.float32)


def _box(P, blockSize):
    h, w = P.shape
    a0 = -(blockSize // 2)
    V = sum(P[KC.r101(np.arange(h) + a0 + i, h), :] for i in range(blockSize))
    return sum(V[:, KC.r101(np.arange(w) + a0 + j, w)] for j in range(blockSize))


def corner_response(img, blockSize, ksize=3, harris=False, k=0.04):
    if ksize not in KC.TAPS:
        raise ValueError("unsupported aperture %r" % (ksize,))
    dx, dy = sobel_f32(img, ksize, blockSize)
    with np.errstate(over="ignore", invalid="ignore"):
        a, b, c = (_box((P).astype(np.float64), blockSize).astype(np.float32) for P in (dx * dx, dx * dy, dy * dy))
        if harris:
            return (a * c - b * b) - np.float32(k) * ((a + c) * (a + c))
        a, c = a * np.float32(0.5), c * np.float32(0.5)
        return (a + c) - np.sqrt((a - c) * (a - c) + b * b)


def bound(img, blockSize, ksize, harris, k=0.04):
    """per-pixel bound of |map - cv2's map| (module docstring)"""
    d, s = scaled_taps(ksize, blockSize)
    A = np.abs(np.asarray(img, np.float64))
    gx, gy = _sep(A, np.abs(d), np.abs(s)), _sep(A, np.abs(s), np.abs(d))
    M = _box(gx * gx + gy * gy, blockSize)
    return F32_ULPS * EPS * (M * M * (1.0 + abs(k)) if harris else M)


def check_map(got, ref, img, blockSize, ksize, harris, what, k=0.04):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape and got.dtype == np.float32, what
    assert np.all(np.isfinite(got)) and np.all(np.isfinite(ref)), what
    excess = np.abs(got.astype(np.float64) - ref.astype(np.float64)) - bound(img, blockSize, ksize, harris, k)
    assert np.all(excess <= 0), (what, float(excess.max()))


class Reference:
    """cv2 signatures over corner_response (+ the oracle's selection for goodFeaturesToTrack)"""

    def __init__(self, oracle):
        self.oracle = oracle

    def cornerMinEigenVal(self, img, blockSize, ksize=3):
        return corner_response(img, blockSize, ksize)

    def cornerHarris(self, img, blockSize, ksize=3, k=0.04):
        return corner_response(img, blockSize, ksize, True, k)

    def goodFeaturesToTrack(self, image, maxCorners, qualityLevel, minDistance, mask=None, blockSize=3,
                            useHarrisDetector=False, k=0.04, gradientSize=3):
        resp = corner_response(image, blockSize, gradientSize, useHarrisDetector, k)
        return self.oracle.gftt_select(resp, mask, maxCorners, qualityLevel, minDistance)


def check_lists(got, ref, harris, what, ref_map=None, oracle=None, mask=None, gp=None):
    """the rule of the aperture checks: cv2's list exactly, or the selection run on cv2's own map (ref_map, when given)
    exactly; failing both, the same corner set up to CORNER_OVERLAP -- or one corner, in short lists.  The maps agree to
    rounding only, so corners of almost equal response may swap: the last one above the threshold or maxCorners, or
    neighbours in the order (on images whose offset dwarfs their gradients, e.g. 1e4 + 250 * texture, many are that close,
    so the order is not compared).  Measured: 159 of kat_f32.npz's 160 lists come out identical, the other (7 corners) swaps one."""
    if np.array_equal(as_corners(got), as_corners(ref)):
        return
    if ref_map is not None:
        sel = oracle.gftt_select(ref_map, mask, gp["maxCorners"], gp["qualityLevel"], gp["minDistance"])
        if np.array_equal(as_corners(got), as_corners(sel)):
            return
    got, ref = as_corners(got), as_corners(ref)
    n = max(len(got), len(ref))
    sg, sr = (set(map(tuple, a.reshape(-1, 2).astype(np.int64).tolist())) for a in (got, ref))
    assert abs(len(got) - len(ref)) <= 1 and len(sr - sg) <= max(1, int((1 - KC.CORNER_OVERLAP) * n)), (what, len(got), len(ref))


def golden_keys(scene, tname, ks):
    return ["%s_%s_g%d_h%d_m%d" % (scene, tname, ks, h, m) for h in (0, 1) for m in (0, 1)]


def check_f32_golden(impl, g, scenes):
    """impl: cv2's cornerMinEigenVal / cornerHarris / goodFeaturesToTrack signatures; g = kat_f32.npz.  Maps: of the texture
    scene's crop under each transform, every aperture and MAP_BLOCKS, within the bound; tiny random images likewise.  Lists:
    both scenes under each transform, every aperture, both responses, with and without the mask."""
    for ti, (tname, T) in enumerate(TRANSFORMS.items()):
        for name, sc in scenes.items():
            f = T(sc["f0"])
            crop = np.ascontiguousarray(f[MAP_CROP])
            for ks in APERTURES:
                if name == "texture":
                    for bs in MAP_BLOCKS:
                        what = (tname, ks, bs)
                        check_map(impl.cornerMinEigenVal(crop, bs, ksize=ks), g["map_%s_mineig_g%d_bs%d" % (tname, ks, bs)],
                                  crop, bs, ks, False, what)
                        check_map(impl.cornerHarris(crop, bs, ks, 0.04), g["map_%s_harris_g%d_bs%d" % (tname, ks, bs)],
                                  crop, bs, ks, True, what)
                gp = F32_SETS[set_index(ti, ks)]
                for key, (harris, m) in zip(golden_keys(name, tname, ks), [(h, m) for h in (0, 1) for m in (None, sc["mask"])]):
                    got = impl.goodFeaturesToTrack(f, mask=m, useHarrisDetector=bool(harris), gradientSize=ks, **gp)
                    check_lists(got, g["gftt_" + key], harris, key)
    for (h, w) in TINY_SIZES:
        img = g["tiny_img_%dx%d" % (h, w)]
        for ks in APERTURES:
            for bs in (2, min(h, w) + 1):
                what = (h, w, ks, bs)
                check_map(impl.cornerMinEigenVal(img, bs, ksize=ks), g["tiny_mineig_%dx%d_g%d_bs%d" % (h, w, ks, bs)], img, bs,
                          ks, False, what)
                check_map(impl.cornerHarris(img, bs, ks, 0.04), g["tiny_harris_%dx%d_g%d_bs%d" % (h, w, ks, bs)], img, bs,
                          ks, True, what)


def tiny_image(h, w, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((h, w)) * 3.1 - 0.7).astype(np.float32)
