"""CPU reference of cv2's corner maps for every Sobel aperture (ksize / gradientSize = -1 (Scharr), 1, 3, 5, 7) and the shared
body of the aperture checks.  The C oracle restates aperture 3 only (oracle/ibt_oracle.c); this is the same front end of
OpenCV's cornerEigenValsVecs in numpy, for any aperture: exact integer Sobel on the u8 image (REFLECT_101, repeated for images
smaller than the aperture), one rounding by the float scale, float products, double window sums (REFLECT_101 on the product
image), then the float response.  Corner lists run the oracle's selection (orc_gftt_select) on these maps."""
import numpy as np

from parity import as_corners, corner_overlap, CORNER_OVERLAP
from harris_cases import MAP_TOL, SAME_RANK

APERTURES = (-1, 1, 3, 5, 7)
OTHER_APERTURES = (-1, 1, 5, 7)
BAD_APERTURES = (0, 2, 9, -3)
SAME_RANK_MINEIG = 0.99
CANCEL_ULPS = 256
TINY_SIZES = [(3, 3), (3, 8), (8, 3), (5, 7), (4, 40), (37, 6), (7, 7)]

# (derivative taps d, smoothing taps s, sden): dx correlates d along x and s along y, scale = 1 / (sden * blockSize * 255)
TAPS = {
    1: ((-1, 0, 1), (0, 1, 0), 1.0),
    3: ((-1, 0, 1), (1, 2, 1), 4.0),
    -1: ((-1, 0, 1), (3, 10, 3), 8.0),
    5: ((-1, -2, 0, 2, 1), (1, 4, 6, 4, 1), 16.0),
    7: ((-1, -4, -5, 0, 5, 4, 1), (1, 6, 15, 20, 15, 6, 1), 64.0),
}

# goodFeaturesToTrack parameter sets of kat_ksize.npz: the reference's (s1:240-243) and a small-blockSize one
KSIZE_SETS = [
    dict(maxCorners=0, qualityLevel=0.007, minDistance=10, blockSize=10),
    dict(maxCorners=300, qualityLevel=0.01, minDistance=5, blockSize=3),
]
MAP_CROP = (slice(40, 112), slice(60, 172))      # the maps of kat_ksize.npz cover this crop of each scene (file size)
MAP_BLOCKS = (3, 10)


def r101(i, n):
    """REFLECT_101 index for any i (numpy)"""
    i = np.asarray(i, np.int64)
    if n == 1:
        return np.zeros_like(i)
    p = 2 * (n - 1)
    i = np.mod(i, p)
    return np.where(i < n, i, p - i)


def sobel_int(img, ksize):
    """exact integer (sx, sy) of the u8 image, int64"""
    d, s, _ = TAPS[ksize]
    img = np.asarray(img, np.int64)
    h, w = img.shape
    R = len(d) // 2
    cols = [r101(np.arange(w) + j - R, w) for j in range(len(d))]
    rows = [r101(np.arange(h) + i - R, h) for i in range(len(d))]
    hd = sum(d[j] * img[:, cols[j]] for j in range(len(d)))
    hs = sum(s[j] * img[:, cols[j]] for j in range(len(d)))
    sx = sum(s[i] * hd[rows[i], :] for i in range(len(d)))
    sy = sum(d[i] * hs[rows[i], :] for i in range(len(d)))
    return sx, sy


def window_sums(sx, sy, blockSize, ksize, oracle_order=False):
    """double window sums of the float products.  oracle_order adds the blockSize^2 terms of a pixel in orc_corner_response's
    order (rows outer, columns inner): the same doubles as the C oracle, at blockSize^2 array passes; otherwise separable."""
    _, _, sden = TAPS[ksize]
    scale = np.float32(1.0 / (sden * blockSize * 255.0))
    dx, dy = sx.astype(np.float32) * scale, sy.astype(np.float32) * scale
    planes = [(dx * dx).astype(np.float64), (dx * dy).astype(np.float64), (dy * dy).astype(np.float64)]
    h, w = sx.shape
    a0 = -(blockSize // 2)
    rows = [r101(np.arange(h) + a0 + i, h) for i in range(blockSize)]
    cols = [r101(np.arange(w) + a0 + j, w) for j in range(blockSize)]
    out = []
    for P in planes:
        if oracle_order:
            acc = np.zeros((h, w), np.float64)
            for ri in rows:
                Pr = P[ri, :]
                for cj in cols:
                    acc += Pr[:, cj]
        else:
            V = sum(P[ri, :] for ri in rows)
            acc = sum(V[:, cj] for cj in cols)
        out.append(acc)
    return out


def corner_response(img, blockSize, ksize=3, harris=False, k=0.04, oracle_order=False):
    if ksize not in TAPS:
        raise ValueError("unsupported aperture %r" % (ksize,))
    sx, sy = sobel_int(img, ksize)
    sxx, sxy, syy = window_sums(sx, sy, blockSize, ksize, oracle_order)
    with np.errstate(over="ignore", invalid="ignore"):
        if harris:
            a, b, c = sxx.astype(np.float32), sxy.astype(np.float32), syy.astype(np.float32)
            kf = np.float32(k)
            return (a * c - b * b) - kf * ((a + c) * (a + c))
        a, b, c = sxx.astype(np.float32) * np.float32(0.5), sxy.astype(np.float32), syy.astype(np.float32) * np.float32(0.5)
        return (a + c) - np.sqrt((a - c) * (a - c) + b * b)


class Reference:
    """cv2 signatures over corner_response (+ the oracle's selection for goodFeaturesToTrack)"""

    def __init__(self, oracle, oracle_order=False):
        self.oracle, self.oracle_order = oracle, oracle_order

    def cornerMinEigenVal(self, img, blockSize, ksize=3):
        return corner_response(img, blockSize, ksize, False, 0.0, self.oracle_order)

    def cornerHarris(self, img, blockSize, ksize=3, k=0.04):
        return corner_response(img, blockSize, ksize, True, k, self.oracle_order)

    def goodFeaturesToTrack(self, image, maxCorners, qualityLevel, minDistance, mask=None, blockSize=3,
                            useHarrisDetector=False, k=0.04, gradientSize=3):
        resp = corner_response(image, blockSize, gradientSize, useHarrisDetector, k, self.oracle_order)
        return self.oracle.gftt_select(resp, mask, maxCorners, qualityLevel, minDistance)


def check_map(got, ref, what, tol=MAP_TOL):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape and got.dtype == np.float32, what
    assert np.abs(got - ref).max() <= tol * max(np.abs(ref).max(), np.float32(1e-30)), what


def check_map_cancel(got, ref, img, blockSize, ksize, harris, what):
    """maps of images dominated by reflections (a few pixels, windows wider than the image): both responses subtract nearly
    equal terms -- lambda_min = (a + c)/2 - sqrt(((a - c)/2)^2 + b^2), Harris = a*c - b^2 - k*(a + c)^2 -- so a rounding
    difference of the window sums shows at the size of those terms, (a + c) resp. (a + c)^2, not of the result.  Allowed per
    pixel: MAP_TOL of the range plus CANCEL_ULPS float epsilons of that scale."""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape and got.dtype == np.float32, what
    sx, sy = sobel_int(img, ksize)
    a, _, c = window_sums(sx, sy, blockSize, ksize)
    scale = (a + c) ** 2 if harris else (a + c)
    bound = MAP_TOL * float(np.abs(ref).max()) + CANCEL_ULPS * float(np.finfo(np.float32).eps) * scale
    assert np.all(np.abs(got.astype(np.float64) - ref) <= bound), (what, float(np.max(np.abs(got - ref) - bound)))


def check_lists(got, ref, harris, what):
    got, ref = as_corners(got), as_corners(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert corner_overlap(got, ref) >= CORNER_OVERLAP, what
    if len(ref):
        same = np.mean(np.all(got == ref, axis=(1, 2)))
        assert same >= (SAME_RANK if harris else SAME_RANK_MINEIG), (what, same)


def check_ksize_golden(impl, g, scenes):
    """impl: anything with cv2's cornerMinEigenVal / cornerHarris / goodFeaturesToTrack signatures; g = kat_ksize.npz"""
    for name, sc in scenes.items():
        f0, mask = sc["f0"], sc["mask"]
        crop = np.ascontiguousarray(f0[MAP_CROP])
        for ks in OTHER_APERTURES:
            for bs in MAP_BLOCKS:
                check_map(impl.cornerMinEigenVal(crop, bs, ksize=ks), g["%s_mineig_g%d_bs%d" % (name, ks, bs)], (name, ks, bs))
                check_map(impl.cornerHarris(crop, bs, ks, 0.04), g["%s_harris_g%d_bs%d" % (name, ks, bs)], (name, ks, bs))
            for si, gp in enumerate(KSIZE_SETS):
                for harris in (0, 1):
                    for mi, m in enumerate((None, mask)):
                        got = impl.goodFeaturesToTrack(f0, mask=m, useHarrisDetector=bool(harris), gradientSize=ks, **gp)
                        key = "%s_gftt%d_g%d_h%d_m%d" % (name, si, ks, harris, mi)
                        check_lists(got, g[key], harris, key)
