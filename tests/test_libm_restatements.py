"""The libm functions whose bits the GPU kernels reproduce, restated and checked against numpy on this host (no GPU).

numpy's hypot calls the C library's hypot / hypotf.  The kernels compute the forward-backward distance (float32, lk.cu)
and the s2 speeds (float64, utm.cu) the way glibc does, so that the tracks and hourly files equal numpy's bit for bit.
If a host's libm computes something else, these tests fail and name the cause, where the GPU tests could only report an
unexplained mismatch in the last bits.

glibc >= 2.35 computes hypot with the algorithm of Borges, "An Improved Algorithm for hypot(a, b)" (arXiv:1904.09481),
non-FMA variant: scale by 2^-600 above 2^511 and by 2^600 below 2^-459, return |x| + |y| when one term is negligible
(ratio 2^-54), otherwise h = sqrt(ax^2 + ay^2) and one correction step h -= (t1 + t2) / (2h).  It is not correctly
rounded.  hypotf is (float) sqrt((double) x * x + (double) y * y), which is correctly rounded but for double rounding.
"""
import numpy as np

SCALE, LARGE, TINY, EPS = 2.0 ** -600, 2.0 ** 511, 2.0 ** -459, 2.0 ** -54


def _kernel(ax, ay):
    """ax >= ay >= 0, squares in range.  Every numpy operation is one IEEE operation, as in the C source."""
    h = np.sqrt(ax * ax + ay * ay)
    near = h <= 2.0 * ay
    d1 = h - ay
    t1a = ax * (2.0 * d1 - ax)
    t2a = (d1 - 2.0 * (ax - ay)) * d1
    d2 = h - ax
    t1b = 2.0 * d2 * (ax - 2.0 * ay)
    t2b = (4.0 * d2 - ay) * ay + d2 * d2
    t1, t2 = np.where(near, t1a, t1b), np.where(near, t2a, t2b)
    return h - (t1 + t2) / (2.0 * h)


def glibc_hypot(x, y):
    """float64 hypot as glibc >= 2.35 computes it without FMA (sysdeps/ieee754/dbl-64/e_hypot.c)"""
    x, y = np.abs(np.asarray(x, np.float64)), np.abs(np.asarray(y, np.float64))
    with np.errstate(all="ignore"):
        ax, ay = np.where(x < y, y, x), np.where(x < y, x, y)
        big = ax > LARGE
        tiny = ~big & (ay < TINY)
        k = np.where(big, _kernel(ax * SCALE, ay * SCALE) / SCALE,
                     np.where(tiny, _kernel(ax / SCALE, ay / SCALE) * SCALE, _kernel(ax, ay)))
        negligible = np.where(tiny, ax >= ay / EPS, ay <= ax * EPS)
        r = np.where(negligible, ax + ay, k)
        return np.where(np.isinf(x) | np.isinf(y), np.inf, np.where(np.isnan(x) | np.isnan(y), np.nan, r))


def glibc_hypotf(x, y):
    """float32 hypot as glibc computes it (sysdeps/ieee754/flt-32/e_hypotf.c)"""
    x, y = np.asarray(x, np.float32).astype(np.float64), np.asarray(y, np.float32).astype(np.float64)
    with np.errstate(all="ignore"):
        r = np.sqrt(x * x + y * y).astype(np.float32)
        return np.where(np.isinf(x) | np.isinf(y), np.float32(np.inf), np.where(np.isnan(x) | np.isnan(y), np.float32(np.nan), r))


def _same(a, b):
    return (a == b) | (np.isnan(a) & np.isnan(b))


def _pairs64(rng, n):
    """magnitudes from 1e-320 to 1e300: independent exponents (mostly the negligible branch), exponents within 2^-20 .. 1 of
    each other (the correction step, both of its branches), near-equal pairs, pairs around 2^-511 .. 2^-459 (where only the
    scaled path gives libm's bits), the scaling bounds, zeros and non-finite"""
    lo, hi = np.log10(1e-320), np.log10(1e300)
    sgn = lambda m: rng.choice([-1.0, 1.0], m)
    m = n // 5
    x1, y1 = 10.0 ** rng.uniform(lo, hi, m), 10.0 ** rng.uniform(lo, hi, m)
    x2 = 10.0 ** rng.uniform(lo, hi, 2 * m)
    y2 = x2 * 2.0 ** rng.uniform(-20, 0, 2 * m)
    x3 = 10.0 ** rng.uniform(lo, hi, m)
    y3 = x3 * (1 + rng.uniform(-1e-3, 1e-3, m))
    x4 = 2.0 ** rng.uniform(-515, -455, m)
    y4 = x4 * 2.0 ** rng.uniform(-3, 0, m)
    edges = np.array([0.0, 5e-324, 2.0 ** -1022, TINY, np.nextafter(TINY, 0), np.nextafter(TINY, 1), LARGE,
                      np.nextafter(LARGE, 0), np.nextafter(LARGE, np.inf), 1.0, 3.0, 1.7976931348623157e308, np.inf, np.nan])
    ex, ey = (a.ravel() for a in np.meshgrid(edges, edges))
    x = np.concatenate([x1, x2, x3, x4, ex]) * np.concatenate([sgn(5 * m), np.ones(len(ex))])
    y = np.concatenate([y1, y2, y3, y4, ey]) * np.concatenate([sgn(5 * m), np.ones(len(ey))])
    swap = rng.random(len(x)) < 0.5
    return np.where(swap, y, x), np.where(swap, x, y)


def test_hypot_float64_is_glibc_restatement():
    rng = np.random.default_rng(11)
    x, y = _pairs64(rng, 1_000_000)
    with np.errstate(all="ignore"):
        got = np.hypot(x, y)
    want = glibc_hypot(x, y)
    bad = np.flatnonzero(~_same(got, want))
    assert not len(bad), "np.hypot is not glibc's non-FMA hypot at %d of %d pairs, e.g. hypot(%r, %r) = %r, restatement %r" % (
        len(bad), len(x), x[bad[0]], y[bad[0]], got[bad[0]], want[bad[0]])
    # the pairs reach the correction step, and it matters: a plain rounded sqrt of the sum of squares differs from it
    with np.errstate(all="ignore"):
        plain = np.sqrt(x * x + y * y)
    normal = (np.abs(x) > 1e-150) & (np.abs(x) < 1e150) & (np.abs(y) > 1e-150) & (np.abs(y) < 1e150)
    assert (~_same(plain, got) & normal).sum() > 100
    # and every branch of the C source runs
    ax, ay = np.maximum(np.abs(x), np.abs(y)), np.minimum(np.abs(x), np.abs(y))
    fin = np.isfinite(ax)
    assert ((ax > LARGE) & (ay > ax * EPS) & fin).any() and ((ay < TINY) & (ay > 0) & (ax * EPS < ay)).any()
    assert ((ax <= LARGE) & (ay >= TINY) & (ay <= ax * EPS)).any()


def test_hypot_float64_scalars_take_the_same_path():
    """Python scalars through np.hypot, as the s2 oracle computes each segment's speed"""
    rng = np.random.default_rng(12)
    x, y = _pairs64(rng, 4000)
    want = glibc_hypot(x, y)
    with np.errstate(all="ignore"):
        got = np.array([np.hypot(float(a), float(b)) for a, b in zip(x, y)])
    assert _same(got, want).all()


def test_hypot_float32_is_double_sqrt():
    rng = np.random.default_rng(13)
    n = 1_000_000
    lo, hi = np.log10(1e-45), np.log10(3e38)
    x = (10.0 ** rng.uniform(lo, hi, n)).astype(np.float32)
    y = (x.astype(np.float64) * 2.0 ** rng.uniform(-30, 0, n)).astype(np.float32)
    # FB distances: |p0 - p0r| of coordinates up to 6000 px that agree to a pixel or so
    p0 = rng.uniform(0, 6000, (n, 2)).astype(np.float32)
    fx, fy = np.abs(p0 - (p0 + rng.normal(0, 0.7, (n, 2))).astype(np.float32)).T
    edges = np.array([0, 1e-45, 1.1754944e-38, 1, 3.4028235e38, np.inf, -np.inf, np.nan], np.float32)
    ex, ey = (a.ravel() for a in np.meshgrid(edges, edges))
    x, y = np.concatenate([x, fx, ex]), np.concatenate([y, fy, ey])
    swap = rng.random(len(x)) < 0.5
    x, y = np.where(swap, y, x), np.where(swap, x, y)
    with np.errstate(all="ignore"):
        got = np.hypot(x, y)
    assert got.dtype == np.float32
    want = glibc_hypotf(x, y)
    bad = np.flatnonzero(~_same(got, want))
    assert not len(bad), "np.hypot(float32) is not (float) sqrt of the double sum at %d pairs, e.g. (%r, %r)" % (
        len(bad), x[bad[0]], y[bad[0]])
    # inf beats NaN, as glibc's hypotf has it
    assert np.hypot(np.float32(np.inf), np.float32(np.nan)) == np.inf
