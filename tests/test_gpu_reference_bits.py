"""GPU: the numbers the reference compares with hard thresholds and writes to its files, bit for bit with numpy.

- The forward-backward distance dist = np.hypot(|p0 - p0r|) (float32, s1:329-333): dist < 1 decides which tracks survive,
  and dist is stored as trackquality in every *_tracks.npz.
- The s2 projection, velocities and speeds (float64, s2:243-343) and the three plausibility criteria built on them: they
  decide which tracks reach the hourly *_utm.npz files, and x, y, u, v and speed are written into them.

numpy's hypot is the C library's (tests/test_libm_restatements.py pins glibc's on the host).  The kernels restate it, so
every value is compared with array_equal, and every threshold is placed exactly on a value it is compared with and then on
that value's neighbour: the decision must flip exactly where numpy's does.  The one exception is the angle criterion:
np.arccos is not libm on every host (SVML dispatch), so its threshold sits 1e-12 relative away from the oracle's angle.
"""
import types

import numpy as np
import pytest

from parity import _f32_same
from test_gpu_lk_exact import NONFINITE, _frames, _points
from test_gpu_sequence import s1_loop_oracle

pytestmark = pytest.mark.gpu

INTERVAL = 60
# (min_speed, max_speed, max_speedfactor, max_angle, speed_threshold): the s2 defaults of the suite's other tests
CRITERIA = (0.0, 1.7, 2.5, 60.0, 0.1)
NEVER = dict(min_speed=-np.inf, max_speed=np.inf, max_speedfactor=np.inf, max_angle=np.inf, speed_threshold=np.inf)
SWEEP_T = (1, 2, 3, 7, 8, 9, 16, 17, 127, 128, 129, 136, 256, 300)


# ---- forward-backward distance -----------------------------------------------------------------------------------------
def _fb_numpy(pts, p0r):
    """s1:329-330 in float32 from the kernel's own p0r"""
    d = np.abs(np.asarray(pts, np.float32).reshape(-1, 2) - np.asarray(p0r, np.float32).reshape(-1, 2))
    return np.hypot(d[:, 0], d[:, 1])


def _fb_case(oracle, cn):
    """a few thousand points of test_gpu_lk_exact's generator: interior, border bands at every level, NONFINITE"""
    rng = np.random.default_rng(300 + cn)
    h, w, win, maxLevel = 240, 321, (21, 21), 3
    I, J = _frames(rng, "tex", h, w, cn, (2.5, -1.75))
    pts, _ = _points(rng, h, w, win, oracle.pyramid_sizes(h, w, win, maxLevel)[1], 2500)
    assert len(pts) > 2500 and _f32_same(pts[-len(NONFINITE):], np.array(NONFINITE, np.float32)).all()
    return I, J, pts, dict(winSize=win, maxLevel=maxLevel, criteria=(3, 30, 0.01))


@pytest.mark.parametrize("cn", [1, 3])
def test_fb_distance_is_numpys(ibt, oracle, cn):
    I, J, pts, lp = _fb_case(oracle, cn)
    r = ibt.calcOpticalFlowPyrLK_FB(I, J, pts, **lp)
    d_o = _fb_numpy(pts, r["p0r"])
    dist, valid = np.asarray(r["dist"]), np.asarray(r["valid"])
    bad = np.flatnonzero(~_f32_same(dist, d_o))
    assert not len(bad), "cn %d: %d FB distances differ from numpy's, e.g. #%d gpu %r numpy %r (%d ulp)" % (
        cn, len(bad), bad[0], dist[bad[0]], d_o[bad[0]],
        abs(int(dist[bad[0]].view(np.int32)) - int(d_o[bad[0]].view(np.int32))))
    assert np.array_equal(valid, d_o < 1), np.flatnonzero(valid != (d_o < 1))[:6]
    # the case reaches both sides of the threshold and non-finite distances
    assert valid.sum() > 100 and (np.isfinite(d_o) & (d_o >= 1)).any() and np.isnan(d_o).any()


@pytest.mark.parametrize("cn", [1, 3])
def test_fb_threshold_knife_edge(ibt, oracle, cn):
    """fb_threshold = numpy's distance of point k: k fails (dist < threshold is false); the next float32 up: k survives.
    LK is deterministic and the threshold is an argument, so this pins the kernel's distance to numpy's bits."""
    I, J, pts, lp = _fb_case(oracle, cn)
    r0 = ibt.calcOpticalFlowPyrLK_FB(I, J, pts, **lp)
    d_o = _fb_numpy(pts, r0["p0r"])
    cand = np.flatnonzero(np.isfinite(d_o) & (d_o > 0))
    by_one = cand[np.argsort(np.abs(d_o[cand] - 1))]
    rng = np.random.default_rng(cn)
    pick = np.unique(np.concatenate([by_one[:12], rng.choice(cand, 8, replace=False)]))
    assert len(pick) >= 15
    for k in pick:
        t = d_o[k]
        for thr, want in ((t, False), (np.nextafter(t, np.float32(np.inf)), True)):
            r = ibt.calcOpticalFlowPyrLK_FB(I, J, pts, fb_threshold=float(thr), **lp)
            assert _f32_same(r["p0r"], r0["p0r"]).all() and _f32_same(r["dist"], r0["dist"]).all()
            assert bool(r["valid"][k]) == want, (cn, int(k), float(t), float(thr))
            assert np.array_equal(r["valid"], d_o < thr), (cn, int(k))


def test_trackquality_equals_s1_restatement(ibt, oracle):
    """One group through SequenceTracker (seed, then track_len steps): tracks and trackquality equal, byte for byte, the s1
    loop restated on the CPU oracle from the same seed corners (the oracle's LK is bit-exact with the kernel's)."""
    from iceberg_tracking_code_b200 import synthetic as syn
    from iceberg_tracking_code_b200.tracking import SequenceTracker
    track_len = 3
    base = syn.base_texture(300, 420, 31)
    rgb = [syn.frame_rgb(base, t, seed=31).numpy() for t in range(track_len + 1)]
    gp = dict(maxCorners=1200, qualityLevel=0.005, minDistance=6, blockSize=5)
    lp = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    trk = SequenceTracker(gp, lp)
    pyr = [trk.prepare(f) for f in rgb]
    n = trk.seed(pyr[0], None, track_len)
    assert n > 500
    corners = trk._tracks[0].cpu().numpy().reshape(-1, 1, 2).copy()
    for t in range(track_len):
        trk.track(pyr[t], pyr[t + 1])
    tracks, quality = trk.harvest()
    same_seed = types.SimpleNamespace(cvtColor=oracle.cvtColor, calcOpticalFlowPyrLK=oracle.calcOpticalFlowPyrLK,
                                      goodFeaturesToTrack=lambda *a, **k: corners)
    ref_t, ref_q = s1_loop_oracle(same_seed, rgb, None, track_len, gp, lp)[0]
    assert ref_q.dtype == np.float32 and quality.dtype == np.float32
    assert tracks.shape == ref_t.shape and tracks.tobytes() == ref_t.tobytes()
    assert quality.shape == ref_q.shape and quality.tobytes() == ref_q.tobytes()
    assert 0 < len(tracks) < n                                          # the FB test pruned some tracks


# ---- projection ----------------------------------------------------------------------------------------------------------
def test_photo_to_utm_past_one_grid_pass(ibt, oracle, golden):
    """n = 1 000 003 vertices: more than one pass of the grid-stride loop (148 x 8 blocks of 256), the golden vertices and
    vertices outside the frame (negative, beyond the sensor, toward the horizon)"""
    g = golden("utm_expected.npz")
    rng = np.random.default_rng(17)
    n = 1_000_003
    out = np.array([[-500.0, -300.0], [7000.0, 5000.0], [-1e4, 2e4], [3e5, -3e5], [0.0, -4000.0], [2999.5, -1e6]], np.float32)
    xy = np.concatenate([g["xy"].reshape(-1, 2).astype(np.float32), out])
    xy = np.concatenate([xy, (rng.random((n - len(xy), 2)) * [6400, 4400] - [200, 200]).astype(np.float32)])
    assert len(xy) == n > 148 * 8 * 256
    got = ibt.photo_to_utm(xy, g["cam"])
    want = oracle.photo_to_utm(xy, g["cam"])
    bad = np.flatnonzero((got != want).any(1))
    assert not len(bad), "%d vertices differ, e.g. #%d %r: %r vs %r" % (len(bad), bad[0], xy[bad[0]], got[bad[0]], want[bad[0]])


# ---- track_velocities against oracle.track_velocities ---------------------------------------------------------------------
def _tracks(rng, M, T):
    """(M, T+1, 2) float32 image tracks: drifts with noise, fast ones, reversals, motionless segments, motionless x"""
    p0 = rng.random((M, 1, 2)) * [5200, 1700] + [100, 1500]
    step = rng.normal(0, 1.0, (M, 1, 2)) + rng.normal(0, 0.4, (M, T, 2))
    step[::9] *= 10.0
    step[4::11] *= -1.0
    step[5::13] = 0.0
    step[6::17, :, 0] = 0.0
    step[7::19, ::3] = 0.0
    return np.concatenate([p0, p0 + np.cumsum(step, 1)], 1).astype(np.float32)


def _run(ibt, oracle, cam, tr, **thr):
    from iceberg_tracking_code_b200.utm import track_velocities
    args = (cam, INTERVAL, thr["min_speed"], thr["max_speed"], thr["max_speedfactor"], thr["max_angle"], thr["speed_threshold"])
    r = track_velocities(tr, *args)
    got = {k: v.cpu().numpy() for k, v in r.items()}
    EN, uv, sp, keep = oracle.track_velocities(tr, *args)
    return got, dict(EN=EN, uv=uv, speed=sp, keep=keep)


def _assert_same(got, ref, what):
    for k in ("EN", "uv", "speed"):
        g, r = got[k], ref[k]
        assert g.shape == r.shape, (what, k)
        bad = np.flatnonzero(~((g == r) | (np.isnan(g) & np.isnan(r))).reshape(len(g), -1).all(1))
        assert not len(bad), "%s: %s differs on %d tracks, e.g. track %d: %r vs %r" % (
            what, k, len(bad), bad[0], g[bad[0]].ravel()[:6], r[bad[0]].ravel()[:6])
    bad = np.flatnonzero(got["keep"] != ref["keep"])
    assert not len(bad), "%s: keep differs on %d tracks, e.g. %s" % (what, len(bad), bad[:6].tolist())


def _ratios_angles(uv, sp):
    """per track: Python max() of the speed ratios and of the angles, with the oracle's own expressions (s2:324-333)"""
    rmax, amax = [], []
    with np.errstate(all="ignore"):
        for u, s in zip(uv, sp):
            rat, ang = [], []
            for c1 in range(len(s) - 1):
                c2 = c1 + 1
                dot = u[c1, 0] * u[c2, 0] + u[c1, 1] * u[c2, 1]
                mag1, mag2 = np.hypot(u[c1, 0], u[c1, 1]), np.hypot(u[c2, 0], u[c2, 1])
                ang.append(abs(np.degrees(np.arccos(dot / (mag1 * mag2)))))
                rat.append(max([s[c1], s[c2]]) / min([s[c1], s[c2]]))
            rmax.append(max(rat) if rat else np.nan)
            amax.append(max(ang) if ang else np.nan)
    return np.array(rmax), np.array(amax)


def _angle_guard(amax, max_angle, what):
    near = np.abs(amax - max_angle) <= 1e-12 * abs(max_angle)
    assert not near.any(), "%s: max angle of tracks %s within 1e-12 of max_angle (acos ulps decide)" % (what, np.flatnonzero(near))


@pytest.mark.parametrize("T", SWEEP_T)
def test_track_velocities_exact(ibt, oracle, golden, T):
    """EN, uv, speed bit for bit and keep on every track, at T on each side of np_sum's 8-accumulator (T >= 8) and
    recursive-halving (T > 128) bounds"""
    cam = golden("utm_expected.npz")["cam"]
    M = 256 if T < 100 else 48
    tr = _tracks(np.random.default_rng(1000 + T), M, T)
    thr = dict(zip(("min_speed", "max_speed", "max_speedfactor", "max_angle", "speed_threshold"), CRITERIA))
    got, ref = _run(ibt, oracle, cam, tr, **thr)
    _angle_guard(_ratios_angles(ref["uv"], ref["speed"])[1], thr["max_angle"], "T %d" % T)
    _assert_same(got, ref, "T %d" % T)
    if T >= 2 and M == 256:
        assert 0.05 < ref["keep"].mean() < 0.98, ref["keep"].mean()     # the criteria fire on this input


def test_track_velocities_many_tracks(ibt, oracle, golden):
    cam = golden("utm_expected.npz")["cam"]
    tr = _tracks(np.random.default_rng(5), 100_000, 2)
    thr = dict(zip(("min_speed", "max_speed", "max_speedfactor", "max_angle", "speed_threshold"), CRITERIA))
    got, ref = _run(ibt, oracle, cam, tr, **thr)
    _angle_guard(_ratios_angles(ref["uv"], ref["speed"])[1], thr["max_angle"], "M 100000")
    _assert_same(got, ref, "M 100000")


def _knife(ibt, oracle, cam, tr, m, on, off, what):
    """on: thresholds at which track m is kept, off: the same with one threshold moved by one step; both runs equal the
    oracle's on every track, and the oracle's keep of track m flips between them"""
    g_on, r_on = _run(ibt, oracle, cam, tr, **on)
    g_off, r_off = _run(ibt, oracle, cam, tr, **off)
    assert r_on["keep"][m] and not r_off["keep"][m], "%s: track %d does not sit on the threshold" % (what, m)
    _assert_same(g_on, r_on, what + " (kept)")
    _assert_same(g_off, r_off, what + " (dropped)")


@pytest.mark.parametrize("T", SWEEP_T)
def test_min_speed_knife_edge(ibt, oracle, golden, T):
    """min_speed = np.mean of track m's speeds: kept; the next float64 up: dropped.  Pins numpy's pairwise summation order."""
    cam = golden("utm_expected.npz")["cam"]
    M = 64 if T < 100 else 16
    tr = _tracks(np.random.default_rng(2000 + T), M, T)
    _, ref = _run(ibt, oracle, cam, tr, **NEVER)
    means = np.array([np.mean(list(s)) for s in ref["speed"]])
    for m in np.flatnonzero(np.isfinite(means) & (means > 0))[:3]:
        mean = means[m]
        _knife(ibt, oracle, cam, tr, m, dict(NEVER, min_speed=mean), dict(NEVER, min_speed=np.nextafter(mean, np.inf)),
               "T %d min_speed track %d" % (T, m))


@pytest.mark.parametrize("T", [1, 2, 9, 129, 300])
def test_speed_threshold_knife_edges(ibt, oracle, golden, T):
    """max_speed = max of track m's speeds: kept, one step down: dropped.  speed_threshold = that max with max_speedfactor 1:
    criteria 2 and 3 are skipped and m is kept, one step down: they run and drop it.  max_speedfactor = m's max ratio: kept,
    one step down: dropped.  max_angle = m's max angle x (1 + 1e-12): kept, x (1 - 1e-12): dropped."""
    cam = golden("utm_expected.npz")["cam"]
    M = 64 if T < 100 else 16
    tr = _tracks(np.random.default_rng(3000 + T), M, T)
    _, ref = _run(ibt, oracle, cam, tr, **NEVER)
    sp = ref["speed"]
    smax = np.array([max(list(s)) for s in sp])
    rmax, amax = _ratios_angles(ref["uv"], sp)
    ok = np.isfinite(smax) & (smax > 0)
    down = lambda v: np.nextafter(v, -np.inf)
    m = int(np.flatnonzero(ok)[0])
    _knife(ibt, oracle, cam, tr, m, dict(NEVER, max_speed=smax[m]), dict(NEVER, max_speed=down(smax[m])),
           "T %d max_speed" % T)
    if T < 2:
        return
    m = int(np.flatnonzero(ok & (rmax > 1))[0])
    _knife(ibt, oracle, cam, tr, m, dict(NEVER, speed_threshold=smax[m], max_speedfactor=1.0),
           dict(NEVER, speed_threshold=down(smax[m]), max_speedfactor=1.0), "T %d speed_threshold" % T)
    crit = dict(NEVER, speed_threshold=-np.inf)
    m = int(np.flatnonzero(ok & np.isfinite(rmax) & (rmax > 1))[0])
    _knife(ibt, oracle, cam, tr, m, dict(crit, max_speedfactor=rmax[m]), dict(crit, max_speedfactor=down(rmax[m])),
           "T %d max_speedfactor" % T)
    m = int(np.flatnonzero(ok & np.isfinite(amax) & (amax > 1))[0])
    others = np.delete(amax, m)
    for f in (1 + 1e-12, 1 - 1e-12):
        _angle_guard(others, amax[m] * f, "T %d max_angle" % T)
    _knife(ibt, oracle, cam, tr, m, dict(crit, max_angle=amax[m] * (1 + 1e-12)), dict(crit, max_angle=amax[m] * (1 - 1e-12)),
           "T %d max_angle" % T)


def test_python_max_nan_quirks(ibt, oracle, golden):
    """Motionless segments make 0/0 speed ratios and angles (NaN) and s/0 ratios (inf); the reference takes Python's max()
    of the lists, which keeps whichever comes first when a NaN is compared.  Crafted tracks, T = 4, speed_threshold 0."""
    cam = golden("utm_expected.npz")["cam"]
    p, d = np.array([2500.0, 2600.0]), np.array([3.0, 2.0])
    rows = [
        [p, p, p, p + d, p],                  # ratios [nan, inf, ~1], angles [nan, nan, 180]: the leading NaN stays the max
        [p, p + d, p, p, p],                  # speeds [s, s, 0, 0]: ratios [~1, inf, nan], angles [180, nan, nan]
        [p, p + d, p + d, p + d, p + 2 * d],  # speeds [s, 0, 0, s]: ratios [inf, nan, inf], angles [nan, nan, nan]
        [p, p + d, p + 2 * d, p + 2 * d, p + 2 * d],   # speeds [s, s, 0, 0], angles [~0 or nan, nan, nan]
    ]
    tr = np.array(rows, np.float32)
    base = dict(min_speed=0.0, max_speed=np.inf, max_angle=60.0, speed_threshold=0.0)
    expect = {2.5: [True, False, False, False], np.inf: [True, False, True, True]}
    for factor, want in expect.items():
        got, ref = _run(ibt, oracle, cam, tr, max_speedfactor=factor, **base)
        _assert_same(got, ref, "crafted, max_speedfactor %g" % factor)
        assert ref["keep"].tolist() == want, (factor, ref["keep"].tolist())
    # T = 1 above speed_threshold: kept (the reference raises on max() of the empty ratio list; documented in utm.cu)
    one = np.array([[p, p + d]], np.float32)
    got, ref = _run(ibt, oracle, cam, one, min_speed=0.0, max_speed=np.inf, max_speedfactor=1.0, max_angle=0.0,
                    speed_threshold=0.0)
    assert got["speed"][0, 0] > 0 and got["keep"].tolist() == [True]
    _assert_same(got, ref, "T 1")
