"""Parity comparators implementing BASELINE.json's criteria (shared by the CPU and GPU tests)."""
import numpy as np

GFTT_SETS = [
    dict(maxCorners=50000000, qualityLevel=0.007, minDistance=10, blockSize=10),
    dict(maxCorners=2000, qualityLevel=0.01, minDistance=7, blockSize=3),
    dict(maxCorners=0, qualityLevel=0.007, minDistance=10, blockSize=10),
    dict(maxCorners=500, qualityLevel=0.05, minDistance=0, blockSize=3),
    dict(maxCorners=300, qualityLevel=0.007, minDistance=10.5, blockSize=10),
    dict(maxCorners=120, qualityLevel=0.02, minDistance=25, blockSize=5),
]
LK_SETS = [
    dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01)),
    dict(winSize=(31, 31), maxLevel=4, criteria=(3, 30, 0.01)),
    dict(winSize=(35, 35), maxLevel=4, criteria=(3, 25, 0.03)),
    dict(winSize=(15, 9), maxLevel=2, criteria=(1, 7, 0.0)),
    dict(winSize=(41, 41), maxLevel=5, criteria=(2, 0, 0.05)),
]

POS_TOL_PX = 0.01          # BASELINE.json: positions within 0.01 px for >= 99 % of both-valid points
POS_FRAC = 0.99
STATUS_FRAC = 0.995        # status flags agree on >= 99.5 % of points
CORNER_OVERLAP = 0.99      # Shi-Tomasi corner set overlap >= 99 %
ERR_TOL = 2e-3             # err (mean |J-I| / 32): float accumulation-order differences only


def lk_agreement(p_a, st_a, p_b, st_b):
    """-> (status agreement fraction, fraction of both-valid points within POS_TOL_PX, max abs diff on both-valid)."""
    p_a, p_b = np.asarray(p_a, np.float32).reshape(-1, 2), np.asarray(p_b, np.float32).reshape(-1, 2)
    st_a, st_b = np.asarray(st_a).reshape(-1), np.asarray(st_b).reshape(-1)
    agree = float(np.mean(st_a == st_b))
    both = (st_a == 1) & (st_b == 1)
    if not both.any():
        return agree, 1.0, 0.0
    d = np.abs(p_a[both] - p_b[both]).max(axis=1)
    return agree, float(np.mean(d <= POS_TOL_PX)), float(d.max())


def assert_lk_parity(p_a, st_a, p_b, st_b, what=""):
    agree, frac, mx = lk_agreement(p_a, st_a, p_b, st_b)
    assert agree >= STATUS_FRAC, "%s: status agreement %.4f < %.3f" % (what, agree, STATUS_FRAC)
    assert frac >= POS_FRAC, "%s: only %.4f of both-valid points within %.3f px (max %.4g)" % (what, frac, POS_TOL_PX, mx)
    return agree, frac, mx


def _f32_same(a, b):
    """element-wise: same float32 bytes, or NaN on both sides (the GPU returns the canonical NaN, x86 keeps the payload)"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def _lk_n(ref):
    return np.asarray(ref["st"]).size if "st" in ref else np.asarray(ref["p1"]).size // 2


def lk_exact_mismatch(gpu, ref):
    """gpu / ref: dicts with any of p1 (N,2) f32, st (N,) u8, err (N,) f32, iters (N,) or per level (N, L) int.  -> bool (N,),
    True where the two differ in any of the keys both hold.  The CUDA solver and the oracle sum the same exact integers and
    round the same float steps, so there is no tolerance: p1 and err by bytes, status and the iteration counts equal."""
    n = _lk_n(ref)
    bad = np.zeros(n, bool)
    for k in ("p1", "st", "err", "iters"):
        if k not in gpu or k not in ref:
            continue
        g, r = np.asarray(gpu[k]), np.asarray(ref[k])
        if k == "p1":
            bad |= ~_f32_same(g.reshape(n, 2), r.reshape(n, 2)).all(1)
        elif k == "err":
            bad |= ~_f32_same(g.reshape(n), r.reshape(n))
        elif k == "iters":
            bad |= g.reshape(n, -1).sum(1) != r.reshape(n, -1).sum(1)
        else:
            bad |= g.reshape(n) != r.reshape(n)
    return bad


def assert_lk_exact(gpu, ref, what="", pts=None, guess=None, show=6):
    """Exact agreement of a CUDA LK result with the oracle's (lk_exact_mismatch).  A failure lists the first `show`
    mismatching points with their input, initial guess and both sides' outputs; `what` names the case (sizes, parameters)."""
    bad = np.flatnonzero(lk_exact_mismatch(gpu, ref))
    if not len(bad):
        return
    lines = []
    for i in bad[:show]:
        s = "  #%d" % i
        if pts is not None:
            s += " pt %r" % (np.asarray(pts, np.float32).reshape(-1, 2)[i].tolist(),)
        if guess is not None:
            s += " guess %r" % (np.asarray(guess, np.float32).reshape(-1, 2)[i].tolist(),)
        for k in ("p1", "st", "err", "iters"):
            if k in gpu and k in ref:
                r = np.asarray(ref[k])
                g, r = np.asarray(gpu[k]).reshape(r.shape[0], -1)[i], r.reshape(r.shape[0], -1)[i]
                if k == "iters":
                    g, r = g.sum(), r.sum()
                s += " | %s gpu %r oracle %r" % (k, np.asarray(g).tolist(), np.asarray(r).tolist())
        lines.append(s)
    n = _lk_n(ref)
    raise AssertionError("%s: %d of %d points differ from the oracle\n%s" % (what, len(bad), n, "\n".join(lines)))


def corner_overlap(a, b):
    """|A n B| / max(|A|, |B|) over integer (x, y) corner sets; None counts as empty."""
    sa = set() if a is None else set(map(tuple, np.asarray(a).reshape(-1, 2).astype(np.int64).tolist()))
    sb = set() if b is None else set(map(tuple, np.asarray(b).reshape(-1, 2).astype(np.int64).tolist()))
    if not sa and not sb:
        return 1.0
    return len(sa & sb) / max(len(sa), len(sb))


def as_corners(p):
    return np.zeros((0, 1, 2), np.float32) if p is None else np.asarray(p, np.float32)
