"""Without a GPU: the multi-channel pyramid and forward-backward entry points reject invalid arguments before any CUDA call,
cv.py raises cv.error for bad colour inputs, and cv2's colour pyramid is its per-channel gray pyramids (the rule the CUDA
path and the oracle route of tests/test_gpu_multichannel_pyramid.py rely on)."""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def N():
    from iceberg_tracking_code_b200 import build
    build.build()
    from iceberg_tracking_code_b200 import _native
    return _native


def _pyr(N, h, w, levels, derivs=True):
    """a well-formed pyramid description at fake (never dereferenced) device addresses"""
    st = N.ibt_pyramid_t()
    st.nlevels = levels
    for l in range(levels):
        st.rows[l], st.cols[l] = h, w
        st.img[l], st.img_pitch[l] = 0x10000000 * (l + 1), (w + 127) // 128 * 128
        if derivs:
            st.deriv[l], st.deriv_pitch[l] = 0x20000000 * (l + 1), (4 * w + 127) // 128 * 128
        h, w = (h + 1) // 2, (w + 1) // 2
    return st


def _arr(N, structs):
    PP = C.POINTER(N.ibt_pyramid_t)
    return (PP * len(structs))(*[C.pointer(s) if s is not None else PP() for s in structs])


def test_version(N):
    assert N.lib().ibt_version() >= 103


def test_pyramid_build_multichannel_rejects(N):
    lib, inv = N.lib(), N.IBT_E_INVALID
    frame, H, W = C.c_void_p(0x30000000), 64, 96
    ok = [_pyr(N, H, W, 3) for _ in range(4)]
    build = lambda f, pitch, cn, arr, d=1: lib.ibt_pyramid_build_multichannel(f, pitch, cn, arr, d, None)
    for cn in (1, 5, 0, -1):
        assert build(frame, W * 4, cn, _arr(N, ok)) == inv, cn
    assert build(None, W * 3, 3, _arr(N, ok)) == inv                          # null frame
    assert build(frame, W * 3, 3, None) == inv                                # null pyramid array
    assert build(frame, W * 3, 3, _arr(N, ok[:2] + [None])) == inv            # null channel pyramid
    assert build(frame, W * 3 - 1, 3, _arr(N, ok)) == inv                     # frame pitch < W * cn
    other = _pyr(N, H, W + 2, 3)
    assert build(frame, W * 3, 3, _arr(N, [ok[0], other, ok[2]])) == inv      # channel geometry differs
    shallow = _pyr(N, H, W, 2)
    assert build(frame, W * 3, 3, _arr(N, [ok[0], ok[1], shallow])) == inv    # level count differs
    bad = _pyr(N, H, W, 3)
    bad.rows[1] = 31                                                          # level 1 is not level 0 halved
    assert build(frame, W * 3, 3, _arr(N, [bad] * 3)) == inv
    bad = _pyr(N, H, W, 3)
    bad.deriv_pitch[0] = 4 * W - 4                                            # derivative pitch below 4 w
    assert build(frame, W * 3, 3, _arr(N, [ok[0], ok[1], bad])) == inv
    bad = _pyr(N, H, W, 3)
    bad.deriv_pitch[1] = 4 * 48 + 2                                           # derivative pitch not a multiple of 4
    assert build(frame, W * 3, 3, _arr(N, [bad] * 3)) == inv
    bad = _pyr(N, H, W, 3)
    bad.img[0] = None                                                         # level 0 is an output: it must exist
    assert build(frame, W * 3, 3, _arr(N, [ok[0], bad, ok[2]])) == inv
    nod = _pyr(N, H, W, 3, derivs=False)
    assert build(frame, W * 3, 3, _arr(N, [nod] * 3), 1) == inv               # derivatives asked, no planes
    bad = _pyr(N, H, W, 3)
    bad.img_pitch[2] = 10                                                     # level pitch < width
    assert build(frame, W * 3, 3, _arr(N, [bad] * 3)) == inv


def test_lk_fb_multichannel_rejects(N):
    lib, inv = N.lib(), N.IBT_E_INVALID
    H, W, n = 64, 96, 5
    pts, out = C.c_void_p(0x40000000), C.c_void_p(0x50000000)
    ok = [_pyr(N, H, W, 3) for _ in range(4)]

    def fb(prev, nxt, cn, win=21, p0=pts, p1=out):
        return lib.ibt_lk_fb_multichannel(prev, nxt, cn, p0, n, win, win, 30, 0.01, 1e-4, 1.0, p1, None, None, None, None,
                                          None, None, None, None, None, None)
    for cn in (1, 5):
        assert fb(_arr(N, ok), _arr(N, ok), cn) == inv, cn
    assert fb(None, _arr(N, ok), 3) == inv and fb(_arr(N, ok), None, 3) == inv
    assert fb(_arr(N, ok[:2] + [None]), _arr(N, ok), 3) == inv
    assert fb(_arr(N, ok), _arr(N, ok), 3, p0=None) == inv and fb(_arr(N, ok), _arr(N, ok), 3, p1=None) == inv
    assert fb(_arr(N, ok), _arr(N, ok), 3, win=2) == inv
    other = _pyr(N, H, W + 2, 3)
    assert fb(_arr(N, ok), _arr(N, [ok[0], ok[1], other]), 3) == inv         # channel geometry differs
    nod = _pyr(N, H, W, 3, derivs=False)
    assert fb(_arr(N, ok), _arr(N, [nod] * 3), 3) == inv                      # next without Scharr planes: no backward pass
    bad = _pyr(N, H, W, 3)
    bad.deriv_pitch[0] = 4 * W + 2
    assert fb(_arr(N, [bad] * 3), _arr(N, ok), 3) == inv                      # bad derivative pitch


def test_colour_inputs_raise_cv_error(N):
    from iceberg_tracking_code_b200 import cv
    rng = np.random.default_rng(0)
    pts = np.zeros((4, 2), np.float32)
    for shape in [(20, 30, 5), (20, 30, 6)]:
        f = rng.integers(0, 256, shape, dtype=np.uint8)
        with pytest.raises(cv.error):
            cv.FramePyramid(f)
        with pytest.raises(cv.error):
            cv.buildOpticalFlowPyramid(f, (21, 21), 3)
        with pytest.raises(cv.error):
            cv.calcOpticalFlowPyrLK(f, f, pts)
    f3 = np.zeros((20, 30, 3), np.float32)
    with pytest.raises(cv.error):
        cv.FramePyramid(f3)
    with pytest.raises(cv.error):
        cv.calcOpticalFlowPyrLK(np.zeros((20, 30, 3), np.uint8), np.zeros((20, 30, 4), np.uint8), pts)


def test_cv2_colour_pyramid_is_per_channel_gray():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(13)
    for cn in (2, 3, 4):
        for h, w, win, ml in [(1, 17, (3, 3), 2), (2, 9, (3, 3), 3), (65, 129, (5, 5), 4), (240, 321, (21, 21), 3)]:
            f = rng.integers(0, 256, (h, w, cn), dtype=np.uint8)
            for derivs in (True, False):
                ml_c, pc = cv2.buildOpticalFlowPyramid(f, win, ml, withDerivatives=derivs)
                k = 2 if derivs else 1
                for c in range(cn):
                    ml_g, pg = cv2.buildOpticalFlowPyramid(np.ascontiguousarray(f[..., c]), win, ml, withDerivatives=derivs)
                    assert ml_g == ml_c
                    for l in range(ml_c + 1):
                        assert np.array_equal(pc[k * l][..., c], pg[k * l]), (cn, h, w, c, l)
                        if derivs:
                            assert np.array_equal(pc[k * l + 1][..., 2 * c:2 * c + 2], pg[k * l + 1]), (cn, h, w, c, l)
