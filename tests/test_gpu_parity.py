"""GPU parity: the CUDA path, called through the C-ABI (cv.py -> libibt.so), against the cv2 golden vectors and the
CPU oracle on the same seeded inputs.  Bit-exact for integer work; BASELINE.json tolerances for LK / GFTT."""
import numpy as np
import pytest
import torch

from parity import (GFTT_SETS, LK_SETS, ERR_TOL, CORNER_OVERLAP, _f32_same, assert_lk_exact, assert_lk_parity, as_corners,
                    corner_overlap)

pytestmark = pytest.mark.gpu
SCENES = ["kat_texture.npz", "kat_iceberg.npz"]


@pytest.mark.parametrize("scene", SCENES)
def test_gray_bit_exact(ibt, golden, scene):
    g = golden(scene)
    assert np.array_equal(ibt.cvtColor(g["rgb"], ibt.COLOR_BGR2GRAY), g["gray"])
    rgba = np.dstack([g["rgb"], g["rgb"][..., 0]])
    assert np.array_equal(ibt.cvtColor(rgba, ibt.COLOR_BGR2GRAY), g["gray4"])
    with pytest.raises(ibt.error):
        ibt.cvtColor(g["f0"], ibt.COLOR_BGR2GRAY)           # 2-D input: "Bad number of channels"


def test_gray_sizes_vs_oracle(ibt, oracle):
    rng = np.random.default_rng(0)
    for (h, w) in [(1, 1), (3, 17), (64, 48), (37, 1029), (1080, 1920)]:
        rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        for cs in (0, 1):
            assert np.array_equal(ibt.cvtColor(rgb, ibt.COLOR_BGR2GRAY, coeffset=cs), oracle.cvtColor(rgb, coeffset=cs)), (h, w, cs)


@pytest.mark.parametrize("scene", SCENES)
def test_pyramid_bit_exact_golden(ibt, golden, scene):
    g = golden(scene)
    assert np.array_equal(ibt.pyrDown(g["f0"]), g["pyrdown"])
    for si, win in enumerate([(21, 21), (35, 35)]):
        ml, pyr = ibt.buildOpticalFlowPyramid(g["f0"], win, 4, True)
        assert ml == int(g["pyr%d_maxlevel" % si])
        for l in range(ml + 1):
            assert np.array_equal(pyr[2 * l], g["pyr%d_L%d" % (si, l)]), (si, l)
            assert np.array_equal(pyr[2 * l + 1], g["pyr%d_D%d" % (si, l)]), (si, l)


def test_pyramid_edge_cases(ibt, golden):
    g = golden("kat_edge.npz")
    for k in g:
        if k.startswith("rnd_"):
            shp = k[4:]
            a = g[k]
            assert np.array_equal(ibt.pyrDown(a), g["pyrdown_" + shp]), shp
            if "scharr_" + shp in g:
                ml, pyr = ibt.buildOpticalFlowPyramid(a, (3, 3), 0, True)
                assert np.array_equal(pyr[1], g["scharr_" + shp]), shp
        if k.startswith("levels_"):
            h, w = [int(v) for v in k.split("_")[1].split("x")]
            win = int(k.split("_w")[1])
            a = np.zeros((h, w), np.uint8)
            ml, pyr = ibt.buildOpticalFlowPyramid(a, (win, win), 4, False)
            assert [ml] + [x for p in pyr for x in p.shape[:2]] == g[k].tolist(), k


@pytest.mark.parametrize("hw", [(1080, 1920), (1001, 1333), (4000, 6000)])
def test_pyramid_bit_exact_large_vs_oracle(ibt, oracle, hw):
    rng = np.random.default_rng(hw[0])
    a = rng.integers(0, 256, hw, dtype=np.uint8)
    ml, pyr = ibt.buildOpticalFlowPyramid(a, (31, 31), 4, True)
    ml_o, pyr_o = oracle.buildOpticalFlowPyramid(a, (31, 31), 4, True)
    assert ml == ml_o
    for i, (x, y) in enumerate(zip(pyr, pyr_o)):
        assert x.shape == y.shape and np.array_equal(x, y), i


@pytest.mark.parametrize("scene", SCENES)
def test_mineig_close(ibt, golden, scene):
    g = golden(scene)
    for bs, tol in ((3, 3e-4), (10, 4e-6)):
        ref = g["mineig_bs%d" % bs]
        got = ibt.cornerMinEigenVal(g["f0"], bs)
        assert np.abs(got - ref).max() <= tol * np.abs(ref).max(), bs


@pytest.mark.parametrize("scene", SCENES)
def test_gftt_golden(ibt, golden, scene):
    g = golden(scene)
    for gi, gp in enumerate(GFTT_SETS):
        for mi, m in enumerate([None, g["mask"]]):
            ref = g["gftt%d_m%d" % (gi, mi)]
            got = as_corners(ibt.goodFeaturesToTrack(g["f0"], mask=m, **gp))
            ov = corner_overlap(got, ref)
            assert ov >= CORNER_OVERLAP, (gi, mi, ov, got.shape, ref.shape)
            if gp["maxCorners"] == 0 or gp["maxCorners"] > len(ref):
                # the eig map is reproducible to ~1e-6 only, so ordered equality is expected but reported softly
                assert got.shape == ref.shape, (gi, mi, got.shape, ref.shape)


def test_gftt_none_conventions(ibt, golden):
    g = golden("kat_edge.npz")
    assert ibt.goodFeaturesToTrack(np.full((40, 50), 77, np.uint8), 100, 0.01, 5) is None
    a = g["emptymask_img"]
    assert ibt.goodFeaturesToTrack(a, 100, 0.01, 5, mask=np.zeros_like(a)) is None


def test_gftt_1080p_vs_oracle(ibt, oracle):
    """BASELINE config 1 seeding: 1920x1080, 2k Shi-Tomasi points."""
    from iceberg_tracking_code_b200 import synthetic as syn
    base = syn.base_texture(1080, 1920, 1)
    f0 = syn.frame_gray(base, 0).numpy()
    for gp in (dict(maxCorners=2000, qualityLevel=0.007, minDistance=10, blockSize=10), GFTT_SETS[0]):
        ref = as_corners(oracle.goodFeaturesToTrack(f0, **gp))
        got = as_corners(ibt.goodFeaturesToTrack(f0, **gp))
        assert corner_overlap(got, ref) >= CORNER_OVERLAP
        assert len(got) == len(ref)
        assert np.mean(np.all(got == ref, axis=(1, 2))) >= 0.99      # same order, too


@pytest.mark.parametrize("scene", SCENES)
def test_lk_golden(ibt, golden, scene):
    g = golden(scene)
    pts = g["lk_pts"]
    for li, lp in enumerate(LK_SETS):
        p1, st, err = ibt.calcOpticalFlowPyrLK(g["f0"], g["f1"], pts, None, **lp)
        assert p1.shape == pts.shape and st.shape == (len(pts), 1) and err.shape == (len(pts), 1)
        assert p1.dtype == np.float32 and st.dtype == np.uint8 and err.dtype == np.float32
        assert_lk_parity(p1, st, g["lk%d_p1" % li], g["lk%d_st" % li], "fwd set %d" % li)
        ok = (st == 1) & (g["lk%d_st" % li] == 1)
        assert np.abs(err - g["lk%d_err" % li])[ok].max(initial=0) <= ERR_TOL
        p0r, st0, err0 = ibt.calcOpticalFlowPyrLK(g["f1"], g["f0"], g["lk%d_p1" % li], None, **lp)
        assert_lk_parity(p0r, st0, g["lk%d_p0r" % li], g["lk%d_st0" % li], "bwd set %d" % li)
        d = np.abs(p1 - g["lk%d_p1" % li]).reshape(-1, 2).max(1)      # failed points: propagated guess (A.7)
        assert np.mean(d <= 0.01) >= 0.99, li


def test_lk_flags_and_conventions(ibt, golden):
    g = golden("kat_texture.npz")
    pts = g["lk_pts"]
    p1, st, _ = ibt.calcOpticalFlowPyrLK(g["f0"], g["f1"], pts, g["lkinit_guess"], flags=ibt.OPTFLOW_USE_INITIAL_FLOW,
                                         **LK_SETS[0])
    assert_lk_parity(p1, st, g["lkinit_p1"], g["lkinit_st"], "initial flow")
    p1, st, err = ibt.calcOpticalFlowPyrLK(g["f0"], g["f1"], pts, None, flags=ibt.OPTFLOW_LK_GET_MIN_EIGENVALS,
                                           **LK_SETS[0])
    assert_lk_parity(p1, st, g["lkeig_p1"], g["lkeig_st"], "min eigenvals")
    ok = (st == 1) & (g["lkeig_st"] == 1)
    assert np.abs(err - g["lkeig_err"])[ok].max() <= 1e-5 * max(1.0, np.abs(g["lkeig_err"][ok]).max())
    # N == 0 -> (None, None, None); float64 points -> error; (N,2) in -> (N,2) out
    assert ibt.calcOpticalFlowPyrLK(g["f0"], g["f1"], np.zeros((0, 1, 2), np.float32), None) == (None, None, None)
    with pytest.raises(ibt.error):
        ibt.calcOpticalFlowPyrLK(g["f0"], g["f1"], pts.astype(np.float64), None)
    p2, st2, _ = ibt.calcOpticalFlowPyrLK(g["f0"], g["f1"], pts.reshape(-1, 2), None, **LK_SETS[0])
    assert p2.shape == (len(pts), 2) and st2.shape == (len(pts), 1)


def test_lk_fb_fused_equals_two_calls(ibt, golden):
    """One launch (forward + backward + FB check) == the reference's two calls + numpy FB arithmetic (s1:323-333)."""
    g = golden("kat_iceberg.npz")
    pts = g["lk_pts"]
    for lp in LK_SETS[:3]:
        p1, st1, err1 = ibt.calcOpticalFlowPyrLK(g["f0"], g["f1"], pts, None, **lp)
        p0r, st0, err0 = ibt.calcOpticalFlowPyrLK(g["f1"], g["f0"], p1, None, **lp)
        diff = abs(pts - p0r).reshape(-1, 2)
        dist = np.hypot(diff[:, 0], diff[:, 1])
        r = ibt.calcOpticalFlowPyrLK_FB(g["f0"], g["f1"], pts, **lp)
        assert np.array_equal(r["p1"], p1) and np.array_equal(r["p0r"], p0r)
        assert np.array_equal(r["st1"], st1) and np.array_equal(r["st0"], st0)
        assert np.array_equal(r["err1"], err1) and np.array_equal(r["err0"], err0)
        assert _f32_same(r["dist"], dist).all() and np.array_equal(r["valid"], dist < 1)
        # the quirk the reference relies on: FB-valid points with status 0 exist and are kept (SURVEY A.7)
    assert ((r["st1"].reshape(-1) == 0) & r["valid"]).sum() > 0


def test_config1_vs_oracle(ibt, oracle):
    """BASELINE config 1: 1920x1080 pair, 2k Shi-Tomasi points, winSize 21, maxLevel 3."""
    from iceberg_tracking_code_b200 import synthetic as syn
    base = syn.base_texture(1080, 1920, 1)
    f0, f1 = syn.frame_gray(base, 0).numpy(), syn.frame_gray(base, 1).numpy()
    gp = dict(maxCorners=2000, qualityLevel=0.007, minDistance=10, blockSize=10)
    lp = LK_SETS[0]
    pts = ibt.goodFeaturesToTrack(f0, **gp)
    assert pts is not None and len(pts) == 2000
    p1, st, err, it = ibt.calcOpticalFlowPyrLK(f0, f1, pts, None, return_iters=True, **lp)
    p1_o, st_o, err_o, it_o = oracle.calcOpticalFlowPyrLK(f0, f1, pts, None, return_iters=True, **lp)
    # exact, iterations too: the BASELINE unit (feature-pair-iterations) counts the same on every point
    assert_lk_exact(dict(p1=p1, st=st, err=err, iters=it), dict(p1=p1_o, st=st_o, err=err_o, iters=it_o), "config 1 fwd", pts)
    p0r, st0, err0, it0 = ibt.calcOpticalFlowPyrLK(f1, f0, p1, None, return_iters=True, **lp)
    p0r_o, st0_o, err0_o, it0_o = oracle.calcOpticalFlowPyrLK(f1, f0, p1, None, return_iters=True, **lp)
    assert_lk_exact(dict(p1=p0r, st=st0, err=err0, iters=it0), dict(p1=p0r_o, st=st0_o, err=err0_o, iters=it0_o),
                    "config 1 bwd", p1)
    # the synthetic shift is known: tracked displacement == (-VX, -VY) content motion seen from the camera
    d = (p1 - pts).reshape(-1, 2)[st.reshape(-1) == 1]
    assert np.abs(np.median(d, 0) - [-syn.VX, -syn.VY]).max() < 0.05


def test_photo_to_utm(ibt, golden):
    g = golden("utm_expected.npz")
    got = ibt.photo_to_utm(g["xy"], g["cam"])
    assert got.dtype == np.float64 and np.array_equal(got, g["EN"])


def test_device_tensors_stay_on_device(ibt, golden):
    g = golden("kat_texture.npz")
    f0, f1 = torch.from_numpy(g["f0"]).cuda(), torch.from_numpy(g["f1"]).cuda()
    pts = torch.from_numpy(g["lk_pts"]).cuda()
    p1, st, err = ibt.calcOpticalFlowPyrLK(f0, f1, pts, None, **LK_SETS[0])
    assert p1.is_cuda and st.is_cuda and err.is_cuda
    assert_lk_parity(p1.cpu().numpy(), st.cpu().numpy(), g["lk0_p1"], g["lk0_st"], "device tensors")
    # cached pyramids give the same answer as images
    pa = ibt.FramePyramid(f0, LK_SETS[0]["winSize"], LK_SETS[0]["maxLevel"], True)
    pb = ibt.FramePyramid(f1, LK_SETS[0]["winSize"], LK_SETS[0]["maxLevel"], True)
    q1, qs, _ = ibt.calcOpticalFlowPyrLK(pa, pb, pts, None, **LK_SETS[0])
    assert torch.equal(q1, p1) and torch.equal(qs, st)


def test_gftt_prefilter_fallback_and_ties_vs_oracle(ibt, oracle):
    """Two paths of the selection kernel that the texture scenes do not reach, against the CPU oracle:
    (1) the top-k prefilter ranks only the strongest ~4*maxCorners candidates, all of them lie in one bright patch, min-distance
        culling leaves fewer than maxCorners of them -> the kernel must start over with every candidate;
    (2) a periodic image: many candidates with EXACTLY equal responses -> OpenCV's tie-break (higher address first) decides."""
    rng = np.random.default_rng(12)
    h, w = 700, 900
    weak = (rng.integers(0, 256, (h, w)).astype(np.float32) - 128) * 0.08 + 128
    img = weak.copy()
    img[150:550, 200:600] = rng.integers(0, 256, (400, 400))          # the strongest corners by far
    img = np.clip(img, 0, 255).astype(np.uint8)
    gp = dict(maxCorners=300, qualityLevel=0.0005, minDistance=30, blockSize=3)
    got = as_corners(ibt.goodFeaturesToTrack(img, **gp))
    ref = as_corners(oracle.goodFeaturesToTrack(img, **gp))
    assert got.shape == ref.shape and got.shape[0] == 300
    assert np.mean(np.all(got == ref, axis=(1, 2))) >= 0.99
    # more than the patch can hold at this distance: the prefix must have come from the full candidate set
    inside = (got[:, 0, 0] >= 200) & (got[:, 0, 0] < 600) & (got[:, 0, 1] >= 150) & (got[:, 0, 1] < 550)
    assert inside.sum() < 300 and (~inside).sum() > 0
    block = rng.integers(0, 256, (16, 16)).astype(np.uint8)
    per = np.tile(block, (16, 20))                                    # 256 x 320, exact period 16: exact response ties
    for gp in (dict(maxCorners=0, qualityLevel=0.01, minDistance=3, blockSize=3),
               dict(maxCorners=150, qualityLevel=0.01, minDistance=9, blockSize=5)):
        got = as_corners(ibt.goodFeaturesToTrack(per, **gp))
        ref = as_corners(oracle.goodFeaturesToTrack(per, **gp))
        assert got.shape == ref.shape and len(ref) > 50
        assert np.array_equal(got, ref), gp                            # order included: ties resolved like OpenCV


def test_harris_branch_golden(ibt, golden):
    """goodFeaturesToTrack(useHarrisDetector=True) / cornerHarris through the C-ABI vs cv2's recorded answers"""
    import harris_cases as HC
    HC.check_harris_golden(ibt, golden("kat_harris.npz"),
                           {"texture": golden("kat_texture.npz"), "iceberg": golden("kat_iceberg.npz")})


def test_multichannel_lk_golden(ibt, golden):
    """calcOpticalFlowPyrLK on 3- / 4-channel frames through the C-ABI (ibt_lk_multichannel) vs cv2's recorded answers"""
    import multichannel_cases as MC
    MC.check_multichannel_golden(ibt, golden("kat_multichannel.npz"))


@pytest.mark.parametrize("win", [(21, 21), (9, 15)])
def test_lk_multichannel_one_plane_equals_gray(ibt, win):
    """ibt_lk_multichannel with one channel plane runs the runtime-cn kernel (cp.async staging); ibt_lk runs the gray kernel
    (window-specialised at 21 x 21, TMA staging).  Both are the one solver body: on the same pyramids p1, status, err and
    iters agree bit for bit, for points inside, near and beyond the border, with and without the two flags."""
    import ctypes as C
    from iceberg_tracking_code_b200 import _native as N, synthetic as syn
    h, w = 1080, 1920
    base = syn.base_texture(h, w, 7)
    pa = ibt.FramePyramid(syn.frame_gray(base, 0).cuda(), win, 3, True)
    pb = ibt.FramePyramid(syn.frame_gray(base, 1).cuda(), win, 3, False)
    rng = np.random.default_rng(7)
    inside = rng.uniform([40, 40], [w - 40, h - 40], (3000, 2))
    near = np.concatenate([rng.uniform([-2, 0], [12, h], (300, 2)), rng.uniform([0, h - 12], [w, h + 2], (300, 2))])
    beyond = np.concatenate([rng.uniform([-60, 0], [-15, h], (100, 2)), rng.uniform([0, h + 15], [w, h + 60], (100, 2))])
    pts = torch.from_numpy(np.concatenate([inside, near, beyond]).astype(np.float32)).cuda()
    guess = pts + torch.from_numpy(rng.normal(0, 1.5, tuple(pts.shape)).astype(np.float32)).cuda()
    n = pts.shape[0]
    one = C.POINTER(N.ibt_pyramid_t) * 1
    for flags in (0, ibt.OPTFLOW_USE_INITIAL_FLOW, ibt.OPTFLOW_LK_GET_MIN_EIGENVALS,
                  ibt.OPTFLOW_USE_INITIAL_FLOW | ibt.OPTFLOW_LK_GET_MIN_EIGENVALS):
        res = []
        for mc in (False, True):
            p1 = guess.clone()
            st = torch.empty(n, dtype=torch.uint8, device="cuda")
            err = torch.empty(n, dtype=torch.float32, device="cuda")
            it = torch.empty(n, dtype=torch.int32, device="cuda")
            tail = (ibt._ptr(pts), ibt._ptr(p1), n, win[0], win[1], 30, 0.01, 1e-4, flags, ibt._ptr(st), ibt._ptr(err),
                    ibt._ptr(it), ibt._stream())
            if mc:
                rc = N.lib().ibt_lk_multichannel(one(C.pointer(pa.c)), one(C.pointer(pb.c)), 1, *tail)
            else:
                rc = N.lib().ibt_lk(C.byref(pa.c), C.byref(pb.c), *tail)
            assert rc == N.IBT_OK
            res.append([t.cpu().numpy() for t in (p1, st, err, it)])
        for name, g, m in zip(("p1", "status", "err", "iters"), *res):
            assert np.array_equal(g, m), (win, flags, name, int((g != m).sum()))
        st = res[0][1]
        assert 0 < st.sum() < n, (win, flags)        # both outcomes occur: the border cases are exercised
