"""GPU tests of the frame loop behind the reference's worker signatures: LucasKanade.run() against the recorded run of
the UNMODIFIED reference class (tests/golden/seq_expected.npz), lucaskanade_tracking / track_sequence against a
restatement of s1:301-395 on the CPU oracle, .npz layout, sharded == unsharded, compaction, mask, config-2 properties."""
import os
import shutil

import numpy as np
import pytest
import torch

from parity import CORNER_OVERLAP, _f32_same, assert_lk_exact, corner_overlap

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEQ = os.path.join(ROOT, "tests", "golden", "seq")


def s1_loop_oracle(orc, frames_rgb, mask, track_len, feature_params, lk_params):
    """Restatement of s1_lucaskanade_tracking.py:301-359, 362, 437-450 with Python lists, on the CPU oracle.
    Returns {seed_counter: (tracks (M,T+1,2) f32, trackquality (M,T) f32)} for every completed group."""
    tracks, trackquality, out = [], [], {}
    prev_gray, seed = None, None
    for counter, frame in enumerate(frames_rgb):
        frame_gray = orc.cvtColor(frame)
        if len(tracks) > 0:
            p0 = np.float32([tr[-1] for tr in tracks]).reshape(-1, 1, 2)
            p1, st, err = orc.calcOpticalFlowPyrLK(prev_gray, frame_gray, p0, None, **lk_params)
            p0r, st, err = orc.calcOpticalFlowPyrLK(frame_gray, prev_gray, p1, None, **lk_params)
            diff = abs(p0 - p0r).reshape(-1, 2)
            dist = np.hypot(diff[:, 0], diff[:, 1])
            valid = dist < 1
            nt, nq = [], []
            for tr, (x, y), ok, trq, d in zip(tracks, p1.reshape(-1, 2), valid, trackquality, dist):
                if ok:
                    tr.append((x, y)); trq.append(d)
                    if (len(tr) - 1) > track_len:
                        del tr[0]
                    nt.append(tr); nq.append(trq)
            tracks, trackquality = nt, nq
        if counter % track_len == 0:
            if counter > 0:
                out[seed] = (np.array(tracks), np.array(trackquality))
            p = orc.goodFeaturesToTrack(frame_gray, mask=mask, **feature_params)
            tracks, trackquality, seed = [], [], counter
            if p is not None:
                for x, y in np.float32(p).reshape(-1, 2):
                    tracks.append([(x, y)]); trackquality.append([])
        prev_gray = frame_gray
    return out


def load_seq():
    from iceberg_tracking_code_b200.tracking import load_image
    names = sorted(os.listdir(SEQ))
    return names, [load_image(os.path.join(SEQ, n)) for n in names]


def test_lucaskanade_run_vs_reference_recording(ibt, golden, capsys):
    """s0_1 LucasKanade(workspace, detect_interval, time_spacing).run(): same printed track counts, same final tracks
    as the unmodified reference class run in the build container (make_golden.py)."""
    from pathlib import Path
    from iceberg_tracking_code_b200.tracking import LucasKanade
    g = golden("seq_expected.npz")
    for di, expect_counts in ((2, None), (3, None)):
        lk = LucasKanade(Path(SEQ), di, 60)
        lk.run()
        ref = g["d%d_final_tracks" % di]
        got = np.float32(lk.tracks)
        assert got.shape == ref.shape, (di, got.shape, ref.shape)
        assert np.abs(got - ref).max() <= 0.01, di
        # per-detection corner lists and surviving-track counts of the reference run
        n_ref = [len(g["d%d_gftt%d" % (di, i)]) for i in range(int(g["d%d_n_gftt" % di]))]
        out = capsys.readouterr().out
        printed = [int(l.split()[0]) for l in out.splitlines() if l.endswith(" tracks")]
        assert len(printed) == len(n_ref)
        assert printed[0] == 0
    # detect_interval 2: reference printed 0, 398, 401 (tests/golden/make_golden.py log)
    lk = LucasKanade(Path(SEQ), 2, 60)
    lk.run()
    assert lk.track_counts == [0, 398, 401]


def test_track_sequence_vs_s1_restatement(ibt, oracle, tmp_path):
    from iceberg_tracking_code_b200 import tracking as trk
    names, frames = load_seq()
    for n in names:
        shutil.copy(os.path.join(SEQ, n), tmp_path / n)
    imagelist = sorted(str(p) for p in tmp_path.glob("*.jpg"))
    h, w = frames[0].shape[:2]
    mask = np.zeros((h, w), np.uint8)
    mask[20:h - 30, 40:w - 10] = 255
    ref = s1_loop_oracle(oracle, frames, mask, 2, trk.FEATURE_PARAMS, trk.LK_PARAMS)
    res = trk.track_sequence(imagelist, mask, 2, 60, startlist=[0])
    assert [r[0] for r in res] == sorted(ref) == [0, 2]
    for seed, path, tracks, quality in res:
        rt, rq = ref[seed]
        assert tracks.shape == rt.shape and tracks.dtype == np.float32 and quality.shape == rq.shape
        assert np.abs(tracks - rt).max() <= 0.01 and np.abs(quality - rq).max() <= 0.01
        # file name + content layout (SURVEY A.8), read back the way s2_cam_to_utm.py:233-247 does
        assert os.path.basename(path) == names[seed].split('.')[0] + "_120sec_at_60sec_tracks.npz"
        z = np.load(path)
        assert z["tracks"].shape == tracks.shape and z["tracks"].dtype == np.float32
        assert z["trackquality"].shape == (len(tracks), 2) and z["trackquality"].dtype == np.float32
        lst = z["tracks"].tolist()
        assert all(len(tr) == 3 and len(tr[0]) == 2 for tr in lst)
    # a missed photo (gap != 60 +- 2 s): the group is tracked but NOT saved (s1:366-390)
    os.rename(imagelist[2], str(tmp_path / "20190724-130230.jpg"))
    for f in tmp_path.glob("*.npz"):
        f.unlink()
    imagelist = sorted(str(p) for p in tmp_path.glob("*.jpg"))
    res = trk.track_sequence(imagelist, mask, 2, 60, startlist=[0])
    assert res == [] and not list(tmp_path.glob("*.npz"))


def test_lucaskanade_tracking_signature(ibt, oracle, tmp_path):
    """Same positional call as s1:219-222, with a CSV parameter sheet and a polygon mask file; crop offsets applied."""
    from iceberg_tracking_code_b200 import tracking as trk
    from iceberg_tracking_code_b200.camera import Camera, PARAM_COLUMNS
    names, frames = load_seq()
    src = tmp_path / "data" / "cam1" / "20190724"
    src.mkdir(parents=True)
    for n in names[:3]:
        shutil.copy(os.path.join(SEQ, n), src / n)
    h, w = frames[0].shape[:2]
    row = dict(camera="cam1", start_day=20190701, end_day=20190801, image_width=w, image_height=h, sensor_width=22.3,
               easting=377280.39, northing=6525846.97, elevation=261.3, antenna_height=1.6, theta=300.0, phi=5.0,
               psi=-1.0, sigma=18.0, crop_left=16, crop_right=8, crop_top=10, crop_bottom=20, tracking_interval=60,
               mask="mask.csv")
    pf = tmp_path / "data" / "parameter_file.csv"
    pf.write_text(",".join(PARAM_COLUMNS) + "\n" + ",".join(str(row[c]) for c in PARAM_COLUMNS) + "\n")
    poly = np.float64([(30, 20), (w - 40, 35), (w - 60, h - 50), (w // 2, h - 90), (50, h - 60)])
    np.savetxt(tmp_path / "data" / "cam1" / "mask.csv", poly, delimiter=",")
    tgt = tmp_path / "out" / "cam1" / "oblique" / "20190724"
    trk.lucaskanade_tracking(str(tmp_path), str(src), str(tgt), "cam1", 2, 60, [0], 1, 0, 0, 0, str(pf), 1)
    files = sorted(tgt.glob("*.npz"))
    assert [f.name for f in files] == ["20190724-130000_120sec_at_60sec_tracks.npz"]
    # oracle: crop (PIL, like camtools.py:79) + polygon mask by the crossing rule + the s1 loop
    cropped = [trk.load_image(str(p)) for p in sorted(tgt.glob("*.jpg"))]
    assert cropped[0].shape[:2] == (h - 30, w - 24)
    cam = Camera("cam1", "20190724", str(pf), mask=1)
    mask = cam.mask_image(h - 30, w - 24).cpu().numpy()
    ys, xs = np.mgrid[0:h - 30, 0:w - 24]
    ref_mask = crossing_mask(poly - [16, 10], xs, ys)
    assert np.array_equal(mask, ref_mask)
    ref = s1_loop_oracle(oracle, cropped, ref_mask, 2, trk.FEATURE_PARAMS, trk.LK_PARAMS)
    z = np.load(files[0])
    assert z["tracks"].shape == ref[0][0].shape and np.abs(z["tracks"] - ref[0][0]).max() <= 0.01

    # crop="view" (SURVEY 8f-1): source files decoded on the GPU and cropped as a view -- no re-encoded copies are written,
    # same .npz name, tracks = the s1 loop on the cropped PIXELS OF THE SOURCE frames (no second JPEG generation)
    tgt2 = tmp_path / "out2" / "cam1" / "oblique" / "20190724"
    trk.lucaskanade_tracking(str(tmp_path), str(src), str(tgt2), "cam1", 2, 60, [0], 1, 0, 0, 0, str(pf), 1, crop="view")
    assert [f.name for f in sorted(tgt2.iterdir())] == ["20190724-130000_120sec_at_60sec_tracks.npz"]
    view = [f[10:h - 20, 16:w - 8] for f in frames[:3]]
    ref2 = s1_loop_oracle(oracle, view, ref_mask, 2, trk.FEATURE_PARAMS, trk.LK_PARAMS)
    z2 = np.load(tgt2 / "20190724-130000_120sec_at_60sec_tracks.npz")
    assert z2["tracks"].shape == ref2[0][0].shape and np.abs(z2["tracks"] - ref2[0][0]).max() <= 0.01

    # crop="emulate": no host pre-pass and no cropped copies either, but the SAME pixels as crop="reencode" (the reference's
    # route): the save-and-reopen round trip of camtools.crop_image_standalone runs as integer arithmetic on the GPU
    tgt3 = tmp_path / "out3" / "cam1" / "oblique" / "20190724"
    trk.lucaskanade_tracking(str(tmp_path), str(src), str(tgt3), "cam1", 2, 60, [0], 1, 0, 0, 0, str(pf), 1, crop="emulate")
    assert [f.name for f in sorted(tgt3.iterdir())] == ["20190724-130000_120sec_at_60sec_tracks.npz"]
    z3 = np.load(tgt3 / "20190724-130000_120sec_at_60sec_tracks.npz")
    assert z3["tracks"].tobytes() == z["tracks"].tobytes() and z3["trackquality"].tobytes() == z["trackquality"].tobytes()


def crossing_mask(poly, xs, ys):
    """numpy restatement of the crossing-number rule matplotlib's Path.contains_points applies (camtools.py:208-209)."""
    inside = np.zeros(xs.shape, bool)
    n = len(poly)
    tx, ty = xs.astype(np.float64), ys.astype(np.float64)
    for i in range(n):
        (x0, y0), (x1, y1) = poly[i - 1], poly[i]
        f0, f1 = y0 >= ty, y1 >= ty
        cross = (f0 != f1) & ((((y1 - ty) * (x0 - x1)) >= ((x1 - tx) * (y0 - y1))) == f1)
        inside ^= cross
    return np.where(inside, 255, 0).astype(np.uint8)


def test_sharded_equals_unsharded(ibt):
    """N time blocks run one after another on one GPU == the 1-rank run, byte for byte (SURVEY 8e determinism)."""
    from iceberg_tracking_code_b200 import sharding as sh, synthetic as syn, tracking as trk
    base = syn.base_texture(200, 320, 5)
    frames = [syn.frame_rgb(base, t, seed=5).numpy() for t in range(9)]
    gp = dict(maxCorners=400, qualityLevel=0.01, minDistance=8, blockSize=5)
    lp = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
    whole = trk.track_sequence(frames, None, 2, 60, loader=None, feature_params=gp, lk_params=lp, save=False)
    assert [r[0] for r in whole] == [0, 2, 4, 6]
    for world in (2, 3, 4):
        parts = []
        for rank in range(world):
            parts += sh.track_sequence_sharded(frames, None, 2, 60, rank=rank, world=world, gather=False, loader=None,
                                               feature_params=gp, lk_params=lp, save=False)
        parts.sort(key=lambda r: r[0])
        assert [p[0] for p in parts] == [r[0] for r in whole]
        for (s, t, q), (s2, _p, t2, q2) in zip(parts, whole):
            assert t.tobytes() == t2.tobytes() and q.tobytes() == q2.tobytes()


def test_tracks_compact_and_empty_group(ibt):
    from iceberg_tracking_code_b200 import synthetic as syn
    from iceberg_tracking_code_b200.tracking import SequenceTracker
    base = syn.base_texture(120, 160, 8)
    f = [syn.frame_gray(base, t).cuda() for t in range(3)]
    lp = dict(winSize=(15, 15), maxLevel=2, criteria=(3, 30, 0.01))
    trk = SequenceTracker(dict(maxCorners=300, qualityLevel=0.01, minDistance=5, blockSize=3), lp)
    pyr = [trk.prepare(x) for x in f]
    n = trk.seed(pyr[0], None, 2)
    trk.track(pyr[0], pyr[1]); trk.track(pyr[1], pyr[2])
    alive = trk._alive.cpu().numpy().astype(bool)
    tracks, quality = trk.harvest()
    tm, qm = trk._tracks.cpu().numpy(), trk._quality.cpu().numpy()
    assert np.array_equal(tracks, tm[:, alive].transpose(1, 0, 2)) and np.array_equal(quality, qm[:, alive].T)
    assert tracks.shape[0] == trk.alive_count() and (quality < 1).all()
    # kill everything: empty -> two (0,) float64 arrays, like np.savez(tracks=[]) at s1:395
    trk._alive.zero_()
    t0, q0 = trk.harvest()
    assert t0.shape == (0,) and t0.dtype == np.float64 and q0.shape == (0,)
    # a flat frame seeds nothing and tracking it is a no-op
    flat = trk.prepare(torch.full((120, 160), 9, dtype=torch.uint8, device="cuda"))
    assert trk.seed(flat, None, 2) == 0
    trk.track(flat, pyr[1])
    assert trk.harvest()[0].shape == (0,)


@pytest.mark.parametrize("n", [1, 262144, 262145, 300000, 2097152, 2097153])
def test_tracks_compact_across_scan_tiles(ibt, n):
    """Compaction of n tracks: its ceil(n / 256) block counts take one 1024-element step of the one-CTA scan up to
    n = 262 144, several steps up to n = 2 097 152 (8 192 counts), and the multi-tile scan (partial sums inside the
    scratch) above."""
    from iceberg_tracking_code_b200.tracking import SequenceTracker
    rng = np.random.default_rng(n)
    T = 3
    tm = rng.standard_normal((T + 1, n, 2)).astype(np.float32)
    qm = rng.random((T, n), dtype=np.float32)
    alive = rng.random(n) < 0.7
    alive[-1] = True
    trk = SequenceTracker()
    trk.n, trk.T, trk.steps = n, T, T
    trk._tracks, trk._quality = torch.from_numpy(tm).cuda(), torch.from_numpy(qm).cuda()
    trk._alive = torch.from_numpy(alive.astype(np.uint8)).cuda()
    want_t, want_q = tm[:, alive].transpose(1, 0, 2), qm[:, alive].T
    for tracks, quality in (trk.harvest(), trk.finalize(trk.harvest_async())):
        assert np.array_equal(tracks, want_t) and np.array_equal(quality, want_q)


def test_config2_full_size_properties(ibt, oracle):
    """BASELINE config 2 at full size (6000x4000, 20k points, win 31, L4): determinism, known synthetic shift,
    FB round trip, and a sampled comparison with the oracle (the oracle is too slow for all 20k)."""
    from iceberg_tracking_code_b200 import synthetic as syn
    H, W = 4000, 6000
    base = syn.base_texture(H, W, 7, device="cuda")
    f0, f1 = syn.frame_gray(base, 0), syn.frame_gray(base, 1)
    del base
    lp = dict(winSize=(31, 31), maxLevel=4, criteria=(3, 30, 0.01))
    pts = ibt.goodFeaturesToTrack(f0, maxCorners=20000, qualityLevel=0.007, minDistance=10, blockSize=10)
    assert pts.shape == (20000, 1, 2)
    xy = pts.reshape(-1, 2).cpu().numpy()
    d2 = ((xy[:2000, None, :] - xy[None, :2000, :]) ** 2).sum(-1) + np.eye(2000) * 1e9
    assert d2.min() >= 100                                   # minDistance 10 respected
    pa, pb = ibt.FramePyramid(f0, (31, 31), 4), ibt.FramePyramid(f1, (31, 31), 4)
    r1 = ibt.calcOpticalFlowPyrLK_FB(pa, pb, pts, return_iters=True, **lp)
    r2 = ibt.calcOpticalFlowPyrLK_FB(pa, pb, pts, **lp)
    assert torch.equal(r1["p1"], r2["p1"]) and torch.equal(r1["dist"], r2["dist"])      # deterministic
    d = (r1["p1"] - pts).reshape(-1, 2)
    med = d.median(0).values.cpu().numpy()
    assert np.abs(med - [-syn.VX, -syn.VY]).max() < 0.02
    assert float(r1["valid"].float().mean()) > 0.99 and float(r1["st1"].float().mean()) > 0.99
    it = r1["iters"].sum().item() / 20000.0
    assert 20 < it < 70                                      # SURVEY 8d: ~41.7 iterations per point per pair
    # sampled parity against the oracle at full size
    sel = np.random.default_rng(0).choice(20000, 300, replace=False)
    g0, g1 = f0.cpu().numpy(), f1.cpu().numpy()
    sp = pts.cpu().numpy()[sel]
    p1_o, st_o, err_o, it_o = oracle.calcOpticalFlowPyrLK(g0, g1, sp, None, return_iters=True, **lp)
    assert_lk_exact(dict(p1=r1["p1"].cpu().numpy()[sel], st=r1["st1"].cpu().numpy()[sel], err=r1["err1"].cpu().numpy()[sel],
                         iters=r1["iters"].cpu().numpy()[sel, 0]), dict(p1=p1_o, st=st_o, err=err_o, iters=it_o),
                    "config 2 sample", sp)
    # corners vs oracle on a 1000x1500 crop of the same frame (full-frame oracle GFTT takes minutes)
    crop = np.ascontiguousarray(g0[500:1500, 1000:2500])
    gp = dict(maxCorners=0, qualityLevel=0.007, minDistance=10, blockSize=10)
    assert corner_overlap(ibt.goodFeaturesToTrack(crop, **gp), oracle.goodFeaturesToTrack(crop, **gp)) >= CORNER_OVERLAP


def test_config4_dense_grid(ibt, oracle):
    """BASELINE config 4 shape: grid-seeded points, maxLevel 5, 30 iterations (reduced frame so the oracle finishes)."""
    from iceberg_tracking_code_b200 import synthetic as syn
    base = syn.base_texture(1200, 1600, 7)
    f0, f1 = syn.frame_gray(base, 0).numpy(), syn.frame_gray(base, 1).numpy()
    pts = syn.grid_points(1200, 1600, step=11, limit=4000).numpy()
    lp = dict(winSize=(31, 31), maxLevel=5, criteria=(3, 30, 0.01))
    p1, st, err, it = ibt.calcOpticalFlowPyrLK(f0, f1, pts, None, return_iters=True, **lp)
    p1_o, st_o, err_o, it_o = oracle.calcOpticalFlowPyrLK(f0, f1, pts, None, return_iters=True, **lp)
    assert_lk_exact(dict(p1=p1, st=st, err=err, iters=it), dict(p1=p1_o, st=st_o, err=err_o, iters=it_o), "config 4", pts)


def test_config4_full_size_sample(ibt, oracle):
    """BASELINE config 4 at FULL size (24 MP pair, np.mgrid[10:4000:11, 10:6000:11] = 197 835 points, maxLevel 5, 30
    iterations, fwd + bwd + FB in one launch); 600 sampled points are re-tracked by the CPU oracle."""
    import torch
    from iceberg_tracking_code_b200 import synthetic as syn
    H, W = 4000, 6000
    lp = dict(winSize=(31, 31), maxLevel=5, criteria=(3, 30, 0.01))
    base = syn.base_texture(H, W, 7, device="cuda")
    g0, g1 = syn.frame_gray(base, 0), syn.frame_gray(base, 1)
    del base
    pts = syn.grid_points(H, W, step=11, start=10).reshape(-1, 2).cuda()
    n = pts.shape[0]
    assert n == 197835
    pa, pb = ibt.FramePyramid(g0, lp["winSize"], lp["maxLevel"], True), ibt.FramePyramid(g1, lp["winSize"], lp["maxLevel"], True)
    assert pa.maxLevel == 5
    p1 = torch.empty((n, 2), dtype=torch.float32, device="cuda")
    fbd = torch.empty((n,), dtype=torch.float32, device="cuda")
    ibt.lk_fb_into(pa, pb, pts, lp, p1, fbd, None, None)
    sel = np.random.default_rng(4).choice(n, 600, replace=False)
    p0s = pts[sel].cpu().numpy()
    g0n, g1n = g0.cpu().numpy(), g1.cpu().numpy()
    p1_o, st_o, _ = oracle.calcOpticalFlowPyrLK(g0n, g1n, p0s, None, **lp)
    p0r_o, _, _ = oracle.calcOpticalFlowPyrLK(g1n, g0n, p1_o, None, **lp)
    d_o, _ = oracle.fb_check(p0s, p0r_o)
    assert_lk_exact(dict(p1=p1[sel].cpu().numpy()), dict(p1=p1_o), "config 4 full size", p0s)
    # the FB distance is numpy's float32 hypot, bit for bit
    assert _f32_same(fbd[sel].cpu().numpy(), d_o).all()
    assert float((fbd < 1).float().mean()) > 0.99          # the synthetic shift is tracked everywhere


def test_config5_tracks_to_utm(ibt, golden):
    from iceberg_tracking_code_b200.camera import Camera
    g = golden("utm_expected.npz")
    params = dict(image_width=6000, image_height=4000, sensor_width=22.3, easting=377280.39, northing=6525846.97,
                  elevation=261.3, antenna_height=1.6, theta=300.0, phi=5.0, psi=-1.0, sigma=18.0, crop_left=250,
                  crop_right=0, crop_top=400, crop_bottom=0)
    cam = Camera("cam1", parameters=params, tide_elevation=0.37)
    tracks = g["xy"].reshape(-1, 2, 2)                       # (M, T+1, 2) with T = 1
    en = cam.tracks_to_utm(tracks)
    assert en.shape == tracks.shape and en.dtype == np.float64
    assert np.array_equal(en.reshape(-1, 2), g["EN"])


def test_async_pieces_equal_synchronous(ibt):
    """The asynchronous forms the pipelined loop uses give the same answers as the synchronous calls they replace:
    gftt_prefetch + seed(prefetched=) vs goodFeaturesToTrack, harvest_async + finalize vs harvest, and the LK launch under an
    occupancy cap (ibt_lk_set_max_ctas_per_sm) vs the full-occupancy launch."""
    from iceberg_tracking_code_b200 import synthetic as syn
    from iceberg_tracking_code_b200.tracking import SequenceTracker
    base = syn.base_texture(700, 900, 11, device="cuda")
    f = [syn.frame_gray(base, t) for t in range(3)]
    gp = dict(maxCorners=3000, qualityLevel=0.007, minDistance=10, blockSize=10)
    lp = dict(winSize=(31, 31), maxLevel=3, criteria=(3, 30, 0.01))
    a, b = SequenceTracker(gp, lp), SequenceTracker(gp, lp)
    pa = [a.prepare(x) for x in f]
    pb = [b.prepare(x) for x in f]
    na = a.seed(pa[0], None, 2)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        pf = b.gftt_prefetch(pb[0], None)
    nb = b.seed(pb[0], None, 2, prefetched=pf)
    assert na == nb and torch.equal(a._tracks[0], b._tracks[0])
    ref = ibt.goodFeaturesToTrack(f[0], **gp)
    assert torch.equal(a._tracks[0], ref.reshape(-1, 2))
    a.track(pa[0], pa[1]); a.track(pa[1], pa[2])
    ibt.set_lk_resident_ctas(1)
    try:
        b.track(pb[0], pb[1])
        ibt.set_lk_resident_ctas(2)
        b.track(pb[1], pb[2])
    finally:
        ibt.set_lk_resident_ctas(0)
    ta, qa = a.harvest()
    tb, qb = b.finalize(b.harvest_async())
    assert np.array_equal(ta, tb) and np.array_equal(qa, qb) and ta.shape[0] > 2000
    # all corners (maxCorners = 0) and a mask through the asynchronous form
    c = SequenceTracker(dict(gp, maxCorners=0), lp)
    mask = torch.zeros((700, 900), dtype=torch.uint8, device="cuda"); mask[100:600, 50:800] = 255
    pc = c.prepare(f[0])
    n = c.seed(pc, mask, 2, prefetched=c.gftt_prefetch(pc, mask))
    ref = ibt.goodFeaturesToTrack(f[0], mask=mask, **dict(gp, maxCorners=0))
    assert n == ref.shape[0] and torch.equal(c._tracks[0], ref.reshape(-1, 2))
