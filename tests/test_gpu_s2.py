"""The s2 consumer (cam_to_utm) on the GPU against the recorded run of the UNMODIFIED reference worker
(tests/golden/s2_expected.npz, make_golden.py:make_s2) and against the oracle restatement of s2:243-343."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _camera_params(g):
    vals = dict(zip(g["params_keys"].tolist(), g["params_vals"].tolist()))
    return vals


def test_cam_to_utm_vs_reference_run(ibt, golden, tmp_path):
    import pandas as pd
    from iceberg_tracking_code_b200.utm import cam_to_utm
    g = golden("s2_expected.npz")
    vals = _camera_params(g)
    src = tmp_path / "output" / "cam1" / "oblique" / "20190724"
    tgt = tmp_path / "output" / "cam1" / "utm"
    src.mkdir(parents=True); tgt.mkdir(parents=True); (tmp_path / "data").mkdir()
    stamps = g["stamps"].tolist()
    for si, stamp in enumerate(stamps):
        name = src / ("%s_120sec_at_60sec_tracks.npz" % stamp)
        if "in%d_tracks" % si in g:
            tr = g["in%d_tracks" % si]
            np.savez(name, tracks=tr, trackquality=np.zeros((len(tr), 2), np.float32))
        else:
            np.savez(name, tracks=[], trackquality=[])
    pf = tmp_path / "data" / "parameter_file.csv"
    pf.write_text(",".join(vals.keys()) + "\n" + ",".join(vals.values()) + "\n")
    tides = pd.DataFrame({"date": pd.to_datetime(g["tide_minutes"].tolist()), "depth_tide_ellipsoid": g["tide_values"]})
    tide_path = tmp_path / "data" / "tide_2019.pickle"
    tides.to_pickle(tide_path)
    cam_to_utm((str(src), str(tgt), "cam1", 1.7, 0.0, 2.5, 60, 0.1, str(pf), str(tide_path)))
    files = sorted(os.listdir(tgt))
    assert files == g["out_files"].tolist()
    for fi, f in enumerate(files):
        z = np.load(tgt / f)
        for k in ("x", "y", "u", "v", "speed", "time"):
            ref = g["out%d_%s" % (fi, k)]
            got = z[k]
            assert got.shape == ref.shape and got.dtype == ref.dtype, (f, k, got.shape, ref.shape, got.dtype, ref.dtype)
            # bit for bit: the projection is the reference's operation order unfused, speed is glibc's hypot restated
            assert np.array_equal(got, ref), (f, k, int((got != ref).sum()))


def test_track_velocities_vs_oracle(ibt, oracle, golden):
    from iceberg_tracking_code_b200.utm import track_velocities
    cam = golden("utm_expected.npz")["cam"]
    rng = np.random.default_rng(4)
    for T in (1, 2, 3, 5):
        M = 400
        p0 = (rng.random((M, 1, 2)) * [5200, 1700] + [100, 1500])
        step = rng.normal(0, 1.0, (M, 1, 2)) + rng.normal(0, 0.4, (M, T, 2))
        step[::9] *= 10.0; step[4::11] *= -1.0; step[5::13] = 0.0; step[6::17, 0] = 0.0
        tr = np.concatenate([p0, p0 + np.cumsum(step, 1)], 1).astype(np.float32)
        args = (cam, 60, 0.0, 1.7, 2.5, 60, 0.1)
        r = track_velocities(tr, *args)
        EN, uv, sp, keep = oracle.track_velocities(tr, *args)
        assert np.array_equal(r["EN"].cpu().numpy(), EN) and np.array_equal(r["uv"].cpu().numpy(), uv), T
        assert np.array_equal(r["speed"].cpu().numpy(), sp, equal_nan=True), T
        got = r["keep"].cpu().numpy()
        assert np.array_equal(got, keep), (T, np.flatnonzero(got != keep)[:6])
        if T >= 2:
            assert 0.1 < keep.mean() < 0.98, keep.mean()          # the criteria actually fire on this input
