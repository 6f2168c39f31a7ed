"""Multi-channel frames on the GPU: the prepare step of a 24 MP 3-channel frame (ibt_pyramid_build_multichannel: level 0 of
every channel from the interleaved frame in one launch, then one launch per further level) and the forward-backward LK step
on cached colour pyramids (ibt_lk_fb_multichannel), against what it replaces: two colour calcOpticalFlowPyrLK calls, each
building both frames' pyramids, plus the FB arithmetic in numpy.

    python tools/bench_colour.py [--steps 30] [--warmup 5]

Timings are medians of CUDA-event windows after warm-up.  The prepare loop rotates through 4 frames (72 MB each) into 2
pyramids (~500 MB written per build), so neither its input nor its output is served from the 126 MB L2.  Bytes are the
algorithmic ones, computed from the shapes: every input byte read once, every output byte written once."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from iceberg_tracking_code_b200 import cv, synthetic as syn          # noqa: E402

PEAK_GBS = 6468.0       # the project's measured HBM bandwidth on the B200 (device-to-device copy)


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                                        str(torch.cuda.current_device())], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name()


def prepare_bytes(p):
    """(level-0 launch, levels >= 1) algorithmic bytes of one build"""
    cn, L = p.cn, p.maxLevel + 1
    (h0, w0) = p.sizes[0]
    lvl0 = h0 * w0 * cn * (1 + 1 + 4) + (p.sizes[1][0] * p.sizes[1][1] * cn if L > 1 else 0)
    rest = 0
    for l in range(1, L):
        h, w = p.sizes[l]
        rest += h * w * cn * (1 + 4) + (p.sizes[l + 1][0] * p.sizes[l + 1][1] * cn if l + 1 < L else 0)
    return lvl0, rest


def median_events(fn, steps, warmup):
    for _ in range(warmup):
        fn(0)
    torch.cuda.synchronize()
    ts = []
    for i in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(i)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def frame_kernel_ms(fn, n):
    """median device time (ms) of the level-0 launch, pyr_frame_kernel, from a profiled run of its own.  The builds are
    separated by a synchronise: the levels of a build are chained by programmatic dependent launch, so a build issued
    right behind another would start its level-0 kernel early and count the wait for the previous build's tail."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            fn(i)
            torch.cuda.synchronize()
    ts = [e.device_time / 1e3 for e in prof.events() if e.device_type.name == "CUDA" and "pyr_frame_kernel" in e.name]
    return float(np.median(ts)) if ts else float("nan")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--points", type=int, default=20000)
    args = ap.parse_args()
    H, W, cn, win, ml = 4000, 6000, 3, (31, 31), 4
    dev = torch.device("cuda")
    res = {"card": card(), "frame": [H, W, cn], "winSize": list(win), "maxLevel": ml}
    print("card (name, power limit):", res["card"])

    base = syn.base_texture(H, W, 11, device="cuda")
    frames = [syn.frame_rgb(base, t, seed=11) for t in range(4)]
    pyrs = [cv.FramePyramid(frames[i], win, ml, True) for i in range(2)]
    torch.cuda.synchronize()
    b0, b1 = prepare_bytes(pyrs[0])
    t_prep = median_events(lambda i: pyrs[i & 1].rebuild(frames[i % 4]), args.steps, args.warmup)
    t0 = frame_kernel_ms(lambda i: pyrs[i & 1].rebuild(frames[i % 4]), 20)
    res["prepare"] = {
        "ms_median": t_prep, "bytes": b0 + b1, "GBs": (b0 + b1) / t_prep / 1e6, "frac_of_peak": (b0 + b1) / t_prep / 1e6 / PEAK_GBS,
        "level0_kernel_ms": t0, "level0_bytes": b0, "level0_GBs": b0 / t0 / 1e6, "level0_frac_of_peak": b0 / t0 / 1e6 / PEAK_GBS,
        "levels_ge1_ms_by_difference": t_prep - t0, "levels_ge1_bytes": b1,
        "peak_GBs": PEAK_GBS}
    print("prepare: %.3f ms median, %.0f MB -> %.0f GB/s (%.2f of %.0f GB/s); level-0 kernel %.3f ms, %.0f MB -> %.0f GB/s (%.2f); "
          "levels >= 1: %.3f ms (by difference)"
          % (t_prep, (b0 + b1) / 1e6, res["prepare"]["GBs"], res["prepare"]["frac_of_peak"], PEAK_GBS, t0, b0 / 1e6,
             res["prepare"]["level0_GBs"], res["prepare"]["level0_frac_of_peak"], t_prep - t0))

    # FB step: pair (frame 0, frame 1), 20 k points on cached pyramids vs two colour calls + numpy
    pyrs[0].rebuild(frames[0])
    pyrs[1].rebuild(frames[1])
    rng = np.random.default_rng(3)
    pts = np.stack([rng.uniform(40, W - 40, args.points), rng.uniform(40, H - 40, args.points)], 1).astype(np.float32)
    pts_d = torch.from_numpy(pts).to(dev)
    lp = dict(winSize=win, maxLevel=ml, criteria=(3, 30, 0.01))
    t_fb = median_events(lambda i: cv.calcOpticalFlowPyrLK_FB(pyrs[0], pyrs[1], pts_d, **lp), args.steps, args.warmup)

    def two_calls():
        p1, st1, err1 = cv.calcOpticalFlowPyrLK(frames[0], frames[1], pts, None, **lp)
        p0r, st0, err0 = cv.calcOpticalFlowPyrLK(frames[1], frames[0], p1, None, **lp)
        d = np.abs(pts - p0r).reshape(-1, 2)
        return np.hypot(d[:, 0], d[:, 1]) < 1
    for _ in range(args.warmup):
        two_calls()
    ts = []
    for _ in range(max(5, args.steps // 3)):
        torch.cuda.synchronize()
        t = time.perf_counter()
        two_calls()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t) * 1e3)
    t_two = float(np.median(ts))
    r = cv.calcOpticalFlowPyrLK_FB(pyrs[0], pyrs[1], pts_d, **lp)
    res["fb_step"] = {"points": args.points, "ms_median_one_launch_cached_pyramids": t_fb,
                      "ms_median_two_colour_calls_plus_numpy": t_two, "speedup": t_two / t_fb,
                      "valid_fraction": float(r["valid"].float().mean())}
    print("FB step, %d points: one launch on cached colour pyramids %.3f ms; two colour calcOpticalFlowPyrLK calls + numpy "
          "FB %.3f ms (x%.1f); %.3f of the points pass FB" % (args.points, t_fb, t_two, t_two / t_fb,
                                                               res["fb_step"]["valid_fraction"]))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
