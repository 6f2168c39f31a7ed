#!/usr/bin/env python
"""bench.py -- tracking hot path throughput on B200 (contract: see the task prompt / DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

--steps K is the number of timed steps of value, with_status_err, e2e and e2e_rgb_frames.  --dump-outputs DIR writes what the
last timed step of value returned (see dump_outputs) as .npy files; the inputs are generated from fixed seeds, so two builds
run with the same arguments can be compared file for file.

Workload = BASELINE.json configs[1]: 24 MP (6000x4000) synthetic frames, 20 000 Shi-Tomasi points, winSize 31,
maxLevel 4, criteria (EPS|COUNT, 30, 0.01), forward-backward check < 1 px.

One STEP = the body of the reference's frame loop for one new frame (s1_lucaskanade_tracking.py:310-359):
    cvtColor(new frame)  ->  [pyramid + Scharr planes of the new frame]  ->  LK forward  ->  LK backward  ->  FB check
against the previous frame, on 20 000 points.  goodFeaturesToTrack runs once per track_len frames in the reference; it
is timed separately ("gftt_ms") and inside "sharded_sequence".  metric = tracked points / s (= 20 000 x frame pairs / s).

  value : inputs (RGB frames, points) resident in HBM; CUDA events; max over ranks.  Frame pairs of this stream are
          independent, so consecutive steps are software-pipelined over two CUDA streams (three pyramid slots).
  e2e   : the public host API fed what the reference's loop is fed (s1:310): the JPEG bytes of every new frame in HOST memory;
          every step copies them host->device (3.8 MB), decodes on the GPU (jpeg.JpegDecoder), builds the pyramid, tracks, and
          reads p1 / FB distance back to the host, inside the timed region.  e2e_rgb_frames is the same loop fed the decoded
          72 MB RGB array (np.array(Image.open(f))) from pinned host memory: PCIe-bound, kept for comparison.
  sharded_sequence : BASELINE configs[2] in small: a fixed list of frames, track_len 2, GFTT re-seeding, sharded by
          contiguous time blocks over the ranks (sharding.track_sequence_sharded), the NCCL gather of all tracks INSIDE
          the timed region.  Total work is fixed: this is the strong-scaling line.
  parity : our outputs on the timed frames against cv2's (BASELINE's four criteria), N = 1 only.
  --impl reference : the reference's own CPU implementation of the same step -- the cv2 calls of s1:311,323,326 +
          the numpy FB arithmetic of s1:329-333 -- on the host cores (falls back to the C oracle port when cv2 is absent).
"""
import argparse
import gc
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the tree may be read-only: the benchmark writes nothing into it

H, W, NPTS = 4000, 6000, 20000
LK = dict(winSize=(31, 31), maxLevel=4, criteria=(3, 30, 0.01))
GFTT = dict(maxCorners=NPTS, qualityLevel=0.007, minDistance=10, blockSize=10)
NFRAMES = 6                    # distinct frames in rotation: 6 x 72 MB RGB = 432 MB  >  126 MB L2
SEED = 7
METRIC = "tracked points/sec (24MP frame pairs, 20k pts, LK fwd+bwd+FB)"
# identical in both arms (the driver compares it)
CONFIG = {
    "workload": "config2: 6000x4000 synthetic pair stream, 20k Shi-Tomasi pts, win 31, maxLevel 4, (3,30,0.01), FB<1px",
    "frames_in_rotation": NFRAMES,
    "l2_policy": "inputs larger than L2: %d distinct 72 MB RGB frames in ping-pong rotation" % NFRAMES,
    "step": "cvtColor(new) + pyramid/Scharr(new) + LK fwd + LK bwd + FB check vs the previous frame (s1:311,323,326,329-333)",
    "sharding": "independent frame-pair streams per rank, no data-path collective",
}
SPIN_CYCLES = int(3e7)         # ~15 ms spin ahead of a timed region: the host enqueues its steps before the GPU starts on them
DUMP_SAMPLE = 1 << 18          # --dump-outputs: pixels per pyramid plane (fixed seeded positions); all files 13 MB <= 64 MB
SEQ_FRAMES = 8 * 46 + 1        # sharded_sequence: 369 frames = 184 groups of track_len 2 (23 per rank at N = 8)
SEQ_T = 2


def pingpong(i):
    """frame index sequence 0,1,..,F-1,F-2,..,1,0,1,.. : consecutive frames always differ by one time step"""
    p = 2 * (NFRAMES - 1)
    k = i % p
    return k if k < NFRAMES else p - k


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons during the timed region (NVML; nvidia-smi as fallback)."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            nv = pynvml
            self.names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            self.ok = True
        except Exception as e:                      # noqa: BLE001
            self.err = repr(e)

    def sample_now(self):
        """One synchronous sample (called while the timed kernels are still in flight, so short runs get one too)."""
        if not self.ok:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:                       # noqa: BLE001
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, name in self.names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:                           # noqa: BLE001
            pass

    def run(self):
        if not self.ok:
            return
        while not self._halt.is_set():
            self.sample_now()
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
def make_frames(device):
    """NFRAMES RGB frames (H,W,3) u8 generated ON DEVICE (never shipped from the host in the device-timed loop)."""
    import torch
    from iceberg_tracking_code_b200 import synthetic as syn
    base = syn.base_texture(H, W, SEED, device=device)
    frames = [syn.frame_rgb(base, t, seed=SEED) for t in range(NFRAMES)]
    del base
    torch.cuda.empty_cache()
    return frames


def cpu_step_fn(threads=None):
    """The reference's per-frame CPU work (s1:311,323,326,329-333) as a callable; prefers cv2 (the dependency the
    reference itself calls), else the C oracle port."""
    try:
        import cv2
        cv2.setNumThreads(os.cpu_count() if threads is None else int(threads))
        kind, cores = "reference", cv2.getNumThreads()
        m = cv2
        desc = "cv2 %s (the OpenCV the reference calls), %d threads" % (cv2.__version__, cores)
    except Exception:                               # noqa: BLE001
        from oracle import oracle as m
        kind, cores = "port", 1
        desc = "oracle/ibt_oracle.c scalar port, 1 thread"

    def step(prev_gray, rgb, p0):
        gray = m.cvtColor(rgb, 6)
        p1, st, err = m.calcOpticalFlowPyrLK(prev_gray, gray, p0, None, **LK)
        p0r, st, err = m.calcOpticalFlowPyrLK(gray, prev_gray, p1, None, **LK)
        diff = abs(p0 - p0r).reshape(-1, 2)
        dist = np.hypot(diff[:, 0], diff[:, 1])
        return gray, p1, dist < 1
    return step, m, kind, cores, desc


def run_cpu(frames_np, grays_np, pts_np, steps, warmup, budget_s=None, threads=None):
    step, m, kind, cores, desc = cpu_step_fn(threads)
    t_total, done = 0.0, 0
    for i in range(warmup + steps):
        a, b = pingpong(i), pingpong(i + 1)
        t0 = time.perf_counter()
        step(grays_np[a], frames_np[b], pts_np[a])
        dt_ = time.perf_counter() - t0
        if i >= warmup:
            t_total += dt_
            done += 1
            if budget_s is not None and t_total > budget_s:
                break
    return dict(value=NPTS * done / t_total, unit="points/s", cores=cores, kind=kind,
                sample="%d frame pairs of the same workload (%s), %.2f s" % (done, desc, t_total),
                pairs_per_s=done / t_total), done, t_total


# ---------------------------------------------------------------------------------------------------------------------
class PairPipeline:
    """The config-2 stream of independent frame pairs, software-pipelined over two CUDA streams and three pyramid slots.
    Step i runs on stream i & 1: it builds the new frame's gray plane + pyramid into slot i % 3 and tracks the step's
    points from slot (i-1) % 3 (built by step i-1 on the other stream; one event wait) to it.  Slot i % 3 was last read
    by step i-2's LK on this same stream, so stream order covers the reuse.  The persistent LK launch of step i+1 fills
    the SMs as the warps of step i run out of points (a 20 k-point launch otherwise idles ~13 % of its time in the tail)."""

    def __init__(self, trk, dev, frame0, want_status_err=False):
        import torch
        from iceberg_tracking_code_b200 import cv
        self.torch, self.cv, self.trk, self.dev = torch, cv, trk, dev
        self.streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
        self.pyr = [trk.prepare(frame0) for _ in range(3)]
        self.ready = [torch.cuda.Event() for _ in range(3)]
        f32 = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
        u8 = lambda *s: torch.empty(s, dtype=torch.uint8, device=dev)
        self.p1 = [f32(NPTS, 2), f32(NPTS, 2)]
        self.fbd = [f32(NPTS), f32(NPTS)]
        self.sterr = None
        if want_status_err:            # what cv2 returns and the reference discards (s1:323,326): st, err of both passes
            self.sterr = [(u8(NPTS), f32(NPTS), f32(NPTS, 2), u8(NPTS), f32(NPTS)) for _ in range(2)]
        self.cnt, self.eps = cv._criteria(LK["criteria"])
        torch.cuda.synchronize()

    def prime(self, frame):
        """slot 2 (= slot of step -1) must hold the frame that step 0 tracks FROM"""
        torch = self.torch
        with torch.cuda.stream(self.streams[1]):
            self.trk.prepare(frame, reuse=self.pyr[2])
            self.ready[2].record(self.streams[1])

    def step(self, i, frame, pts, iter_total=None, probe=None):
        torch, cv = self.torch, self.cv
        import ctypes as C
        from iceberg_tracking_code_b200 import _native as N
        k = i & 1
        st = self.streams[k]
        with torch.cuda.stream(st):
            cur = self.trk.prepare(frame, reuse=self.pyr[i % 3], probe=probe)
            self.ready[i % 3].record(st)
            st.wait_event(self.ready[(i - 1) % 3])
            prev = self.pyr[(i - 1) % 3]
            p = cv._ptr
            if self.sterr is None:
                st1 = err1 = p0r = st0 = err0 = None
            else:
                st1, err1, p0r, st0, err0 = self.sterr[k]
            N.check(N.lib().ibt_lk_fb(C.byref(prev.c), C.byref(cur.c), p(pts), NPTS, 31, 31, self.cnt, self.eps, 1e-4, 1.0,
                                      p(self.p1[k]), p(st1), p(err1), p(p0r), p(st0), p(err0), p(self.fbd[k]), None, None,
                                      p(iter_total), cv._stream()), "ibt_lk_fb")
        return k

    def join(self, stream):
        """make `stream` wait for everything issued so far on both pipeline streams"""
        for s in self.streams:
            ev = self.torch.cuda.Event()
            ev.record(s)
            stream.wait_event(ev)


def timed_steps(pipe, frames, pts, first, n, iter_total=None, probes=None):
    for k in range(n):
        i = first + k
        pipe.step(i, frames[pingpong(i + 1)], pts[pingpong(i)], iter_total, None if probes is None else probes[k])


def dump_outputs(out_dir, p1, fb_dist, pyr):
    """--dump-outputs: what the last timed step returned to its caller, as float32 .npy files in out_dir: p1 (NPTS, 2) tracked
    positions and fb_dist (NPTS,) forward-backward distances of every point, and of the new frame's pyramid (what
    SequenceTracker.prepare returns) DUMP_SAMPLE pixels per level at positions drawn from SEED: level<l> (gray) and
    scharr<l> (dx, dy)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"p1": p1, "fb_dist": fb_dist}
    rng = np.random.default_rng(SEED)
    for l, (img, der) in enumerate(zip(pyr.levels, pyr.derivs)):
        n = img.numel()
        idx = torch.from_numpy(np.sort(rng.choice(n, min(n, DUMP_SAMPLE), replace=False))).to(img.device)
        arrays["level%d" % l] = img.reshape(-1)[idx]
        arrays["scharr%d" % l] = der.reshape(-1, 2)[idx]
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_from_files(trk, pipe, pts, host_frames, steps, cv, dev, ndec=None):
    """Same step, but the new frame arrives as the JPEG FILE the reference opens with Pillow (s1:310): the bytes are
    copied host->device compressed and csrc/jpeg.cu decodes them straight to the gray plane (bit-exact with Pillow +
    cv2.cvtColor).  The decodes of frames i+2 and i+3 (two decoders, two high-priority streams, no host wait: decode_async,
    convergence confirmed before the frame is used) run BESIDE the LK launch of pair i, which is capped at two of its three
    CTAs per SM (cv.set_lk_resident_ctas(2)); p1 / FB distance of every step are read back to the host and consumed one
    step later.  The CPU figure beside it is the reference's np.array(Image.open(f)) on the same bytes."""
    import io
    import torch
    from PIL import Image
    from iceberg_tracking_code_b200 import jpeg
    blobs = []
    for f in host_frames:
        bio = io.BytesIO()
        Image.fromarray(f.numpy()).save(bio, "JPEG")          # Pillow defaults, as the reference's cropping step saves
        blobs.append(bio.getvalue())
    # the loop keeps ND decodes in flight beside the tracker: their latency is hidden, so the entry-state probe of the Huffman pass
    # (a full-grid kernel that saves two of nine low-occupancy synchronisation rounds) is switched off for its duration
    jpeg.set_probe(os.environ.get("IBT_BENCH_PROBE") is not None)
    dec = jpeg.JpegDecoder(dev)
    g = dec.decode(blobs[0], rgb=False, gray=True)[1]
    ref = cv.cvtColor(torch.from_numpy(np.array(Image.open(io.BytesIO(blobs[0])))).to(dev))
    exact = bool(torch.equal(g, ref))
    h_p1 = [torch.empty((NPTS, 2), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_fbd = [torch.empty((NPTS,), dtype=torch.float32).pin_memory() for _ in range(2)]
    done = [torch.cuda.Event(), torch.cuda.Event()]
    # ND decoders on ND high-priority streams: a decode is a chain of small latency-bound kernels that runs ~2x slower beside
    # the LK launch (which keeps 80 % of the issue slots busy), so the step time is (decode latency under contention) / ND
    # until the LK launches themselves are the limit
    ND = int(ndec or os.environ.get("IBT_BENCH_NDEC", "2"))
    NS = ND + 2                                               # pyramid slots: two being tracked, ND being decoded ahead
    pyr = list(pipe.pyr) + [trk.prepare(g) for _ in range(NS - len(pipe.pyr))]
    main = torch.cuda.current_stream()
    decs = [dec] + [jpeg.JpegDecoder(dev) for _ in range(ND - 1)]
    for d in range(1, ND):
        decs[d].decode(blobs[d % len(blobs)], rgb=False, gray=True)
    dstream = [torch.cuda.Stream(device=dev, priority=-1) for _ in range(ND)]
    lk_done = [None] * NS
    redone = [0]

    # the host side of a decode (copy of the file bytes into page-locked memory, marker parsing: ~1 ms) runs on two worker threads
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=max(2, ND))
    staged = {}

    def prestage(j):
        if j not in staged:
            staged[j] = pool.submit(decs[j % ND].stage, blobs[pingpong(j)])

    def stage(j):
        """decode frame j (asynchronously: no host wait) -> gray -> pyramid into pyr[j % NS]; returns (handle, ready event)"""
        d = j % ND
        for a in range(ND + 1):
            prestage(j + a)
        sj = staged.pop(j).result()
        with torch.cuda.stream(dstream[d]):
            if lk_done[j % NS] is not None:
                dstream[d].wait_event(lk_done[j % NS])
            h = decs[d].decode_async(rgb=False, gray=True, staged=sj)
            trk.prepare(h["gray"], reuse=pyr[j % NS])
            ev = torch.cuda.Event()
            ev.record(dstream[d])
        return h, ev

    def confirm(j, st):
        """the Huffman pass of frame j had converged (else: decoded again, pyramid rebuilt)"""
        h, _ev = st
        if h["flags"] is None:
            return
        before = decs[j % ND].last_rounds
        decs[j % ND].confirm(h)
        if decs[j % ND].last_rounds == 0 or (before and decs[j % ND].last_rounds > h["rounds"]):
            redone[0] += 1
        if h.get("redo"):
            trk.prepare(h["gray"], reuse=pyr[j % NS])

    host = {"stage": 0.0, "confirm": 0.0, "lk": 0.0, "wait": 0.0}       # host seconds spent per phase (breakdown only)
    pc = time.perf_counter

    def loop(n, skip_lk=False):
        acc = 0.0
        st = {j: stage(j) for j in range(ND + 1)}
        for i in range(n):
            k = i & 1
            t0 = pc()
            if i == 0:
                confirm(0, st[0])
            confirm(i + 1, st[i + 1])
            t1 = pc()
            main.wait_event(st.pop(i)[1]); main.wait_event(st[i + 1][1])
            if not skip_lk:
                cv.lk_fb_into(pyr[i % NS], pyr[(i + 1) % NS], pts[pingpong(i)], LK, pipe.p1[k], pipe.fbd[k], None, None)
            e = torch.cuda.Event(); e.record(main)
            lk_done[i % NS] = e                               # pyr[i % NS] may be rebuilt once this launch has finished
            h_p1[k].copy_(pipe.p1[k], non_blocking=True); h_fbd[k].copy_(pipe.fbd[k], non_blocking=True)
            done[k].record(main)
            t2 = pc()
            if i + ND + 1 <= n:
                st[i + ND + 1] = stage(i + ND + 1)            # decoded beside the LK launches of pairs i .. i+ND-1
            t3 = pc()
            if i >= 1:
                done[k ^ 1].synchronize()
                acc += float(h_fbd[k ^ 1][0])
            t4 = pc()
            host["confirm"] += t1 - t0; host["lk"] += t2 - t1; host["stage"] += t3 - t2; host["wait"] += t4 - t3
        done[(n - 1) & 1].synchronize()
        for f in staged.values():                             # frames staged beyond the end of this loop: release their buffers
            f.result()["slot"]["free"].set()
        staged.clear()
        return acc + float(h_fbd[(n - 1) & 1][0])
    cv.set_lk_resident_ctas(2)
    try:
        loop(12 + 4 * ND)                                     # (every pinned staging buffer of every decoder exists afterwards)
        torch.cuda.synchronize()
        for k_ in host:
            host[k_] = 0.0
        gc.collect(); gc.disable()
        t0 = time.perf_counter()
        loop(steps)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / steps
        gc.enable()
        breakdown = None
        if os.environ.get("IBT_BENCH_BREAKDOWN"):
            # where a from-files step goes: host time per phase of the loop above, the same loop without the LK launches
            # (decode + pyramid + copies only) and the LK launches alone at the same occupancy cap
            breakdown = {"host_ms_per_step": {k: v * 1e3 / steps for k, v in host.items()}}
            torch.cuda.synchronize(); t0 = time.perf_counter()
            loop(steps, skip_lk=True)
            torch.cuda.synchronize()
            breakdown["decode_prepare_only_ms"] = (time.perf_counter() - t0) * 1e3 / steps
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                cv.lk_fb_into(pyr[i % NS], pyr[(i + 1) % NS], pts[pingpong(i)], LK, pipe.p1[i & 1], pipe.fbd[i & 1], None, None)
            e1.record(); torch.cuda.synchronize()
            breakdown["lk_only_capped_ms"] = e0.elapsed_time(e1) / steps
    finally:
        cv.set_lk_resident_ctas(0)
        jpeg.set_probe(True)
        pool.shutdown(wait=True)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    dec.last_rounds = 0                                       # a lone synchronous decode (probe on again): fresh round-count hint
    for k in range(2):
        dec.decode(blobs[k], rgb=False, gray=True)
    e0.record()
    for k in range(10):
        dec.decode(blobs[k % len(blobs)], rgb=False, gray=True)
    e1.record(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(3):
        np.array(Image.open(io.BytesIO(blobs[k])))
    pil_ms = (time.perf_counter() - t0) * 1e3 / 3
    return {"value": NPTS / (ms * 1e-3), "unit": "points/s", "ms_per_step": ms, "steps": steps,
            "h2d_bytes_per_step": int(np.mean([len(b) for b in blobs])), "d2h_bytes_per_step": int(h_p1[0].numel() * 4 + h_fbd[0].numel() * 4),
            "jpeg_decode_ms": e0.elapsed_time(e1) / 10, "huffman_sync_rounds": dec.last_rounds,
            "pillow_decode_ms_1_core": pil_ms, "bit_exact_vs_pillow_cvtcolor": exact, "decodes_repeated": redone[0], "decoders": ND,
            **({"breakdown": breakdown} if breakdown else {}),
            "api": "jpeg.JpegDecoder.decode_async(gray, no entry-state probe) on two streams + SequenceTracker.prepare + fused LK (2 of 3 CTAs per SM), "
                   "JPEG bytes in host memory, the next two frames decode beside the LK launches, p1 + FB distance read back "
                   "every step; wall clock"}


def run_sharded_sequence(dev, rank, world, dist):
    """BASELINE configs[2] in small (reference loop: s1:296-450; its day loop is serial, s1:194-195).  SEQ_FRAMES frames
    of 24 MP, track_len 2, top-20k Shi-Tomasi re-seeding, consecutive-pair tracking; groups sharded by contiguous time
    blocks (one halo frame per block), the final gather of every rank's tracks (NCCL) inside the timed region, rank 0
    then holds all tracks on the host.  Frames are synthesised on device before the timed region."""
    import torch
    from iceberg_tracking_code_b200 import sharding as sh, synthetic as syn, tracking as trk
    total = sh.n_groups(SEQ_FRAMES, SEQ_T)
    g0, n = sh.shard_groups(total, rank, world)
    first, last = sh.frame_range(g0, n, SEQ_T)
    base = syn.base_texture(H, W, 100, device=dev)
    # the scene drifts and wraps every 12 frames so that a long sequence stays inside the texture margin
    frames = {t: syn.frame_rgb(base, t % 12, seed=100 + t) for t in range(first, last + 1)}
    del base
    torch.cuda.synchronize()
    imagelist = list(range(SEQ_FRAMES))
    from iceberg_tracking_code_b200 import camera
    cam = camera.Camera(camname="cam1", parameters=dict(image_width=W, image_height=H, sensor_width=22.3, easting=377280.39,
                        northing=6525846.97, elevation=261.3, antenna_height=0.0, theta=300.0, phi=5.0, psi=-1.0, sigma=18.0))
    tracker = trk.SequenceTracker(GFTT, LK)
    kw = dict(loader=lambda t: frames[t], tracker=tracker, save=False, check_time=False, decode_workers=0)
    # warm-up: the whole job once, untimed (allocator pools, pinned staging buffers, NCCL channels, kernels)
    dev_res = {}
    res = trk.track_sequence(imagelist, None, SEQ_T, 60, first_group=g0, n_groups=n, device_results=dev_res, **kw)
    for _seed, (t_d, _q_d) in dev_res.items():
        cam.tracks_to_utm(t_d)
    sh.gather_results(res, SEQ_T, to_host="rank0", device_results=dev_res)
    del res, dev_res
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    gc.collect(); gc.disable()                             # (see main(): no collector pauses inside the timed region)
    t0 = time.perf_counter()
    dev_res = {}
    res = trk.track_sequence(imagelist, None, SEQ_T, 60, first_group=g0, n_groups=n, device_results=dev_res, **kw)
    torch.cuda.synchronize()
    t_track = time.perf_counter() - t0
    # BASELINE configs[4]: every track vertex of this rank's block projected to map coordinates (fp64 ray / plane,
    # camtools.py:286-332 via s2:243-254) with the synthetic camera of SURVEY 8d -- on the device-resident group arrays
    utm_vertices, utm_sum = 0, 0.0
    for _seed, (t_d, _q_d) in dev_res.items():
        en = cam.tracks_to_utm(t_d)
        utm_vertices += en.shape[0] * en.shape[1]
        last = en
    if utm_vertices:
        utm_sum = float(last[0, 0, 0])                                      # one host read: the projection has finished
    torch.cuda.synchronize()
    t_utm = time.perf_counter() - t0 - t_track
    allres = sh.gather_results(res, SEQ_T, to_host="rank0", device_results=dev_res)
    torch.cuda.synchronize()
    t_all = time.perf_counter() - t0
    gc.enable()
    if dist is not None:
        dist.barrier()
    tt = torch.tensor([t_all, t_track, t_all - t_track - t_utm, t_utm], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_all, t_track, t_gather, t_utm = [float(v) for v in tt.tolist()]
    nv = torch.tensor([utm_vertices], dtype=torch.int64, device=dev)
    if dist is not None:
        dist.all_reduce(nv)
    utm_vertices = int(nv.item())
    if rank != 0:
        return None
    ntracks = sum(len(t) for _s, t, _q in allres if getattr(t, "ndim", 1) == 3)
    hsh = hashlib.sha1()
    for _s, t, q in allres:
        if getattr(t, "ndim", 1) == 3:
            hsh.update(np.ascontiguousarray(t).tobytes()); hsh.update(np.ascontiguousarray(q).tobytes())
    pairs = total * SEQ_T
    return {"workload": "configs 3+5 in small: %d synthetic 24 MP frames, track_len %d, top-%d Shi-Tomasi re-seeding every %d frames, "
                        "win 31, L4; groups sharded by time block; every track vertex projected to UTM (fp64); NCCL gather of all "
                        "tracks inside the timed region"
                        % (SEQ_FRAMES, SEQ_T, NPTS, SEQ_T),
            "scaling": "strong", "n_gpus": world, "frames": SEQ_FRAMES, "groups": total, "frame_pairs": pairs,
            "seconds": t_all, "frame_pairs_per_s": pairs / t_all, "points_per_s": ntracks * SEQ_T / t_all,
            "tracks_gathered": ntracks, "track_ms_max_rank": t_track * 1e3, "gather_ms": t_gather * 1e3,
            "utm_vertices": utm_vertices, "utm_ms_max_rank": t_utm * 1e3,
            "ms_per_frame_pair_per_gpu": t_track * 1e3 / (pairs / world),
            "tracks_sha1": hsh.hexdigest(),
            "api": "sharding.track_sequence_sharded path: tracking.track_sequence per rank + sharding.gather_results"}


def run_parity(frames, grays, pts, trk, dev):
    """BASELINE's four criteria on the frames the bench times: our outputs vs cv2's on the same inputs (N = 1)."""
    import torch
    from iceberg_tracking_code_b200 import cv
    try:
        import cv2
    except Exception as e:                          # noqa: BLE001
        return {"skipped": "cv2 not importable: %r" % (e,)}
    cv2.setNumThreads(os.cpu_count())
    g0, g1 = grays[0].cpu().numpy(), grays[1].cpu().numpy()
    rgb1 = frames[1].cpu().numpy()
    out = {"against": "cv2 %s on the timed frames (pair 0 -> 1)" % cv2.__version__}
    out["gray_bit_exact"] = bool(np.array_equal(cv2.cvtColor(rgb1, cv2.COLOR_BGR2GRAY), g1))
    pa = cv.FramePyramid(grays[0], LK["winSize"], LK["maxLevel"], True)
    pb = cv.FramePyramid(grays[1], LK["winSize"], LK["maxLevel"], True)
    ml, ref = cv2.buildOpticalFlowPyramid(g1, LK["winSize"], LK["maxLevel"], withDerivatives=True)
    ok = ml == pb.maxLevel
    for l in range(ml + 1):
        ok = ok and np.array_equal(pb.levels[l].cpu().numpy(), ref[2 * l]) and np.array_equal(pb.derivs[l].cpu().numpy(), ref[2 * l + 1])
    out["pyramid_levels_and_scharr_bit_exact"] = bool(ok)
    c_ref = cv2.goodFeaturesToTrack(g0, **GFTT).reshape(-1, 2)
    c_our = pts[0].cpu().numpy().reshape(-1, 2)
    sa = set(map(tuple, c_our.astype(np.int64).tolist())); sb = set(map(tuple, c_ref.astype(np.int64).tolist()))
    out["corner_overlap"] = len(sa & sb) / max(1, len(sb))
    nmin = min(len(c_our), len(c_ref))
    out["corner_count"] = [int(len(c_our)), int(len(c_ref))]
    out["corner_same_rank_fraction"] = float(np.mean(np.all(c_our[:nmin] == c_ref[:nmin], axis=1))) if nmin else None
    p0 = c_ref.reshape(-1, 1, 2).astype(np.float32)
    r = cv.calcOpticalFlowPyrLK_FB(pa, pb, torch.from_numpy(p0).to(dev), **LK)
    p1c, st1c, _ = cv2.calcOpticalFlowPyrLK(g0, g1, p0, None, **LK)
    p0rc, st0c, _ = cv2.calcOpticalFlowPyrLK(g1, g0, p1c, None, **LK)
    p1 = r["p1"].cpu().numpy().reshape(-1, 2); p0r = r["p0r"].cpu().numpy().reshape(-1, 2)
    st1 = r["st1"].cpu().numpy().reshape(-1); st0 = r["st0"].cpu().numpy().reshape(-1)
    st1c, st0c = st1c.reshape(-1), st0c.reshape(-1)
    out["status_agree"] = float(np.mean(np.concatenate([st1 == st1c, st0 == st0c])))
    both = (st1 == 1) & (st1c == 1)
    d = np.abs(p1 - p1c.reshape(-1, 2)).max(1)
    out["pos_within_0.01"] = float(np.mean(d[both] <= 0.01)) if both.any() else None
    out["pos_max_abs_diff_px"] = float(d[both].max()) if both.any() else None
    bothb = (st0 == 1) & (st0c == 1)
    db = np.abs(p0r - p0rc.reshape(-1, 2)).max(1)
    out["backward_pos_within_0.01"] = float(np.mean(db[bothb] <= 0.01)) if bothb.any() else None
    distc = np.hypot(*np.abs(p0.reshape(-1, 2) - p0rc.reshape(-1, 2)).T)
    out["fb_valid_agree"] = float(np.mean((r["dist"].cpu().numpy() < 1) == (distc < 1)))
    out["points"] = int(p0.shape[0])
    out["criteria"] = "BASELINE: pyramid bit-exact; status >= 0.995; positions within 0.01 px >= 0.99; corner overlap >= 0.99"
    return out


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sequence", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="issue every step on one stream (no overlap between steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    steps = max(1, args.steps)

    import torch
    if args.impl == "reference":
        if rank != 0:
            return 0
        return main_reference(args, steps, max(0, args.warmup))
    warmup = max(3, args.warmup)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from iceberg_tracking_code_b200 import _native
    _native.lib()                                   # libibt.so as build() left it; raises when it was not built
    numa_node = _native.bind_to_gpu_numa_node(local_rank) if os.environ.get("IBT_NO_NUMA_BIND") is None else None
    from iceberg_tracking_code_b200 import cv
    from iceberg_tracking_code_b200.tracking import SequenceTracker

    # ---- setup (untimed): frames on device, per-frame seeds, pyramids ------------------------------------------
    frames = make_frames(dev)
    grays = [cv.cvtColor(f, cv.COLOR_BGR2GRAY) for f in frames]
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    pts, gftt_ms = [], []
    for g in grays:
        cv.goodFeaturesToTrack(g, **GFTT)
        t0.record()
        p = cv.goodFeaturesToTrack(g, **GFTT)
        t1.record(); torch.cuda.synchronize()
        gftt_ms.append(t0.elapsed_time(t1))
        assert p is not None and p.shape[0] == NPTS, "synthetic scene must yield %d corners" % NPTS
        pts.append(p.reshape(NPTS, 2).contiguous())
    trk = SequenceTracker(GFTT, LK, count_iterations=True)
    pipe = PairPipeline(trk, dev, frames[0])
    # a full (generation-2) collection of CPython's cyclic GC walks every container object of the process -- ~0.1 s with torch
    # imported -- and fires at arbitrary points: one of them inside a 50 ms timed region (seen at N = 8: max over ranks) is a
    # host stall, not a property of the path.  Everything alive now is moved out of the collector's sight; the timed regions
    # below additionally run with the collector off and collect explicitly between them.
    gc.collect(); gc.freeze()
    # the form the frame loop uses (ibt_gftt_async: both launches enqueued, count left on the device, no host round trip)
    gftt_async_ms = []
    for k in range(4):
        t0.record()
        pf = trk.gftt_prefetch(pipe.pyr[0], None)
        t1.record(); torch.cuda.synchronize()
        gftt_async_ms.append(t0.elapsed_time(t1))
        assert int(pf[2][0]) == NPTS
        trk._unpin(pf[2])
    if args.no_pipeline:
        pipe.streams[1] = pipe.streams[0]
    nlev = pipe.pyr[0].maxLevel + 1
    own_launches_per_step = 1 + nlev + 1          # gray, one fused pyrDown+Scharr launch per level, fused LK fwd+bwd+FB
    main_stream = torch.cuda.current_stream()

    def run_region(pipe_, n, first=0, iter_total=None):
        """n pipelined steps bracketed by events on the main stream; returns the elapsed ms"""
        torch.cuda.synchronize()
        pipe_.prime(frames[pingpong(first)])
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(SPIN_CYCLES)
        e0.record(main_stream)
        for s in pipe_.streams:
            s.wait_event(e0)
        timed_steps(pipe_, frames, pts, first, n, iter_total)
        pipe_.join(main_stream)
        e1.record(main_stream)
        return e0, e1

    # ---- warm-up ----------------------------------------------------------------------------------------------------------
    run_region(pipe, warmup)
    torch.cuda.synchronize()

    # ---- timed region: device-resident inputs ---------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    trk.iter_total.zero_()
    gc.collect(); gc.disable()
    sampler.start()
    e0, e1 = run_region(pipe, steps, 0, trk.iter_total)
    sampler.sample_now()                       # the GPU is still working through the queued steps
    torch.cuda.synchronize()
    gc.enable()
    if dist is not None:
        dist.barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    iters = int(trk.iter_total.item())
    last = steps - 1                            # PairPipeline.step(last) wrote p1 / fbd[last & 1] and pyramid slot last % 3
    alive_frac = float((pipe.fbd[last & 1] < 1).float().mean().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pipe.p1[last & 1], pipe.fbd[last & 1], pipe.pyr[last % 3])

    # ---- the same loop returning what cv2 returns: status + err of both passes (OpenCV's level-0 residual stage) ----------
    pipe_se = PairPipeline(trk, dev, frames[0], want_status_err=True)
    if args.no_pipeline:
        pipe_se.streams[1] = pipe_se.streams[0]
    n_se = steps
    run_region(pipe_se, 6); torch.cuda.synchronize()
    e0, e1 = run_region(pipe_se, n_se)
    torch.cuda.synchronize()
    ms_se = e0.elapsed_time(e1) / n_se
    del pipe_se

    # ---- roofline of the HBM-bound part: the whole per-frame prepare (cvtColor + all pyramid levels with Scharr planes),
    # issued alone on one stream, CUDA events around every prepare and around its level-0 launch --------------------------
    n_k1 = 60
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_k1)]
    probes = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_k1)]
    torch.cuda._sleep(int(3e7))                 # ~15 ms spin: the host enqueues every prepare before the GPU starts on them
    for k in range(n_k1 + 4):                   # whole prepare, launches back to back (no events inside the chain)
        j = k - 4
        if j >= 0:
            ev[j][0].record()
        trk.prepare(frames[pingpong(k)], reuse=pipe.pyr[k % 3])
        if j >= 0:
            ev[j][1].record()
    torch.cuda.synchronize()
    torch.cuda._sleep(int(3e7))
    for k in range(n_k1):                       # once more with events around the level-0 launch
        trk.prepare(frames[pingpong(k)], reuse=pipe.pyr[k % 3], probe=probes[k])
    torch.cuda.synchronize()
    prep_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    k1_ms = float(np.mean([a.elapsed_time(b) for a, b in probes]))

    # ---- e2e: public API, pinned host frames, H2D + D2H inside the timed region ----------------------------------------
    host_frames = [f.cpu().pin_memory() for f in frames]
    h_p1 = [torch.empty((NPTS, 2), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_fbd = [torch.empty((NPTS,), dtype=torch.float32).pin_memory() for _ in range(2)]
    d2h_done = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_loop(n, first):
        pipe.prime(frames[pingpong(first)])
        handles = {first: trk.upload(host_frames[pingpong(first + 1)])}
        if n > 1:
            handles[first + 1] = trk.upload(host_frames[pingpong(first + 2)])
        acc = 0.0
        for k in range(n):
            i = first + k
            s = pipe.step(i, handles.pop(i), pts[pingpong(i)])
            if k + 2 < n:
                handles[i + 2] = trk.upload(host_frames[pingpong(i + 3)])      # two uploads in flight on the copy stream
            with torch.cuda.stream(pipe.streams[s]):
                h_p1[s].copy_(pipe.p1[s], non_blocking=True); h_fbd[s].copy_(pipe.fbd[s], non_blocking=True)
                d2h_done[s].record(pipe.streams[s])
            if k >= 1:                      # the caller consumes step i-1's result while step i runs
                d2h_done[s ^ 1].synchronize()
                acc += float(h_fbd[s ^ 1][0])
        d2h_done[(first + n - 1) & 1].synchronize()
        acc += float(h_fbd[(first + n - 1) & 1][0])
        return acc
    n_e2e = steps
    e2e_loop(max(3, warmup // 2) * 2, 0)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    gc.collect(); gc.disable()
    tw0 = time.perf_counter()
    e2e_loop(n_e2e, 0)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - tw0) * 1e3            # wall clock around host-visible results (>= any device-side figure)
    gc.enable()
    h2d = int(host_frames[0].numel())
    d2h = int(h_p1[0].numel() * 4 + h_fbd[0].numel() * 4)

    # ---- from files: every step starts from the JPEG bytes the reference reads at s1:310 (host memory).  Every rank runs its
    # own stream (weak scaling); the aggregate uses the slowest rank's time.  3.8 MB instead of 72 MB cross PCIe per step.
    from_files = None
    try:
        if dist is not None:
            dist.barrier()
        from_files = run_from_files(trk, pipe, pts, host_frames, steps, cv, dev)
    except ImportError as e:                        # Pillow missing on the box: the section is skipped, not faked
        from_files = {"skipped": repr(e)}
    if dist is not None and "ms_per_step" in from_files:
        tf = torch.tensor([from_files["ms_per_step"]], dtype=torch.float64, device=dev)
        dist.all_reduce(tf, op=dist.ReduceOp.MAX)
        from_files["ms_per_step"] = float(tf.item())
        from_files["value"] = world * NPTS / (from_files["ms_per_step"] * 1e-3)

    # ---- parity on the timed frames (N = 1) and the CPU rows need the host copies; free the rest first ---------------------
    parity = None
    if world == 1:
        parity = run_parity(frames, grays, pts, trk, dev)
    frames_np = grays_np = pts_np = None
    if world == 1 and not args.no_cpu_baseline:
        frames_np = [f.numpy() for f in host_frames]
        grays_np = [g.cpu().numpy() for g in grays]
        pts_np = [p.cpu().numpy().reshape(-1, 1, 2) for p in pts]
    del pipe, frames, grays, host_frames
    torch.cuda.empty_cache()

    # ---- sharded sequence (strong scaling, gather inside the timed region) --------------------------------------------------
    seq = None
    if not args.no_sequence:
        seq = run_sharded_sequence(dev, rank, world, dist)

    # ---- reduce over ranks (max time) -------------------------------------------------------------------------------------
    if dist is not None:
        t = torch.tensor([ms, e2e_ms, k1_ms, prep_ms, ms_se], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms, k1_ms, prep_ms, ms_se = [float(v) for v in t.tolist()]
        it_t = torch.tensor([iters], dtype=torch.int64, device=dev)
        dist.all_reduce(it_t)
        iters = int(it_t.item())
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:                               # noqa: BLE001
        pass
    peak, peak_src = (peaks["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs") if "hbm_gbs" in peaks else (6650.0, "fallback 6.65 TB/s")
    n0 = H * W
    lev = [(H, W)]
    for _ in range(nlev - 1):
        lev.append(((lev[-1][0] + 1) // 2, (lev[-1][1] + 1) // 2))
    npx = [h * w for h, w in lev]
    # SURVEY 8(d): K0 reads 3 B + writes 1 B per pixel; K1 reads every level once, writes levels >= 1 and 4 B of Scharr per pixel
    prep_bytes = 4 * n0 + sum(npx) + sum(npx[1:]) + 4 * sum(npx)
    k1_bytes = n0 + 4 * n0 + npx[1]                # level 0 alone: read level 0 once, write (dx,dy) int16, write level 1
    achieved = prep_bytes / (prep_ms * 1e-3) / 1e9
    value = world * NPTS * steps / (ms * 1e-3)
    out = {
        "metric": METRIC, "value": value, "unit": "points/s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32 fixed point + f32 2x2 solve", "data": "synthetic",
        "config": CONFIG,
        "timed_steps": steps, "timed_region_ms": ms,
        "numa_node_rank0": numa_node,
        "pipelining": "none (one stream)" if args.no_pipeline else "consecutive (independent) frame pairs overlap on two CUDA streams, three pyramid slots",
        "frame_pairs_per_s": world * steps / (ms * 1e-3),
        "feature_pair_iterations_per_s": iters / (ms * 1e-3),
        "iterations_per_point_pair": iters / (world * NPTS * steps),
        "fb_valid_fraction_last_step": alive_frac,
        "with_status_err": {"ms_per_step": ms_se, "value": world * NPTS / (ms_se * 1e-3), "unit": "points/s", "steps": n_se,
                            "note": "same step with st/err buffers of both passes passed (what cv2 returns, s1:323,326): "
                                    "adds OpenCV's level-0 bounds test and residual"},
        "gftt_ms": float(np.median(gftt_ms)),
        "gftt_async_ms": float(np.median(gftt_async_ms[1:])),
        "gpu_launches": own_launches_per_step * steps,
        "clocks": clocks,
        "e2e_rgb_frames": {"value": world * NPTS * n_e2e / (e2e_ms * 1e-3), "unit": "points/s", "h2d_bytes_per_step": h2d,
                           "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / n_e2e, "steps": n_e2e,
                           "api": "SequenceTracker.upload/prepare + fused LK (ibt_lk_fb), pinned host RGB frames (the array "
                                  "np.array(Image.open(f)) returns, s1:310), p1 + FB distance read back to the host every step; "
                                  "wall clock.  PCIe-bound: 72 MB per step"},
        "roofline": {"kernel": "per-frame prepare: gray_c3_vec_kernel + pyr_level_tma_kernel x %d levels (fused pyrDown + Scharr)" % nlev,
                     "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "peak_source": peak_src, "bytes_per_launch": prep_bytes, "avg_launch_ms": prep_ms, "traffic": None,
                     "launches": 1 + nlev,
                     "level0": {"kernel": "pyr_level_tma_kernel<deriv,down,4> level 0", "bytes_per_launch": k1_bytes,
                                "avg_launch_ms": k1_ms, "achieved": k1_bytes / (k1_ms * 1e-3) / 1e9,
                                "frac": k1_bytes / (k1_ms * 1e-3) / 1e9 / peak}},
        "lk": {"kernel": "lk_kernel<31,31> (fwd+bwd+FB, warp per point)", "bound": "instruction issue (not HBM, not tensor)",
               "iterations_per_s": iters / (ms * 1e-3), "target_iterations_per_s": 200e6,
               "share_of_step": "see profiles/ launch list"},
    }
    # the declared end-to-end number starts where the reference's loop starts: the JPEG file of s1:310 in host memory
    if from_files is not None and "value" in from_files:
        out["from_files"] = from_files
        out["e2e"] = {k: from_files[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "ms_per_step", "steps", "api")}
        out["e2e"]["input"] = "JPEG bytes of every new frame in host memory (what the reference opens at s1:310); decode on the GPU"
    else:
        if from_files is not None:
            out["from_files"] = from_files
        out["e2e"] = dict(out["e2e_rgb_frames"])
        out["e2e"]["input"] = "decoded RGB frames in pinned host memory"
    if seq is not None:
        out["sharded_sequence"] = seq
    if parity is not None:
        out["parity"] = parity
    traffic_file = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(traffic_file):
        try:
            tf = json.load(open(traffic_file))
            out["roofline"]["traffic"] = tf.get("dram_bytes_per_prepare", tf.get("dram_bytes_per_launch"))
            out["roofline"]["traffic_source"] = tf.get("source")
            out["lk"]["ncu"] = tf.get("lk")
            # issue roofline of the dominant kernel: warp-instructions per point pair (ncu, same kernel) x the point pairs per
            # second measured in this run, against 4 issue slots per SM per clock at the SM clock sampled in this run
            ipp = (tf.get("lk") or {}).get("p1_fbdist_only", {}).get("warp_instructions_per_point_pair")
            mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz")
            if ipp and mhz:
                ach = ipp * (value / world)                       # per GPU
                pk = 148 * 4 * mhz * 1e6
                out["lk"]["issue_roofline"] = {"bound": "instruction issue", "achieved": ach, "peak": pk, "unit": "warp-instructions/s",
                                               "frac": ach / pk, "note": "whole step time in the denominator (LK is ~92 % of it)"}
        except Exception:                           # noqa: BLE001
            pass
    if frames_np is not None:
        cb, _, _ = run_cpu(frames_np, grays_np, pts_np, steps=100, warmup=1, budget_s=12.0)
        c1, _, _ = run_cpu(frames_np, grays_np, pts_np, steps=3, warmup=0, budget_s=8.0, threads=1)
        cb["one_thread"] = {"value": c1["value"], "unit": "points/s", "cores": 1, "sample": c1["sample"]}
        out["cpu_baseline"] = cb
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main_reference(args, steps, warmup):
    """Reference arm: the CPU path of the reference on this box's host cores, same config / metric / unit / steps / warmup."""
    import torch
    from iceberg_tracking_code_b200 import synthetic as syn
    dev = "cuda" if torch.cuda.is_available() else "cpu"          # frame SYNTHESIS only; the timed path is pure CPU
    base = syn.base_texture(H, W, SEED, device=dev)
    frames_np = [syn.frame_rgb(base, t, seed=SEED).cpu().numpy() for t in range(NFRAMES)]
    del base
    step, m, kind, cores, desc = cpu_step_fn()
    grays_np = [m.cvtColor(f, 6) for f in frames_np]
    pts_np = []
    for g in grays_np:
        p = m.goodFeaturesToTrack(g, **GFTT)
        pts_np.append(np.ascontiguousarray(p, np.float32).reshape(-1, 1, 2))
    cb, done, t_total = run_cpu(frames_np, grays_np, pts_np, steps=steps, warmup=warmup)
    out = {
        "impl": "reference", "metric": METRIC,
        "value": cb["value"], "unit": "points/s", "n_gpus": args.gpus, "steps": done, "warmup": warmup,
        "ms_per_step": t_total / done * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/int16 fixed point + f32 (OpenCV CPU)", "data": "synthetic",
        "config": CONFIG,
        "reference_calls": "cv2.cvtColor + cv2.calcOpticalFlowPyrLK fwd + bwd + numpy FB (s1:311,323,326,329-333)",
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
