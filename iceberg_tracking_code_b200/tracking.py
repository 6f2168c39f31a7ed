"""The reference's frame loop on the GPU, behind the reference's own worker signatures.

    SequenceTracker            device-resident state of one tracking group (seed frame + track_len pairs)
    track_sequence(...)        s1_lucaskanade_tracking.py:296-450 (loop, FB prune, group save, re-seed)
    lucaskanade_tracking(...)  s1_lucaskanade_tracking.py:234-236 (same positional arguments)
    LucasKanade(...).run()     s0_1_test_lucaskanade_tracking.py:29-181 (same constructor, same printed counts)

What differs from the reference by design (SURVEY.md Appendix C "N"): every frame's pyramid + Scharr planes are
built once and cached (the reference rebuilds them 4x per pair inside cv2); forward LK, backward LK and the FB check
are one kernel launch; tracks live in time-major device arrays with an alive mask and become the (M,T+1,2)/(M,T)
float32 arrays of the .npz file by one compaction at the group boundary instead of per-track Python lists.
Plotting, movie making and JPEG deletion (s1:397-434, 452-479) are outside the hot path and are not implemented.
"""
import ctypes as C
import datetime as dt
import glob
import os
import os.path as osp

import numpy as np
import torch

from . import _native as N
from . import cv

# s1_lucaskanade_tracking.py:240-248 == s0_1_test_lucaskanade_tracking.py:37-45
FEATURE_PARAMS = dict(maxCorners=50000000, qualityLevel=0.007, minDistance=10, blockSize=10)
LK_PARAMS = dict(winSize=(35, 35), maxLevel=4,
                 criteria=(cv.TERM_CRITERIA_EPS | cv.TERM_CRITERIA_COUNT, 25, 0.03))


def load_image(path):
    """np.array(Image.open(image)) (s1:310): (H,W,3) u8 RGB on the host.  `.npy` frames are accepted too."""
    path = str(path)
    if path.endswith(".npy"):
        return np.load(path)
    from PIL import Image
    return np.array(Image.open(path))


def read_file(path):
    """The compressed frame as it lies on disk (the GPU decodes it: jpeg.py)."""
    with open(str(path), "rb") as f:
        return f.read()


class GpuJpegLoader:
    """loader="gpu": path -> (gray CUDA tensor, ready event, confirm), the handle SequenceTracker.prepare() accepts.
    Two decoders on two high-priority CUDA streams take the frames alternately and never make the host wait
    (jpeg.JpegDecoder.decode_async): a decode is a chain of small latency-bound kernels, so two in flight -- beside the LK
    launch of the pair being tracked, which track_sequence caps at two of its three CTAs per SM -- cost little more than one.
    confirm() must be called before the frame is consumed: it waits for the decode, checks that the speculative Huffman
    pass had converged and returns None, or (gray, event) of a repeated decode."""

    def __init__(self, device, coeffset=0, crop_box=None, reencode=None):
        """crop_box = (left, upper, right, lower) as PIL's Image.crop takes it (camtools.py:79): the decoded plane is cropped
        as a view on the device instead of decoding a cropped, re-encoded copy of the file (SURVEY 8f-1; see
        lucaskanade_tracking(crop="view")).  reencode = (quality, subsampling), e.g. (75, "4:2:0") = Pillow's defaults: the
        cropped RGB view additionally goes through the save-and-reopen round trip of camtools.crop_image_standalone on the GPU
        (ibt_jpeg_recompress), so the gray plane equals that of the re-encoded file bit for bit (crop="emulate")."""
        from . import jpeg as _jpeg
        self.device = device
        self.coeffset = coeffset
        self.crop_box = None if crop_box is None else tuple(int(v) for v in crop_box)
        self.reencode = reencode
        self.decs = [_jpeg.JpegDecoder(device), _jpeg.JpegDecoder(device)]
        self.dec = self.decs[0]
        self.streams = [torch.cuda.Stream(device=device, priority=-1), torch.cuda.Stream(device=device, priority=-1)]
        self.stream = self.streams[0]
        self._n = 0

    def _crop(self, h, dec):
        """decode handle -> the gray plane the tracker takes (enqueued on the current stream)"""
        if self.reencode is not None:
            rgb = h["rgb"]
            if self.crop_box is not None:
                l, u, r, b = self.crop_box
                rgb = rgb[u:b, l:r]                      # a view: the kernel takes the row pitch
            return dec.recompress(rgb, self.reencode[0], self.reencode[1], rgb=False, gray=True, coeffset=self.coeffset)[1]
        gray = h["gray"]
        if self.crop_box is None:
            return gray
        l, u, r, b = self.crop_box
        return gray[u:b, l:r].contiguous()

    def stage(self, path, index):
        """read + stage + parse the file for the decoder that will take frame `index` (worker threads)"""
        return self.decs[index & 1].stage(path)

    def decode(self, data=None, staged=None):
        k = self._n & 1
        self._n += 1
        dec, st = self.decs[k], self.streams[k]
        with torch.cuda.device(self.device), torch.cuda.stream(st):
            re = self.reencode is not None
            h = dec.decode_async(data, rgb=re, gray=not re, coeffset=self.coeffset, staged=staged)     # s1:310-311 in one pass
            if re and h["rgb"] is None:
                raise ValueError("crop='emulate' needs colour source frames")
            gray = self._crop(h, dec)
            ev = torch.cuda.Event()
            ev.record(st)

        def confirm():
            with torch.cuda.device(self.device), torch.cuda.stream(st):
                dec.confirm(h)
                if not h.get("redo"):
                    return None
                g2 = self._crop(h, dec)
                e2 = torch.cuda.Event()
                e2.record(st)
            return g2, e2
        return gray, ev, confirm

    def __call__(self, path):
        return self.decode(read_file(path))


class ViewLoader:
    """lucaskanade_tracking(crop="view"): source file -> cropped gray plane decoded on the GPU.  Files the GPU decoder must not
    or cannot take -- a scan that ends early (no EOI marker), a crop box that leaves the frame (PIL pads with zeros), a
    progressive / CMYK / 12-bit file -- are read with Pillow exactly as camtools.crop_image_standalone reads them (truncated
    scans logged to logfile_image_cropping.log, re-read with LOAD_TRUNCATED_IMAGES, announced) and uploaded as pixels."""

    def __init__(self, gpu_loader, crop_box, sources):
        self.gpu = gpu_loader
        self.box = tuple(int(v) for v in crop_box)
        self.sources = sources                            # {name in ws_target: source path}
        self.fallbacks = 0

    def __call__(self, name):
        from . import jpeg as _jpeg
        path = self.sources[name]
        data = read_file(path)
        ok = False
        try:
            info = _jpeg.parse(data)
            l, u, r, b = self.box
            ok = data.rstrip(b'\x00')[-2:] == b'\xff\xd9' and 0 <= l < r <= info.width and 0 <= u < b <= info.height
        except (_jpeg.Unsupported, RuntimeError):
            ok = False
        if ok:
            return self.gpu.decode(data)
        from ._crop import open_cropped
        self.fallbacks += 1
        img = open_cropped(path, name, self.box)
        if getattr(self.gpu, "reencode", None) is not None:   # crop="emulate": the reference's save + reopen, in memory
            import io
            from PIL import Image
            buf = io.BytesIO()
            img.save(buf, format="JPEG")
            buf.seek(0)
            return np.array(Image.open(buf))
        return np.array(img.convert("RGB"))


class FrameStager:
    """Pinned double buffer + copy stream: the host->device copy of frame t+1 overlaps the kernels of frame t."""

    def __init__(self, device):
        self.device = device
        self.copy_stream = torch.cuda.Stream(device=device)
        self._pinned = [None, None]
        self._k = 0

    def upload(self, frame):
        """host (H,W,C) u8 numpy / torch CPU tensor -> device tensor, asynchronously on the copy stream.
        Returns (device_tensor, event); wait on the event before consuming.  A tensor that is already pinned is
        copied straight from its own memory (the caller keeps it alive and unchanged until the event fires)."""
        t = torch.from_numpy(np.ascontiguousarray(frame)) if isinstance(frame, np.ndarray) else frame.contiguous()
        if t.is_pinned():
            host = t
            free_ev = None
        else:
            k = self._k
            self._k ^= 1
            buf = self._pinned[k]
            if buf is None or buf[0].shape != t.shape:
                buf = (torch.empty(t.shape, dtype=torch.uint8).pin_memory(), torch.cuda.Event())
                self._pinned[k] = buf
            host, free_ev = buf
            free_ev.synchronize()                # the previous copy out of this pinned buffer has finished
            host.copy_(t)
        with torch.cuda.stream(self.copy_stream):
            dev = host.to(self.device, non_blocking=True)
            if free_ev is not None:
                free_ev.record(self.copy_stream)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        return dev, ev


class SequenceTracker:
    """Device-side state of the tracking loop.  One instance per GPU."""

    def __init__(self, feature_params=None, lk_params=None, fb_threshold=1.0, device=None, count_iterations=False):
        self.feature_params = dict(FEATURE_PARAMS if feature_params is None else feature_params)
        self.lk_params = dict(LK_PARAMS if lk_params is None else lk_params)
        self.fb_threshold = float(fb_threshold)
        self.device = cv._device() if device is None else torch.device(device)
        self.stager = FrameStager(self.device)
        self.iter_total = torch.zeros((1,), dtype=torch.int64, device=self.device) if count_iterations else None
        self.n = 0                 # seeds of the current group
        self.steps = 0             # pairs tracked in the current group
        self.T = 0
        self._tracks = self._quality = self._alive = None
        # prepare + goodFeaturesToTrack of upcoming frames (track_sequence); high priority: its CTAs take the SM slots that the
        # persistent LK launch frees while its last warps finish, ahead of the next LK launch
        self.side = torch.cuda.Stream(device=self.device, priority=-1)
        self._pinned = {}          # free pinned host buffers by size (results travel D2H asynchronously)
        self._ws = None            # private goodFeaturesToTrack workspace (one call in flight per tracker)

    # -- frames ---------------------------------------------------------------------------------------
    def upload(self, frame):
        """Start the host->device copy of a frame on the copy stream; pass the returned handle to prepare()."""
        return self.stager.upload(frame)

    def prepare(self, frame, reuse=None, probe=None):
        """frame (H,W,3|4) u8 RGB (host numpy / device tensor / upload() handle) or (H,W) u8 gray -> FramePyramid with
        derivatives = np.array(Image.open(...)) upload + cv2.cvtColor (s1:310-311) + the pyramids cv2 builds inside LK.
        reuse: a FramePyramid of the same frame size to rebuild in place; its gray plane is reused too, so the steady
        state allocates nothing (and streams never share allocator blocks)."""
        with torch.cuda.device(self.device):
            if isinstance(frame, tuple):
                handle = frame
            elif isinstance(frame, np.ndarray) or (isinstance(frame, torch.Tensor) and not frame.is_cuda):
                handle = self.stager.upload(frame)
            else:
                handle = None
            if handle is not None:
                frame, ev = handle[0], handle[1]
                torch.cuda.current_stream().wait_event(ev)
                frame.record_stream(torch.cuda.current_stream())
            if frame.ndim == 3:
                own = getattr(reuse, "_own_gray", None) if reuse is not None else None
                if own is not None and tuple(own.shape) != tuple(frame.shape[:2]):
                    own = None
                gray = cv.cvtColor(frame, cv.COLOR_BGR2GRAY, dst=own)
            else:
                gray = frame
            if reuse is not None:
                pyr = reuse.rebuild(gray, probe)
            else:
                pyr = cv.FramePyramid(gray, self.lk_params["winSize"], self.lk_params["maxLevel"], True)
            if frame.ndim == 3:
                pyr._own_gray = gray
            return pyr

    # -- group life cycle -----------------------------------------------------------------------------
    def _pin(self, shape, dtype):
        """pinned host tensor from the tracker's pool (give it back with _unpin)"""
        key = (tuple(shape), dtype)
        lst = self._pinned.get(key)
        if lst:
            return lst.pop()
        return torch.empty(shape, dtype=dtype).pin_memory()

    def _unpin(self, t):
        self._pinned.setdefault((tuple(t.shape), t.dtype), []).append(t)

    def gftt_prefetch(self, pyr, mask=None):
        """Enqueue cv2.goodFeaturesToTrack(frame_gray, mask=mask, **feature_params) (s1:437) of a frame that will seed a
        group, on the CURRENT stream, without waiting for it (ibt_gftt_async): returns the handle seed(prefetched=) takes.
        track_sequence issues it on the side stream one frame ahead, so the corners are ready when the group starts."""
        fp = self.feature_params
        harris, hk = (1 if fp.get("useHarrisDetector", False) else 0), float(fp.get("k", 0.04))
        q, md, bs = float(fp["qualityLevel"]), float(fp["minDistance"]), int(fp.get("blockSize", 3))
        if not (q > 0) or md < 0:
            raise cv.error("goodFeaturesToTrack: qualityLevel must be > 0 and minDistance >= 0")
        gsize = cv._aperture(fp.get("gradientSize", 3), "goodFeaturesToTrack", "gradientSize")
        img = pyr.levels[0]
        H, W = img.shape
        if H < 3 or W < 3:
            return None
        m = None
        if mask is not None:
            m = cv._to_dev(mask, np.uint8, "goodFeaturesToTrack mask")
            if tuple(m.shape) != (H, W):
                raise cv.error("goodFeaturesToTrack: mask must be (H,W) u8 of the image size")
        nbytes = N.lib().ibt_gftt_workspace_bytes(H, W)
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty((nbytes,), dtype=torch.uint8, device=self.device)
        maxc = int(fp["maxCorners"])
        cap = H * W // 4 + 4096
        if 0 < maxc < cap:
            cap = maxc
        out = torch.empty((cap, 2), dtype=torch.float32, device=self.device)
        cnt = torch.zeros((1,), dtype=torch.int32, device=self.device)
        p = cv._ptr
        N.check(N.lib().ibt_gftt_async_ksize(p(img), img.stride(0), p(m), W, H, W, maxc, q, md, bs, gsize, harris, hk,
                                             p(self._ws), self._ws.numel(), p(out), cap, p(cnt), cv._stream()),
                "ibt_gftt_async_ksize")
        # (nout, error) of the workspace counters (GfttCounters: maxbits, ncand, nsel, nacc, nout, error): a capacity overflow
        # raised on the device must not pass as "no corners"
        h = self._pin((2,), torch.int32)
        h.copy_(self._ws[16:24].view(torch.int32), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        return out, cnt, h, ev

    def seed(self, pyr, mask=None, track_len=2, points=None, prefetched=None):
        """Re-seed (s1:437-448): Shi-Tomasi corners of the frame (or the given (N,1,2) points) start a new group.
        prefetched: handle of gftt_prefetch() for this frame (the corners were computed ahead on another stream)."""
        if prefetched is not None:
            out, _cnt, h, ev = prefetched
            ev.synchronize()                              # (issued a frame ago: normally long finished)
            n, err = int(h[0]), int(h[1])
            self._unpin(h)
            N.check(err, "ibt_gftt_async_ksize")
            torch.cuda.current_stream().wait_event(ev)
            out.record_stream(torch.cuda.current_stream())
            p = out[:n] if n else None
        elif points is None:
            p = cv.goodFeaturesToTrack(pyr.levels[0], mask=mask, **self.feature_params)
        else:
            p = cv._to_dev(points, np.float32, "seed points")
        self.T = int(track_len)
        self.steps = 0
        self.n = 0 if p is None else p.numel() // 2
        n = self.n
        if n == 0:
            self._tracks = self._quality = self._alive = None
            return 0
        self._tracks = torch.empty((self.T + 1, n, 2), dtype=torch.float32, device=self.device)
        self._tracks[0] = p.reshape(n, 2)
        self._quality = torch.zeros((self.T, n), dtype=torch.float32, device=self.device)
        self._alive = torch.ones((n,), dtype=torch.uint8, device=self.device)
        return n

    def track(self, prev_pyr, cur_pyr):
        """One frame pair (s1:313-359): LK forward, LK backward, FB distance, prune -- one kernel launch."""
        if self.n == 0:
            return
        if self.steps >= self.T:
            raise RuntimeError("group is full: seed() again (the reference re-seeds every track_len frames, s1:362)")
        t = self.steps
        cnt, eps = cv._criteria(self.lk_params["criteria"])
        w = self.lk_params["winSize"]
        p = cv._ptr
        if torch.cuda.current_device() != self.device.index:
            raise RuntimeError("SequenceTracker was created for %s but cuda:%d is current (wrap the loop in torch.cuda.device)"
                               % (self.device, torch.cuda.current_device()))
        N.check(N.lib().ibt_lk_fb(C.byref(prev_pyr.c), C.byref(cur_pyr.c), p(self._tracks[t]), self.n, int(w[0]), int(w[1]),
                                  cnt, eps, float(self.lk_params.get("minEigThreshold", 1e-4)), self.fb_threshold,
                                  p(self._tracks[t + 1]), None, None, None, None, None, p(self._quality[t]),
                                  p(self._alive), None, p(self.iter_total), cv._stream()), "ibt_lk_fb")
        self.steps += 1

    def harvest(self, to_host=True):
        """Surviving tracks of the current group: tracks (M, steps+1, 2) f32, trackquality (M, steps) f32 in seed order
        (what np.savez receives at s1:395).  M == 0 -> two empty (0,) float64 arrays, like np.array([])."""
        empty = (np.zeros((0,), np.float64), np.zeros((0,), np.float64))
        if self.n == 0:
            return empty
        if self.steps == 0:
            tr = self._tracks[0].reshape(self.n, 1, 2)
            q = torch.zeros((self.n, 0), dtype=torch.float32, device=self.device)
            return (tr.cpu().numpy(), q.cpu().numpy()) if to_host else (tr, q)
        n, k = self.n, self.steps
        scratch = torch.empty((n + 1,), dtype=torch.int32, device=self.device)
        out_t = torch.empty((n, k + 1, 2), dtype=torch.float32, device=self.device)
        out_q = torch.empty((n, k), dtype=torch.float32, device=self.device)
        cnt = C.c_int(0)
        p = cv._ptr
        N.check(N.lib().ibt_tracks_compact(p(self._tracks), p(self._quality), p(self._alive), n, k, p(scratch), p(out_t),
                                           p(out_q), C.byref(cnt), cv._stream()), "ibt_tracks_compact")
        m = cnt.value
        if m == 0:
            return empty
        if to_host:
            return out_t[:m].cpu().numpy(), out_q[:m].cpu().numpy()
        return out_t[:m], out_q[:m]

    def harvest_async(self):
        """harvest() without waiting: compaction and the device->host copies of the current group are enqueued on the
        current stream; finalize(handle) returns the arrays later (track_sequence finalises a group while the next one
        is being tracked)."""
        if self.n == 0 or self.steps == 0:
            return ("done", self.harvest())
        n, k = self.n, self.steps
        scratch = torch.empty((n + 1,), dtype=torch.int32, device=self.device)
        out_t = torch.empty((n, k + 1, 2), dtype=torch.float32, device=self.device)
        out_q = torch.empty((n, k), dtype=torch.float32, device=self.device)
        p = cv._ptr
        N.check(N.lib().ibt_tracks_compact_async(p(self._tracks), p(self._quality), p(self._alive), n, k, p(scratch), p(out_t),
                                                 p(out_q), cv._stream()), "ibt_tracks_compact_async")
        h_t, h_q, h_m = self._pin((n, k + 1, 2), torch.float32), self._pin((n, k), torch.float32), self._pin((1,), torch.int32)
        h_t.copy_(out_t, non_blocking=True); h_q.copy_(out_q, non_blocking=True); h_m.copy_(scratch[n:], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        return ("pending", h_t, h_q, h_m, ev, out_t, out_q)

    def finalize(self, handle, with_device=False):
        """-> (tracks (M, steps+1, 2) f32, trackquality (M, steps) f32) of a harvest_async() handle (M == 0: two (0,) f64).
        with_device=True appends the device-resident copies (tracks, quality) -- or None for an empty group -- which the
        multi-GPU gather sends without going through the host again."""
        if handle[0] == "done":
            return handle[1] + ((None,) if with_device else ())
        _tag, h_t, h_q, h_m, ev, out_t, out_q = handle
        ev.synchronize()
        m = int(h_m[0])
        if m == 0:
            res = (np.zeros((0,), np.float64), np.zeros((0,), np.float64))
            dev = None
        else:
            res = (h_t[:m].numpy().copy(), h_q[:m].numpy().copy())
            dev = (out_t[:m], out_q[:m])
        self._unpin(h_t); self._unpin(h_q); self._unpin(h_m)
        return res + ((dev,) if with_device else ())

    def alive_count(self):
        return 0 if self.n == 0 else int(self._alive.sum().item())


# -----------------------------------------------------------------------------------------------------
def npz_name(seed_path, track_len, track_len_sec):
    """s1:394 -- note path.split('.')[0] (kept: dotted directory names break it in the reference too)."""
    return '{}_{}sec_at_{}sec_tracks.npz'.format(str(seed_path).split('.')[0], track_len * track_len_sec, track_len_sec)


def group_time_ok(paths, track_len_sec):
    """s1:368-390: every consecutive gap of the group's frames must be track_len_sec + {-2..2} s, parsed from
    '%Y%m%d-%H%M%S.jpg' names; uses timedelta.seconds like the reference."""
    times = [dt.datetime.strptime(osp.basename(str(p)), '%Y%m%d-%H%M%S.jpg') for p in paths]
    for a, b in zip(times[:-1], times[1:]):
        if (b - a).seconds not in [track_len_sec - 2, track_len_sec - 1, track_len_sec, track_len_sec + 1, track_len_sec + 2]:
            return False
    return True


def track_sequence(imagelist, mask, track_len, track_len_sec, startlist=(0,), feature_params=None, lk_params=None,
                   save=True, loader=load_image, tracker=None, check_time=True, on_group=None, first_group=0,
                   n_groups=None, decode_workers=4, device_results=None):
    """The loop of s1:296-450 over `imagelist` (paths, or in-memory frames when loader is None).
    Returns the list of (seed_index, npz_path_or_None, tracks, trackquality) of every completed group.

    first_group / n_groups select a contiguous block of groups (time-block sharding, SURVEY 8e): group g of start s
    covers frames s+g*T .. s+(g+1)*T; a block needs one halo frame shared with the next block.

    loader: callable path -> (H,W,3) u8 RGB host array (default: Pillow, as the reference, s1:310), None for in-memory
    frames, or the string "gpu": the file bytes go to the GPU compressed and csrc/jpeg.cu decodes them (bit-exact with
    Pillow) straight into the gray plane; files it does not handle raise jpeg.Unsupported.

    device_results: a dict; if given, {seed_index: (tracks, trackquality) CUDA tensors} of every non-empty group is left
    in it (sharding.gather_results sends those instead of re-uploading the host arrays).

    decode_workers: a host loader (PIL JPEG decode, ~0.25 s per 24 MP frame, far slower than the GPU step) runs in a
    thread pool that keeps `decode_workers` frames ahead of the tracker; the order of processing is unchanged.  Ignored
    by the "gpu" loader (its decode is pipelined on a CUDA stream instead)."""
    T = int(track_len)
    trk = tracker or SequenceTracker(feature_params, lk_params)
    if isinstance(loader, str):
        if loader != "gpu":
            raise ValueError("loader must be a callable, None or 'gpu'")
        if getattr(trk, "_gpu_loader", None) is None:      # pinned staging, workspace and stream live as long as the tracker
            trk._gpu_loader = GpuJpegLoader(trk.device)
        loader = trk._gpu_loader
    gpu = loader if isinstance(loader, GpuJpegLoader) else None
    host_loader = None if gpu is not None else loader               # what the thread pool runs
    if mask is not None:
        mask = cv._to_dev(mask, np.uint8, "mask")
    results = []
    for start in startlist:
        frames = imagelist[start:]
        total_groups = max(0, (len(frames) - 1) // T)
        g0 = first_group
        g1 = total_groups if n_groups is None else min(total_groups, first_group + n_groups)
        if g1 <= g0:
            continue
        prev = None
        seed_idx = None
        counters = range(g0 * T, g1 * T + 1)
        pool, futures = None, {}
        if gpu is not None and decode_workers:
            # the GPU decoder's host side (file read, copy into pinned memory, marker parsing: ~2 ms per 24 MP frame) runs on two
            # worker threads, four frames ahead; frames must reach the two decoders alternately, in order
            from concurrent.futures import ThreadPoolExecutor
            pool = ThreadPoolExecutor(max_workers=2)
            gpu._n = 0
            for i, c in enumerate(counters[:4]):
                futures[c] = pool.submit(gpu.stage, frames[c], i)
        elif host_loader is not None and gpu is None and decode_workers and decode_workers > 1:
            from concurrent.futures import ThreadPoolExecutor
            pool = ThreadPoolExecutor(max_workers=int(decode_workers))
            for c in counters[:decode_workers]:
                futures[c] = pool.submit(host_loader, frames[c])

        def fetch(c):
            """frame c as prepare() takes it (host array, device tensor, or (device tensor, event) from the GPU decoder)"""
            if pool is not None and gpu is not None:
                nxt = c + 4
                if nxt <= counters[-1]:
                    futures[nxt] = pool.submit(gpu.stage, frames[nxt], nxt - counters[0])
                return gpu.decode(staged=futures.pop(c).result())
            if pool is not None:
                nxt = c + decode_workers
                if nxt <= counters[-1]:
                    futures[nxt] = pool.submit(host_loader, frames[nxt])
                data = futures.pop(c).result()
            elif gpu is not None:
                return gpu(frames[c])             # file -> pinned staging -> device -> gray plane, on the decoder's stream
            else:
                data = host_loader(frames[c]) if host_loader is not None else frames[c]
            return data

        # ---- pipelined loop.  Side stream: gray + pyramid of frame c+1 (and goodFeaturesToTrack if it seeds a group) are
        # issued BEFORE the LK launch of frame c on the main stream, so they fill the SMs that a persistent LK launch leaves
        # idle while its last warps finish.  Four pyramid slots: slot (c+1) % 4 was last read by the LK launch of frame c-2.
        # A finished group is compacted and copied to pinned host memory asynchronously and finalised (np.savez, callbacks)
        # one group later.  The order of all arithmetic is that of the reference loop.
        on_gpu = gpu is not None or isinstance(loader, ViewLoader)
        LOOK = 2 if on_gpu else 1                         # frames prepared ahead (two decoders work in parallel)
        NSLOT = LOOK + 3
        if on_gpu:
            cv.set_lk_resident_ctas(2)                    # the JPEG decodes of the next frames share the SMs with the tracker
            from . import jpeg as _jpeg
            _jpeg.set_probe(False)                        # decode latency hides behind the tracker: no full-grid probe kernel
        main = torch.cuda.current_stream()
        side = trk.side
        slots = getattr(trk, "_slots", None)
        if slots is None or len(slots) != NSLOT:
            slots = trk._slots = [None] * NSLOT
        lk_done = [None] * NSLOT
        side.wait_stream(main)

        def is_seed(c):
            return (c - g0 * T) % T == 0 and c < g1 * T

        def build_on_side(c, data):
            k = c % NSLOT
            with torch.cuda.stream(side):
                if lk_done[k] is not None:
                    side.wait_event(lk_done[k])
                reuse = slots[k]
                pyr = None
                if reuse is not None:
                    try:
                        pyr = trk.prepare(data, reuse=reuse)
                    except cv.error:                      # frame size changed: build a fresh pyramid
                        pyr = None
                if pyr is None:
                    pyr = trk.prepare(data)
                slots[k] = pyr
                pyr.levels[0].record_stream(main)         # (a decoder-owned gray plane is read by the LK launches on `main`)
                pf = trk.gftt_prefetch(pyr, mask) if is_seed(c) else None
                ev = torch.cuda.Event()
                ev.record(side)
            return pyr, ev, pf

        def prepare_ahead(c):
            data = fetch(c)
            conf = data[2] if isinstance(data, tuple) and len(data) > 2 else None
            return build_on_side(c, data) + (conf, c)

        def confirmed(item):
            """the frame's GPU decode had converged -- else its pyramid (and corners) are rebuilt from the repeated decode"""
            pyr, ev, pf, conf, c = item
            if conf is not None:
                again = conf()
                if again is not None:
                    pyr, ev, pf = build_on_side(c, again)
            return pyr, ev, pf

        pending = []                                      # (seed_idx, ok, path, harvest handle) of groups not finalised yet

        def finalize_oldest():
            sidx, ok, path, handle = pending.pop(0)
            tracks, quality, dev = trk.finalize(handle, with_device=True)
            if ok and device_results is not None and dev is not None:
                device_results[start + sidx] = dev
            if ok and path is not None:
                np.savez(path, tracks=tracks, trackquality=quality)
            if ok:
                results.append((start + sidx, path, tracks, quality))
                if on_group is not None:
                    on_group(start + sidx, tracks, quality)

        try:
            queue = [prepare_ahead(c) for c in counters[:LOOK]]
            for counter in counters:
                cur, ev_cur, pf_cur = confirmed(queue.pop(0))
                # the next frames are fetched and prepared now: GPU decode / upload / pyramid build overlap this frame's kernels
                if counter + LOOK <= counters[-1]:
                    queue.append(prepare_ahead(counter + LOOK))
                main.wait_event(ev_cur)
                if prev is not None and trk.n > 0:
                    trk.track(prev, cur)
                if prev is not None:
                    e = torch.cuda.Event()
                    e.record(main)
                    lk_done[(counter - 1) % NSLOT] = e        # frame counter-1 has been read for the last time
                if (counter - g0 * T) % T == 0:
                    if seed_idx is not None:
                        ok = True
                        if check_time and loader is not None:
                            ok = group_time_ok(frames[counter - T: counter + 1], track_len_sec)
                        path = npz_name(frames[seed_idx], T, track_len_sec) if (ok and save and loader is not None) else None
                        pending.append((seed_idx, ok, path, trk.harvest_async()))
                        if len(pending) > 1:
                            finalize_oldest()
                    if counter < g1 * T:
                        trk.seed(cur, mask, T, prefetched=pf_cur)
                        seed_idx = counter
                prev = cur
            while pending:
                finalize_oldest()
        finally:
            if pool is not None:
                pool.shutdown(wait=False)
            main.wait_stream(side)
            if on_gpu:
                cv.set_lk_resident_ctas(0)
                _jpeg.set_probe(True)
    return results


def lucaskanade_tracking(file_path, ws_source, ws_target, camname, track_len, track_len_sec, startlist, mask_switch,
                         plot_switch, movie_switch, delete_jpgs_switch, paramfile_path, n_proc, camera=None, crop="reencode"):
    """Same positional signature as s1_lucaskanade_tracking.py:234-236; side effect = the .npz files of SURVEY A.8.
    `camera` (keyword, optional) injects a ready camera.Camera instead of reading `paramfile_path`.
    plot_switch / movie_switch are accepted and ignored (matplotlib / mencoder work, out of scope); delete_jpgs_switch == 1
    removes the cropped copies after tracking like the reference (s1:475-479).

    crop="reencode" (default) is the reference: every source frame is decoded, cropped and re-saved as a JPEG by Pillow
    (camtools.py:237-258, ~0.3 s of host time per 24 MP frame) and the tracker reads those files -- the lossy re-encode is
    part of the pixels the reference tracks, so this is the mode whose tracks equal the reference's.
    crop="emulate" gives the SAME tracks without that pre-pass and without the cropped copies: the source files are decoded on
    the GPU, cropped as a view and sent through the save-and-reopen round trip as integer arithmetic (RGB->YCbCr, 4:2:0 box
    filter, islow FDCT, quality-75 quantisation, dequantisation, islow IDCT, fancy upsampling, YCbCr->RGB: ibt_jpeg_recompress,
    bit-exact with Pillow's save + open), ~0.1 ms per 24 MP frame instead of ~0.3 s.
    crop="view" (SURVEY 8f-1) decodes the SOURCE files on the GPU and crops the plane as a view: no host decode, no
    re-encode, no second generation of JPEG loss -- tracks differ slightly from the reference's by construction; the .npz
    files are named after <ws_target>/<frame>.jpg exactly as in the other mode."""
    from .camera import Camera
    ws_source, ws_target = str(ws_source), str(ws_target)
    datestring = osp.basename(ws_source)
    cam = camera or Camera(camname=camname, date=datestring, paramfile_path=paramfile_path, mask=mask_switch)
    imagelist = sorted(glob.glob(ws_source + '/*.jpg'))
    if len(imagelist) <= track_len:                                    # s1:262
        return
    if not osp.isdir(ws_target):
        os.makedirs(ws_target)
    from . import jpeg as _jpeg
    if crop in ("view", "emulate"):
        l, u, r, b = (int(v) for v in cam.crop_box())
        h, w = b - u, r - l
        if mask_switch == 1:
            mask = cam.mask_image(h, w)
        else:
            mask = np.full((h, w), 255, np.uint8)
        tracker = SequenceTracker()
        sources = {osp.join(ws_target, osp.basename(p)): p for p in imagelist}
        gpu = GpuJpegLoader(tracker.device, crop_box=(l, u, r, b), reencode=(75, "4:2:0") if crop == "emulate" else None)
        track_sequence(sorted(sources), mask, track_len, track_len_sec, startlist, tracker=tracker,
                       loader=ViewLoader(gpu, (l, u, r, b), sources), decode_workers=0)
        return                                                         # (no cropped copies were written: nothing to delete)
    if crop != "reencode":
        raise ValueError("crop must be 'reencode', 'emulate' or 'view'")
    cam.crop_image_parallel(imagelist, ws_target, n_proc)              # s1:272
    imagelist = sorted(glob.glob(ws_target + '/*.jpg'))                # s1:278
    info = _jpeg.parse(read_file(imagelist[0]))
    h, w = info.height, info.width
    if mask_switch == 1:                                               # s1:285-294
        mask = cam.mask_image(h, w)
    else:
        mask = np.full((h, w), 255, np.uint8)
    # the cropping step above re-saved every frame with Pillow (baseline JPEG): the GPU decoder handles all of them
    track_sequence(imagelist, mask, track_len, track_len_sec, startlist, loader="gpu")
    if delete_jpgs_switch == 1:                                        # s1:475-479: delete the cropped .jpgs to open up space
        for img in imagelist:
            os.remove(img)


class LucasKanade:
    """s0_1_test_lucaskanade_tracking.py:29-181 without the plots: same constructor, same printed track counts,
    `self.tracks` ends up as the same list of lists of (x, y) vertices."""

    def __init__(self, workspace, detect_interval, time_spacing, loader="gpu"):
        """loader: "gpu" (frames decoded by csrc/jpeg.cu) or a callable path -> RGB array such as load_image (Pillow)."""
        from pathlib import Path
        self.loader = loader
        workspace = Path(workspace)
        self.detect_interval = detect_interval
        self.time_spacing = time_spacing
        self.feature_params = dict(FEATURE_PARAMS)
        self.lk_params = dict(LK_PARAMS)
        self.track_len = self.detect_interval
        self.tracks = []
        self.imagelist = sorted(workspace.glob('*.jpg'))
        self.distthreshold = 1.0
        self.mask = 0
        self.date = workspace.parts[-1]
        self.workspace = workspace
        self.track_counts = []

    def run(self):
        trk = SequenceTracker(self.feature_params, self.lk_params, fb_threshold=self.distthreshold)
        prev = None
        loader = GpuJpegLoader(trk.device) if self.loader == "gpu" else self.loader
        for counter, image in enumerate(self.imagelist):
            frame = loader(image)
            if isinstance(frame, tuple) and len(frame) > 2:      # GPU decode: confirm it before the frame is used
                frame = frame[2]() or frame[:2]
            cur = trk.prepare(frame)
            if prev is not None and trk.n > 0:
                trk.track(prev, cur)
            if counter % self.detect_interval == 0:
                n_alive = trk.alive_count() if counter > 0 else 0
                self.track_counts.append(n_alive)
                print('{} tracks'.format(n_alive))
                trk.seed(cur, None, self.track_len)      # mask is all-255 in the reference (s0_1:73-74)
            prev = cur
            self.prev_gray = cur.levels[0]
            print('{} / {} done...'.format(counter + 1, len(self.imagelist)))
        tracks, _ = trk.harvest()
        self.tracks = [[(x, y) for x, y in tr] for tr in tracks] if tracks.ndim == 3 else []
