"""Drop-in replacements for the three OpenCV calls on the reference's tracking hot path, with cv2's
signatures, shapes, dtypes and None conventions (SURVEY.md 8b), running on sm_100a kernels through libibt.so.

    cvtColor                 s1_lucaskanade_tracking.py:283,311   s0_1_test_lucaskanade_tracking.py:71,80
    goodFeaturesToTrack      s1:437                               s0_1:167
    calcOpticalFlowPyrLK     s1:323,326                           s0_1:92,95
    buildOpticalFlowPyramid / pyrDown / cornerMinEigenVal         (inside the above; exposed as test hooks)

Inputs may be numpy arrays (copied to the GPU, results come back as numpy, like cv2) or torch CUDA tensors
(results stay on the device).  There is no CPU fallback: without a CUDA device or libibt.so these raise.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N

COLOR_BGR2GRAY = 6
COLOR_RGB2GRAY = 7
COLOR_BGRA2GRAY = 10          # cv2 computes these exactly like 6 / 7 (3 or 4 channels in, alpha ignored)
COLOR_RGBA2GRAY = 11
TERM_CRITERIA_COUNT = 1
TERM_CRITERIA_MAX_ITER = 1
TERM_CRITERIA_EPS = 2
OPTFLOW_USE_INITIAL_FLOW = 4
OPTFLOW_LK_GET_MIN_EIGENVALS = 8


class error(Exception):
    """Raised where cv2 raises cv2.error (bad dtype / shape / argument)."""


def _device():
    if not torch.cuda.is_available():
        raise RuntimeError("iceberg_tracking_code_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _is_np(a):
    return isinstance(a, np.ndarray)


def _to_dev(a, dtype, what):
    """numpy / torch -> contiguous CUDA tensor of `dtype` (no dtype conversion: mismatch is an error)."""
    if _is_np(a):
        if a.dtype != dtype:
            raise error("%s: expected %s, got %s" % (what, np.dtype(dtype).name, a.dtype.name))
        return torch.from_numpy(np.ascontiguousarray(a)).to(_device(), non_blocking=False)
    if isinstance(a, torch.Tensor):
        want = {np.uint8: torch.uint8, np.float32: torch.float32}[dtype]
        if a.dtype != want:
            raise error("%s: expected %s, got %s" % (what, want, a.dtype))
        if not a.is_cuda:
            a = a.to(_device())
        return a.contiguous()
    raise error("%s: expected a numpy array or torch tensor, got %r" % (what, type(a)))


def _out(t, as_numpy):
    return t.cpu().numpy() if as_numpy else t


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


# ---------------------------------------------------------------------------------------------------
def cvtColor(src, code=COLOR_BGR2GRAY, dst=None, dstCn=0, *, coeffset=0):
    """cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY) (s1:311), positional order of cv2's cvtColor(src, code[, dst[, dstCn]]).
    (H,W,3|4) u8 -> (H,W) u8.  Channel 0 gets the 0.114 weight whatever it holds; the reference feeds PIL's RGB array under
    the BGR code and that quirk is kept.
    coeffset (keyword only) 0 = OpenCV 4.x 15-bit coefficients, 1 = OpenCV 3.x 14-bit (SURVEY A.1).
    dst: preallocated contiguous (H,W) u8 CUDA tensor to write into (steady-state loops allocate nothing)."""
    if dstCn not in (0, 1):
        raise error("cvtColor: a gray conversion has one destination channel")
    if code not in (COLOR_BGR2GRAY, COLOR_RGB2GRAY, COLOR_BGRA2GRAY, COLOR_RGBA2GRAY):
        raise error("cvtColor: only COLOR_BGR2GRAY / COLOR_RGB2GRAY / COLOR_BGRA2GRAY / COLOR_RGBA2GRAY are implemented")
    code = {COLOR_BGRA2GRAY: COLOR_BGR2GRAY, COLOR_RGBA2GRAY: COLOR_RGB2GRAY}.get(code, code)
    as_np = _is_np(src)
    s = _to_dev(src, np.uint8, "cvtColor src")
    if s.ndim != 3 or s.shape[2] not in (3, 4):
        raise error("cvtColor: Bad number of channels (expected (H,W,3) or (H,W,4), got %s)" % (tuple(s.shape),))
    if code == COLOR_RGB2GRAY:
        s = s[..., [2, 1, 0] + ([3] if s.shape[2] == 4 else [])].contiguous()
    H, W, cn = s.shape
    if dst is None:
        dst = torch.empty((H, W), dtype=torch.uint8, device=s.device)
    elif not (isinstance(dst, torch.Tensor) and dst.is_cuda and dst.dtype == torch.uint8 and tuple(dst.shape) == (H, W)
              and dst.is_contiguous()):
        raise error("cvtColor: dst must be a contiguous (H,W) u8 CUDA tensor")
    if H and W:
        N.check(N.lib().ibt_gray_u8(_ptr(s), H, W, cn, W * cn, _ptr(dst), W, int(coeffset), _stream()), "ibt_gray_u8")
    return _out(dst, as_np)


def pyrDown(src):
    """cv2.pyrDown(u8 (H,W)) -> ((H+1)//2, (W+1)//2) u8 (SURVEY A.2)."""
    as_np = _is_np(src)
    s = _to_dev(src, np.uint8, "pyrDown src")
    if s.ndim != 2:
        raise error("pyrDown: expected a single-channel (H,W) u8 image")
    H, W = s.shape
    dst = torch.empty(((H + 1) // 2, (W + 1) // 2), dtype=torch.uint8, device=s.device)
    N.check(N.lib().ibt_pyr_level_u8(_ptr(s), H, W, W, None, 0, _ptr(dst), dst.shape[1], _stream()), "ibt_pyr_level_u8")
    return _out(dst, as_np)


def _round_up(v, m):
    return (v + m - 1) // m * m


def _frame_dev(img, what):
    """(H,W,C) u8 frame -> CUDA tensor whose pixels are interleaved (strides (pitch, C, 1)); a device view with a row pitch (a
    crop) is used as it is, anything else is made contiguous."""
    f = img if isinstance(img, torch.Tensor) and img.is_cuda and img.dtype == torch.uint8 else _to_dev(img, np.uint8, what)
    if f.ndim == 3 and f.shape[0] > 0 and not (f.stride(2) == 1 and f.stride(1) == f.shape[2]
                                               and f.stride(0) >= f.shape[1] * f.shape[2]):
        f = f.contiguous()
    return f


class FramePyramid:
    """Device-resident Gaussian pyramid (+ Scharr derivative planes) of one frame, as the LK solver consumes it.
    Built ONCE per frame and reused as `next` of pair t-1, `prev` of pair t and by both FB directions (the reference
    rebuilds it four times per pair inside cv2.calcOpticalFlowPyrLK; SURVEY Appendix C).  Accepted by
    calcOpticalFlowPyrLK in place of an image, like cv2 accepts buildOpticalFlowPyramid's output.
    A gray (H,W) frame gives levels[l] (h,w) u8 and derivs[l] (h,w,2) int16.  An (H,W,C) frame, C = 2..4, gives one pyramid
    per channel plane (what cv2 builds for it): levels[l] (C,h,w) u8 and derivs[l] (C,h,w,2) int16, planar; `cn` is C."""

    def __init__(self, gray, winSize=(21, 21), maxLevel=3, withDerivatives=True):
        colour = hasattr(gray, "ndim") and gray.ndim == 3
        if colour and not (2 <= gray.shape[2] <= 4):
            raise error("FramePyramid: a multi-channel frame is (H,W,C) u8 with C = 2..4, got %s" % (tuple(gray.shape),))
        g = _frame_dev(gray, "FramePyramid frame") if colour else _to_dev(gray, np.uint8, "FramePyramid gray")
        if g.ndim not in (2, 3) or g.shape[0] < 1 or g.shape[1] < 1:
            raise error("FramePyramid: expected a single-channel (H,W) or an (H,W,C) u8 image")
        if not (0 <= int(maxLevel) < N.IBT_MAX_LEVELS):
            raise error("FramePyramid: maxLevel must be in [0, %d]" % (N.IBT_MAX_LEVELS - 1))
        self.winSize = (int(winSize[0]), int(winSize[1]))
        self.with_derivs = bool(withDerivatives)
        self.cn = int(g.shape[2]) if colour else 1
        H, W = g.shape[:2]
        sizes = (C.c_int * (2 * N.IBT_MAX_LEVELS))()
        ml = N.lib().ibt_pyramid_levels(H, W, self.winSize[0], self.winSize[1], int(maxLevel), sizes)
        if ml < 0:
            N.check(ml, "ibt_pyramid_levels")
        self.maxLevel = ml
        self.sizes = [(sizes[2 * l], sizes[2 * l + 1]) for l in range(ml + 1)]
        if colour:
            self._init_planes(g)
            return
        dev = g.device
        g = self._level0(g)
        self._img_buf = [g]
        self._deriv_buf = []
        self.levels = [g]
        self.derivs = []
        st = N.ibt_pyramid_t()
        st.nlevels = ml + 1
        for l, (h, w) in enumerate(self.sizes):
            if l > 0:
                pitch = _round_up(w, 128)
                buf = torch.empty((h, pitch), dtype=torch.uint8, device=dev)
                self._img_buf.append(buf)
                self.levels.append(buf[:, :w])
            else:
                pitch = g.stride(0)
            st.rows[l], st.cols[l] = h, w
            st.img[l] = self._img_buf[l].data_ptr()
            st.img_pitch[l] = pitch
            if self.with_derivs:
                dpitch = _round_up(w * 4, 128)
                dbuf = torch.empty((h, dpitch // 2), dtype=torch.int16, device=dev)
                self._deriv_buf.append(dbuf)
                self.derivs.append(dbuf[:, :2 * w].unflatten(1, (w, 2)))
                st.deriv[l] = dbuf.data_ptr()
                st.deriv_pitch[l] = dpitch
        self.c = st
        self._build(None)

    def _init_planes(self, frame):
        """one ibt_pyramid_t per channel plane; every level of every channel (level 0 too: it is de-interleaved from the frame)
        in buffers of 128-byte row pitch"""
        cn, dev = self.cn, frame.device
        self._img_buf, self._deriv_buf, self.levels, self.derivs = [], [], [], []
        self.chans = [N.ibt_pyramid_t() for _ in range(cn)]
        for st in self.chans:
            st.nlevels = self.maxLevel + 1
        for l, (h, w) in enumerate(self.sizes):
            pitch = _round_up(w, 128)
            buf = torch.empty((cn, h, pitch), dtype=torch.uint8, device=dev)
            self._img_buf.append(buf)
            self.levels.append(buf[:, :, :w])
            if self.with_derivs:
                dpitch = _round_up(w * 4, 128)
                dbuf = torch.empty((cn, h, dpitch // 2), dtype=torch.int16, device=dev)
                self._deriv_buf.append(dbuf)
                self.derivs.append(dbuf[:, :, :2 * w].unflatten(2, (w, 2)))
            for c, st in enumerate(self.chans):
                st.rows[l], st.cols[l] = h, w
                st.img[l] = buf[c].data_ptr()
                st.img_pitch[l] = pitch
                if self.with_derivs:
                    st.deriv[l] = self._deriv_buf[l][c].data_ptr()
                    st.deriv_pitch[l] = dpitch
        self.c = None
        self.chan_ptrs = (C.POINTER(N.ibt_pyramid_t) * cn)(*[C.pointer(st) for st in self.chans])
        self._build_planes(frame, None)

    def _build_planes(self, frame, probe):
        if probe is not None:
            probe[0].record()
        N.check(N.lib().ibt_pyramid_build_multichannel(_ptr(frame), frame.stride(0), self.cn, self.chan_ptrs,
                                                       1 if self.with_derivs else 0, _stream()), "ibt_pyramid_build_multichannel")
        if probe is not None:
            probe[1].record()

    def level(self, l):
        """level l in cv2's layout: (h,w) u8, or (h,w,C) u8 for a multi-channel frame"""
        return self.levels[l] if self.cn == 1 else self.levels[l].permute(1, 2, 0)

    def deriv(self, l):
        """Scharr planes of level l in cv2's layout: (h,w,2) int16 (dx, dy), or (h,w,2C) int16 with channel c's (dx, dy) at
        [2c, 2c+1]"""
        if self.cn == 1:
            return self.derivs[l]
        d = self.derivs[l]
        return d.permute(1, 2, 0, 3).reshape(d.shape[1], d.shape[2], 2 * self.cn)

    def _level0(self, g):
        """Level 0 is the caller's gray image itself when its rows are 16-byte aligned (the TMA staging paths need that);
        otherwise it is copied once into a row-padded buffer (view [:, :W]) so that odd widths also take the fast paths."""
        H, W = g.shape
        if W % 16 == 0 and g.data_ptr() % 16 == 0:
            return g
        pad = getattr(self, "_l0_pad", None)
        if pad is None or pad.shape[0] != H:
            pad = torch.empty((H, _round_up(W, 128)), dtype=torch.uint8, device=g.device)
            self._l0_pad = pad
        view = pad[:, :W]
        view.copy_(g)
        return view

    def _build(self, probe):
        if probe is None:
            N.check(N.lib().ibt_pyramid_build(C.byref(self.c), 1 if self.with_derivs else 0, _stream()), "ibt_pyramid_build")
            return
        # same launches issued level by level so that CUDA events can bracket the level-0 launch (bench.py roofline)
        c, L = self.c, self.maxLevel + 1
        for l in range(L):
            if l == 0:
                probe[0].record()
            N.check(N.lib().ibt_pyr_level_u8(c.img[l], c.rows[l], c.cols[l], c.img_pitch[l],
                                             c.deriv[l] if self.with_derivs else None, c.deriv_pitch[l],
                                             c.img[l + 1] if l + 1 < L else None, c.img_pitch[l + 1] if l + 1 < L else 0,
                                             _stream()), "ibt_pyr_level_u8")
            if l == 0:
                probe[1].record()

    def rebuild(self, gray, probe=None):
        """Recompute this pyramid in place for another frame of the same size (no allocation: steady-state loop).
        probe = (start_event, end_event) records CUDA events around the level-0 launch (multi-channel frames: around the
        whole build, which is one call)."""
        if self.cn > 1:
            f = _frame_dev(gray, "FramePyramid frame")
            if tuple(f.shape) != tuple(self.sizes[0]) + (self.cn,):
                raise error("FramePyramid.rebuild: frame size or channel count changed")
            self._build_planes(f, probe)
            return self
        g = _to_dev(gray, np.uint8, "FramePyramid gray")
        if tuple(g.shape) != tuple(self.sizes[0]):
            raise error("FramePyramid.rebuild: frame size changed")
        g = self._level0(g)
        self._img_buf[0] = g
        self.levels[0] = g
        self.c.img[0] = g.data_ptr()
        self.c.img_pitch[0] = g.stride(0)
        self._build(probe)
        return self

    @property
    def shape(self):
        return self.sizes[0]

    def nbytes(self):
        return sum(b.numel() * b.element_size() for b in self._img_buf + self._deriv_buf)


def buildOpticalFlowPyramid(img, winSize, maxLevel, withDerivatives=True):
    """cv2.buildOpticalFlowPyramid -> (maxLevelOut, [L0, D0, L1, D1, ...]) (SURVEY A.3): levels (h,w) u8,
    derivatives (h,w,2) int16 (dx, dy); an (H,W,C) frame, C = 2..4, gives cv2's (h,w,C) u8 levels and (h,w,2C) int16
    derivatives (channel c's dx, dy at 2c, 2c+1).  cv2 returns views into padded buffers; these are plain arrays."""
    as_np = _is_np(img)
    p = FramePyramid(img, winSize, maxLevel, withDerivatives)
    out = []
    for l in range(p.maxLevel + 1):
        out.append(_out(p.level(l).contiguous(), as_np))
        if withDerivatives:
            out.append(_out(p.deriv(l).contiguous(), as_np))
    return p.maxLevel, out


# ---------------------------------------------------------------------------------------------------
def _criteria(criteria):
    typ, cnt, eps = criteria
    typ = int(typ)
    if not (typ & TERM_CRITERIA_COUNT):
        cnt = 30
    if not (typ & TERM_CRITERIA_EPS):
        eps = 0.01
    return int(cnt), float(eps)


def _as_pyramid(img, winSize, maxLevel, need_derivs, what):
    if isinstance(img, FramePyramid):
        if img.winSize != (int(winSize[0]), int(winSize[1])):
            raise error("%s: pyramid was built for winSize %s, call uses %s" % (what, img.winSize, tuple(winSize)))
        if need_derivs and not img.with_derivs:
            raise error("%s: pyramid has no derivative planes" % what)
        return img
    if hasattr(img, "ndim") and img.ndim == 3 and img.shape[2] == 1:      # (H,W,1) is a single-channel image for cv2 as well
        img = img[..., 0]
    return FramePyramid(img, winSize, maxLevel, need_derivs)


def _channels(img):
    """a FramePyramid's cn; 1 for an (H,W) / (H,W,1) image, C for an (H,W,C) image"""
    if isinstance(img, FramePyramid):
        return img.cn
    if not hasattr(img, "ndim") or img.ndim != 3:
        return 1
    return int(img.shape[2])


def calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, nextPts=None, status=None, err=None, winSize=(21, 21), maxLevel=3,
                         criteria=(TERM_CRITERIA_COUNT | TERM_CRITERIA_EPS, 30, 0.01), flags=0, minEigThreshold=1e-4,
                         *, return_iters=False):
    """cv2.calcOpticalFlowPyrLK(img0, img1, p0, None, **lk_params) (s1:323,326; SURVEY A.5), positional order of cv2's
    calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, nextPts[, status[, err[, winSize[, maxLevel[, criteria[, flags[,
    minEigThreshold]]]]]]]); status / err are cv2's optional output placeholders: results are always returned, never written there.
    Returns (nextPts, status (N,1) u8, err (N,1) f32); nextPts has prevPts' shape; N == 0 -> (None, None, None).
    err is 0 where status == 0 (cv2 leaves uninitialised memory there).  prevImg / nextImg may be FramePyramid
    objects.  return_iters=True appends the (N,) int32 count of inner iterations executed per point."""
    cn = _channels(prevImg)
    if cn != _channels(nextImg):
        raise error("calcOpticalFlowPyrLK: prevImg and nextImg differ in the number of channels")
    if cn > 4:
        raise error("calcOpticalFlowPyrLK: at most 4 channels")
    as_np = _is_np(prevPts)
    if as_np and prevPts.dtype != np.float32:
        raise error("calcOpticalFlowPyrLK: prevPts must be float32 (cv2 asserts the same)")
    pts = _to_dev(prevPts, np.float32, "calcOpticalFlowPyrLK prevPts")
    shp = tuple(pts.shape)
    if pts.numel() == 0:
        return (None, None, None) + ((None,) if return_iters else ())
    if pts.numel() % 2 != 0 or shp[-1] != 2:
        raise error("calcOpticalFlowPyrLK: prevPts must be (N,1,2) or (N,2) float32")
    pts = pts.reshape(-1, 2)
    n = pts.shape[0]
    w = (int(winSize[0]), int(winSize[1]))
    if not (3 <= w[0] <= N.IBT_MAX_WIN and 3 <= w[1] <= N.IBT_MAX_WIN):
        raise error("calcOpticalFlowPyrLK: winSize components must be in [3, %d]" % N.IBT_MAX_WIN)
    if maxLevel < 0:
        raise error("calcOpticalFlowPyrLK: maxLevel must be >= 0")
    cnt, eps = _criteria(criteria)
    # (H,W,C) u8 frames, C = 2..4 (cv2 takes 3-channel frames; the reference converts to gray first, s1:311): one pyramid per
    # channel plane, window sums taken over pixels and channels
    pI = _as_pyramid(prevImg, w, maxLevel, True, "calcOpticalFlowPyrLK prevImg")
    pJ = _as_pyramid(nextImg, w, maxLevel, False, "calcOpticalFlowPyrLK nextImg")
    if pI.sizes[0] != pJ.sizes[0]:
        raise error("calcOpticalFlowPyrLK: prevImg and nextImg differ in size")
    if pI.maxLevel != pJ.maxLevel:
        raise error("calcOpticalFlowPyrLK: pyramids differ in depth")
    flags = int(flags)
    if flags & OPTFLOW_USE_INITIAL_FLOW:
        if nextPts is None:
            raise error("calcOpticalFlowPyrLK: OPTFLOW_USE_INITIAL_FLOW needs nextPts")
        nxt = _to_dev(nextPts, np.float32, "calcOpticalFlowPyrLK nextPts").reshape(-1, 2).clone()
        if nxt.shape[0] != n:
            raise error("calcOpticalFlowPyrLK: nextPts and prevPts differ in length")
    else:
        nxt = torch.empty((n, 2), dtype=torch.float32, device=pts.device)
    st = torch.empty((n,), dtype=torch.uint8, device=pts.device)
    err = torch.empty((n,), dtype=torch.float32, device=pts.device)
    iters = torch.empty((n,), dtype=torch.int32, device=pts.device) if return_iters else None
    if cn == 1:
        N.check(N.lib().ibt_lk(C.byref(pI.c), C.byref(pJ.c), _ptr(pts), _ptr(nxt), n, w[0], w[1], cnt, eps,
                               float(minEigThreshold), flags, _ptr(st), _ptr(err), _ptr(iters), _stream()), "ibt_lk")
    else:
        N.check(N.lib().ibt_lk_multichannel(pI.chan_ptrs, pJ.chan_ptrs, cn, _ptr(pts), _ptr(nxt), n, w[0], w[1], cnt, eps, float(minEigThreshold),
                                            flags, _ptr(st), _ptr(err), _ptr(iters), _stream()), "ibt_lk_multichannel")
    res = (_out(nxt.reshape(shp), as_np), _out(st.reshape(n, 1), as_np), _out(err.reshape(n, 1), as_np))
    return res + ((_out(iters, as_np),) if return_iters else ())


def calcOpticalFlowPyrLK_FB(prev, next, p0, winSize=(21, 21), maxLevel=3,
                            criteria=(TERM_CRITERIA_COUNT | TERM_CRITERIA_EPS, 30, 0.01), minEigThreshold=1e-4,
                            fb_threshold=1.0, alive=None, iter_total=None, return_iters=False):
    """The reference's whole per-pair block in one launch (s1:323-333), on gray or (H,W,C) frames (C = 2..4) or FramePyramids:
        p1, st, err  = calcOpticalFlowPyrLK(prev, next, p0, None, **lk_params)
        p0r, st, err = calcOpticalFlowPyrLK(next, prev, p1, None, **lk_params)
        dist = hypot(|p0 - p0r|); valid = dist < 1
    Returns a dict with p1, st1, err1, p0r, st0, err0, dist, valid (and iters (N,2) when asked).  `alive`
    (torch u8 (N,), device) is updated in place when given: dead points are skipped, survivors &= valid."""
    as_np = _is_np(p0)
    pts = _to_dev(p0, np.float32, "calcOpticalFlowPyrLK_FB p0")
    shp = tuple(pts.shape)
    if pts.numel() == 0:
        return None
    pts = pts.reshape(-1, 2)
    n = pts.shape[0]
    w = (int(winSize[0]), int(winSize[1]))
    pA = _as_pyramid(prev, w, maxLevel, True, "calcOpticalFlowPyrLK_FB prev")
    pB = _as_pyramid(next, w, maxLevel, True, "calcOpticalFlowPyrLK_FB next")
    if pA.sizes != pB.sizes:
        raise error("calcOpticalFlowPyrLK_FB: prev and next differ in size")
    if pA.cn != pB.cn:
        raise error("calcOpticalFlowPyrLK_FB: prev and next differ in the number of channels")
    cnt, eps = _criteria(criteria)
    dev = pts.device
    f32 = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
    u8 = lambda *s: torch.empty(s, dtype=torch.uint8, device=dev)
    p1, p0r, err1, err0, dist = f32(n, 2), f32(n, 2), f32(n), f32(n), f32(n)
    st1, st0 = u8(n), u8(n)
    own_alive = alive is None
    if own_alive:
        alive = torch.ones((n,), dtype=torch.uint8, device=dev)
    iters = torch.zeros((n, 2), dtype=torch.int32, device=dev) if return_iters else None
    tail = (_ptr(pts), n, w[0], w[1], cnt, eps, float(minEigThreshold), float(fb_threshold), _ptr(p1), _ptr(st1), _ptr(err1),
            _ptr(p0r), _ptr(st0), _ptr(err0), _ptr(dist), _ptr(alive), _ptr(iters), _ptr(iter_total), _stream())
    if pA.cn == 1:
        N.check(N.lib().ibt_lk_fb(C.byref(pA.c), C.byref(pB.c), *tail), "ibt_lk_fb")
    else:
        N.check(N.lib().ibt_lk_fb_multichannel(pA.chan_ptrs, pB.chan_ptrs, pA.cn, *tail), "ibt_lk_fb_multichannel")
    r = dict(p1=_out(p1.reshape(shp), as_np), st1=_out(st1.reshape(n, 1), as_np), err1=_out(err1.reshape(n, 1), as_np),
             p0r=_out(p0r.reshape(shp), as_np), st0=_out(st0.reshape(n, 1), as_np), err0=_out(err0.reshape(n, 1), as_np),
             dist=_out(dist, as_np), valid=_out(alive.bool(), as_np))
    if return_iters:
        r["iters"] = _out(iters, as_np)
    return r


def set_lk_resident_ctas(ctas):
    """Process-wide occupancy cap of the persistent LK launches (ibt_lk_set_max_ctas_per_sm): 0 = fill the SMs (default), 2 =
    leave a third of every SM to kernels of other streams (the GPU JPEG decode of the next frame runs beside the tracker)."""
    N.check(N.lib().ibt_lk_set_max_ctas_per_sm(int(ctas)), "ibt_lk_set_max_ctas_per_sm")


def lk_fb_into(prev, next, p0, lk_params, p1, fbdist, alive=None, iter_total=None):
    """Allocation-free form of calcOpticalFlowPyrLK_FB for steady-state loops: prev / next are FramePyramids with
    derivatives, p0 (N,2) f32, p1 (N,2) f32 and fbdist (N,) f32 are preallocated device tensors; alive (N,) u8 is
    updated in place when given; iter_total (1,) int64 accumulates the inner iterations executed."""
    cnt, eps = _criteria(lk_params["criteria"])
    w = lk_params["winSize"]
    n = p0.shape[0]
    N.check(N.lib().ibt_lk_fb(C.byref(prev.c), C.byref(next.c), _ptr(p0), n, int(w[0]), int(w[1]), cnt, eps,
                              float(lk_params.get("minEigThreshold", 1e-4)), 1.0, _ptr(p1), None, None, None, None, None,
                              _ptr(fbdist), _ptr(alive), None, _ptr(iter_total), _stream()), "ibt_lk_fb")


# ---------------------------------------------------------------------------------------------------
APERTURES = (-1, 1, 3, 5, 7)      # cv2's Sobel apertures of the corner detector: -1 = Scharr


def _aperture(ksize, what, name):
    """cv2's ksize / gradientSize -> int; cv2 also takes odd values up to 31 but documents only these"""
    if isinstance(ksize, bool) or int(ksize) != ksize or int(ksize) not in APERTURES:
        raise error("%s: %s must be one of -1 (Scharr), 1, 3, 5, 7 (got %r)" % (what, name, ksize))
    return int(ksize)


def _corner_src(src, what):
    """the image of the corner family -> (CUDA tensor, is_float): u8 or float32 (cv2: CV_8UC1 || CV_32FC1); any other dtype
    raises like cv2's assertion in corner.cpp"""
    dt = src.dtype if isinstance(src, (np.ndarray, torch.Tensor)) else None
    if dt in (np.float32, torch.float32):
        return _to_dev(src, np.float32, what), True
    if dt is None or dt in (np.uint8, torch.uint8):
        return _to_dev(src, np.uint8, what), False
    raise error("%s: src.type() == CV_8UC1 || src.type() == CV_32FC1 (got %s)" % (what, dt))


def cornerMinEigenVal(src, blockSize, dst=None, ksize=3):
    """cv2.cornerMinEigenVal(src, blockSize[, dst[, ksize]]): u8 or float32 (H,W) -> (H,W) f32 (SURVEY A.6 steps 1-3); dst is
    cv2's output placeholder (the map is returned).  ksize: Sobel aperture -1 (Scharr), 1, 3, 5 or 7.  A float32 image takes
    cv2's CV_32F scale (no factor 255); NaN / inf pixels give NaN / inf responses, as in cv2."""
    ksize = _aperture(ksize, "cornerMinEigenVal", "ksize")
    as_np = _is_np(src)
    s, f32 = _corner_src(src, "cornerMinEigenVal src")
    if s.ndim != 2:
        raise error("cornerMinEigenVal: expected a single-channel (H,W) u8 or float32 image")
    H, W = s.shape
    eig = torch.empty((H, W), dtype=torch.float32, device=s.device)
    if f32:
        N.check(N.lib().ibt_min_eigen_f32src(_ptr(s), H, W, W * 4, int(blockSize), ksize, _ptr(eig), W * 4, _stream()),
                "ibt_min_eigen_f32src")
        return _out(eig, as_np)
    N.check(N.lib().ibt_min_eigen_ksize_f32(_ptr(s), H, W, W, int(blockSize), ksize, _ptr(eig), W * 4, _stream()),
            "ibt_min_eigen_ksize_f32")
    return _out(eig, as_np)


def cornerHarris(src, blockSize, ksize=3, k=0.04):
    """cv2.cornerHarris(u8 (H,W), blockSize, ksize, k) -> (H,W) f32: the response goodFeaturesToTrack(useHarrisDetector=True)
    ranks.  The reference leaves useHarrisDetector at False (s1:240-243); cv2's signature carries it (SURVEY 8b).
    ksize: Sobel aperture -1 (Scharr), 1, 3, 5 or 7.  src may also be float32 (cv2's CV_32F scale, as cornerMinEigenVal)."""
    ksize = _aperture(ksize, "cornerHarris", "ksize")
    as_np = _is_np(src)
    s, f32 = _corner_src(src, "cornerHarris src")
    if s.ndim != 2:
        raise error("cornerHarris: expected a single-channel (H,W) u8 or float32 image")
    H, W = s.shape
    dst = torch.empty((H, W), dtype=torch.float32, device=s.device)
    if f32:
        N.check(N.lib().ibt_corner_harris_f32src(_ptr(s), H, W, W * 4, int(blockSize), ksize, float(k), _ptr(dst), W * 4,
                                                 _stream()), "ibt_corner_harris_f32src")
        return _out(dst, as_np)
    N.check(N.lib().ibt_corner_harris_ksize_f32(_ptr(s), H, W, W, int(blockSize), ksize, float(k), _ptr(dst), W * 4,
                                                _stream()), "ibt_corner_harris_ksize_f32")
    return _out(dst, as_np)


_gftt_ws = {}
_gftt_lock = __import__("threading").Lock()


def _gftt_workspace(dev, H, W):
    """One workspace per device for the cv2-style call, regrown when a larger frame arrives (a SequenceTracker keeps its own:
    tracking.SequenceTracker.gftt_prefetch).  Calls from several host threads on one device must not overlap on a workspace:
    the lock covers the lookup, callers serialise on the stream like any cv2 call."""
    nbytes = N.lib().ibt_gftt_workspace_bytes(H, W)
    cap = H * W // 4 + 4096
    with _gftt_lock:
        ws = _gftt_ws.get(dev.index)
        if ws is None or ws[0].numel() < nbytes or ws[1].shape[0] < cap:
            ws = (torch.empty((nbytes,), dtype=torch.uint8, device=dev), torch.empty((cap, 2), dtype=torch.float32, device=dev))
            _gftt_ws[dev.index] = ws
    return ws


def goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance, corners=None, mask=None, blockSize=3,
                        useHarrisDetector=False, k=0.04, gradientSize=3):
    """cv2.goodFeaturesToTrack(frame_gray, mask=mask, **feature_params) (s1:437; SURVEY A.6), positional order of cv2's
    goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance[, corners[, mask[, blockSize[, useHarrisDetector[, k]]]]])
    (corners is cv2's output placeholder; gradientSize, of cv2's second overload, is the Sobel aperture: -1 (Scharr), 1, 3 (the
    first overload's and the reference's), 5 or 7).
    Returns (K,1,2) float32 integer-valued (x, y) ordered by response, or None when there is no corner
    (callers test `if p is not None`, s1:445).  useHarrisDetector=True ranks cv2.cornerHarris(image, blockSize, gradientSize, k)
    instead of the minimal eigenvalue (the reference never sets it).
    image may also be float32 (cv2's CV_32F scale): an image whose response is not finite everywhere (a NaN / inf pixel, or
    derivative products beyond float range) raises cv.error rather than return corners derived from it."""
    if not (qualityLevel > 0) or minDistance < 0:
        raise error("goodFeaturesToTrack: qualityLevel must be > 0 and minDistance >= 0")
    gradientSize = _aperture(gradientSize, "goodFeaturesToTrack", "gradientSize")
    as_np = _is_np(image)
    img, f32 = _corner_src(image, "goodFeaturesToTrack image")
    if img.ndim != 2:
        raise error("goodFeaturesToTrack: expected a single-channel (H,W) u8 or float32 image")
    H, W = img.shape
    m = None
    if mask is not None:
        m = _to_dev(mask, np.uint8, "goodFeaturesToTrack mask")
        if tuple(m.shape) != (H, W):
            raise error("goodFeaturesToTrack: mask must be (H,W) u8 of the image size")
    if H < 3 or W < 3:
        return None
    ws, out = _gftt_workspace(img.device, H, W)
    cnt = C.c_int(0)
    if f32:
        rc = N.lib().ibt_gftt_f32src(_ptr(img), W * 4, _ptr(m), W, H, W, int(maxCorners), float(qualityLevel),
                                     float(minDistance), int(blockSize), gradientSize, 1 if useHarrisDetector else 0, float(k),
                                     _ptr(ws), ws.numel(), _ptr(out), out.shape[0], C.byref(cnt), _stream())
        if rc == N.IBT_E_UNSUPPORTED:
            raise error("goodFeaturesToTrack: the float32 image gives a non-finite corner response (NaN / inf pixels, or "
                        "derivative products beyond float range)")
        N.check(rc, "ibt_gftt_f32src")
        if cnt.value == 0:
            return None
        return _out(out[:cnt.value].reshape(-1, 1, 2).clone(), as_np)
    rc = N.lib().ibt_gftt_ksize(_ptr(img), W, _ptr(m), W, H, W, int(maxCorners), float(qualityLevel), float(minDistance),
                                int(blockSize), gradientSize, 1 if useHarrisDetector else 0, float(k), _ptr(ws), ws.numel(),
                                _ptr(out), out.shape[0], C.byref(cnt), _stream())
    N.check(rc, "ibt_gftt_ksize")
    if cnt.value == 0:
        return None
    return _out(out[:cnt.value].reshape(-1, 1, 2).clone(), as_np)


def photo_to_utm(xy, cam):
    """Camera.photocords_cropped_to_uncropped + Camera.photo_to_utm for (n,2) float32 vertices
    (imports/camtools.py:414-421, 286-332; SURVEY A.9).  cam: 12 float64 (include/ibt.h).  -> (n,2) float64."""
    as_np = _is_np(xy)
    p = _to_dev(xy, np.float32, "photo_to_utm xy").reshape(-1, 2)
    n = p.shape[0]
    out = torch.empty((n, 2), dtype=torch.float64, device=p.device)
    camv = (C.c_double * 12)(*[float(v) for v in cam])
    N.check(N.lib().ibt_photo_to_utm(_ptr(p), n, camv, _ptr(out), _stream()), "ibt_photo_to_utm")
    return _out(out, as_np)
