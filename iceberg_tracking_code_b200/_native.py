"""ctypes binding of libibt.so (include/ibt.h).  This is the ONLY compute back end of the package:
there is no CPU or PyTorch fallback -- if the library is missing or a call fails, an exception is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libibt.so")

IBT_MAX_LEVELS = 8
IBT_MAX_WIN = 63
IBT_OK, IBT_E_INVALID, IBT_E_CUDA, IBT_E_WORKSPACE, IBT_E_CAPACITY, IBT_E_UNSUPPORTED = 0, -1, -2, -3, -4, -5


class IbtError(RuntimeError):
    def __init__(self, code, where, detail=""):
        self.code = code
        super().__init__("%s failed: %s%s" % (where, _errstr(code), (" -- " + detail) if detail else ""))


class ibt_pyramid_t(C.Structure):
    """HOST mirror of `struct ibt_pyramid` in include/ibt.h."""
    _fields_ = [
        ("nlevels", C.c_int32),
        ("rows", C.c_int32 * IBT_MAX_LEVELS),
        ("cols", C.c_int32 * IBT_MAX_LEVELS),
        ("img", C.c_void_p * IBT_MAX_LEVELS),
        ("img_pitch", C.c_int64 * IBT_MAX_LEVELS),
        ("deriv", C.c_void_p * IBT_MAX_LEVELS),
        ("deriv_pitch", C.c_int64 * IBT_MAX_LEVELS),
    ]


class ibt_jpeg_info_t(C.Structure):
    """HOST mirror of `struct ibt_jpeg_info` in include/ibt.h."""
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("ncomp", C.c_int32),
        ("hsamp", C.c_int32 * 3), ("vsamp", C.c_int32 * 3),
        ("qsel", C.c_int32 * 3), ("dcsel", C.c_int32 * 3), ("acsel", C.c_int32 * 3),
        ("restart_interval", C.c_int32), ("reserved", C.c_int32),
        ("scan_offset", C.c_int64), ("scan_bytes", C.c_int64),
        ("quant", (C.c_uint16 * 64) * 4),
        ("dc_bits", (C.c_uint8 * 16) * 4), ("dc_vals", (C.c_uint8 * 16) * 4),
        ("ac_bits", (C.c_uint8 * 16) * 4), ("ac_vals", (C.c_uint8 * 256) * 4),
    ]


# name -> (restype, argtypes); every symbol include/ibt.h declares
_vp, _i, _i64, _d, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_float, C.c_size_t
_PYR = C.POINTER(ibt_pyramid_t)
_JPG = C.POINTER(ibt_jpeg_info_t)
SIGNATURES = {
    "ibt_version": (_i, []),
    "ibt_error_string": (C.c_char_p, [_i]),
    "ibt_last_cuda_error": (C.c_char_p, []),
    "ibt_gray_u8": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _i, _vp]),
    "ibt_pyramid_levels": (_i, [_i, _i, _i, _i, _i, C.POINTER(C.c_int)]),
    "ibt_pyr_level_u8": (_i, [_vp, _i, _i, _i64, _vp, _i64, _vp, _i64, _vp]),
    "ibt_pyramid_build": (_i, [_PYR, _i, _vp]),
    "ibt_pyramid_build_multichannel": (_i, [_vp, _i64, _i, C.POINTER(_PYR), _i, _vp]),
    "ibt_lk": (_i, [_PYR, _PYR, _vp, _vp, _i, _i, _i, _i, _d, _d, _i, _vp, _vp, _vp, _vp]),
    "ibt_lk_multichannel": (_i, [C.POINTER(_PYR), C.POINTER(_PYR), _i, _vp, _vp, _i, _i, _i, _i, _d, _d, _i, _vp, _vp, _vp, _vp]),
    "ibt_lk_fb": (_i, [_PYR, _PYR, _vp, _i, _i, _i, _i, _d, _d, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                       _vp, _vp]),
    "ibt_lk_fb_multichannel": (_i, [C.POINTER(_PYR), C.POINTER(_PYR), _i, _vp, _i, _i, _i, _i, _d, _d, _f, _vp, _vp, _vp, _vp,
                                    _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ibt_min_eigen_f32": (_i, [_vp, _i, _i, _i64, _i, _vp, _i64, _vp]),
    "ibt_gftt_workspace_bytes": (_sz, [_i, _i]),
    "ibt_corner_harris_f32": (_i, [_vp, _i, _i, _i64, _i, _d, _vp, _i64, _vp]),
    "ibt_gftt": (_i, [_vp, _i64, _vp, _i64, _i, _i, _i, _d, _d, _i, _i, _d, _vp, _sz, _vp, _i, C.POINTER(C.c_int), _vp]),
    "ibt_gftt_async": (_i, [_vp, _i64, _vp, _i64, _i, _i, _i, _d, _d, _i, _i, _d, _vp, _sz, _vp, _i, _vp, _vp]),
    "ibt_min_eigen_ksize_f32": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _i64, _vp]),
    "ibt_corner_harris_ksize_f32": (_i, [_vp, _i, _i, _i64, _i, _i, _d, _vp, _i64, _vp]),
    "ibt_gftt_ksize": (_i, [_vp, _i64, _vp, _i64, _i, _i, _i, _d, _d, _i, _i, _i, _d, _vp, _sz, _vp, _i, C.POINTER(C.c_int),
                            _vp]),
    "ibt_gftt_async_ksize": (_i, [_vp, _i64, _vp, _i64, _i, _i, _i, _d, _d, _i, _i, _i, _d, _vp, _sz, _vp, _i, _vp, _vp]),
    "ibt_gftt_f32src": (_i, [_vp, _i64, _vp, _i64, _i, _i, _i, _d, _d, _i, _i, _i, _d, _vp, _sz, _vp, _i, C.POINTER(C.c_int),
                             _vp]),
    "ibt_min_eigen_f32src": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _i64, _vp]),
    "ibt_corner_harris_f32src": (_i, [_vp, _i, _i, _i64, _i, _i, _d, _vp, _i64, _vp]),
    "ibt_tracks_compact": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, C.POINTER(C.c_int), _vp]),
    "ibt_tracks_compact_async": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "ibt_photo_to_utm": (_i, [_vp, _i64, C.POINTER(C.c_double), _vp, _vp]),
    "ibt_track_velocities": (_i, [_vp, _i, _i, C.POINTER(C.c_double), _d, _d, _d, _d, _d, _d, _vp, _vp, _vp, _vp, _vp]),
    "ibt_polygon_mask": (_i, [_vp, _i, _i, _i, _vp, _i64, _i, _vp]),
    "ibt_grid_bin_workspace_bytes": (_i64, [_i64, _i, _i]),
    "ibt_grid_bin": (_i, [_vp, _vp, _vp, _vp, _i64, _d, _d, _d, _i, _i, _vp, _i64, _vp, _vp, _vp, _vp]),
    "ibt_points_in_polygon": (_i, [_vp, _i, _vp, _i64, _vp, _vp]),
    "ibt_jpeg_parse": (_i, [_vp, _i64, _JPG]),
    "ibt_jpeg_workspace_bytes": (_i64, [_JPG]),
    "ibt_jpeg_decode": (_i, [_vp, _JPG, _vp, _i64, _vp, _i64, _vp, _i64, _i, C.POINTER(C.c_int), _vp]),
    "ibt_jpeg_async_host_bytes": (_i64, []),
    "ibt_jpeg_decode_async": (_i, [_vp, _JPG, _vp, _i64, _vp, _i64, _vp, _i64, _i, _i, _vp, _i64, _vp]),
    "ibt_jpeg_set_probe": (_i, [_i]),
    "ibt_jpeg_recompress_workspace_bytes": (_i64, [_i, _i, _i, _i]),
    "ibt_jpeg_recompress": (_i, [_vp, _i64, _i, _i, _i, _i, _i, _vp, _i64, _vp, _i64, _vp, _i64, _i, _vp]),
    "ibt_lk_set_max_ctas_per_sm": (_i, [_i]),
}

_lib = None


def lib():
    """Load libibt.so (once).  Raises ImportError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libibt.so is missing (%s). Build it with `python -m iceberg_tracking_code_b200.build` "
                "(needs nvcc); there is no CPU fallback." % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)       # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def _errstr(code):
    try:
        return lib().ibt_error_string(code).decode()
    except Exception:
        return "error %d" % code


def check(rc, where):
    if rc != IBT_OK:
        detail = lib().ibt_last_cuda_error().decode() if rc == IBT_E_CUDA else ""
        raise IbtError(rc, where, detail)


def bind_to_gpu_numa_node(device_index):
    """Pin this process (and so the pages it touches first: pinned staging buffers) to the CPUs of the NUMA node the GPU hangs
    off.  With one process per GPU, frames that travel host -> device every step otherwise all stream out of whichever node
    the ranks happened to start on, and 4-8 ranks can saturate that node's memory / inter-socket link.  Returns the node, or
    None when the topology cannot be read -- as on this pool's VMs, which expose one node and no GPU affinity; their host
    fabric stops at ~115 GB/s for 4+ GPUs whatever the placement (then nothing is changed)."""
    import os
    try:
        import torch
        bus = torch.cuda.get_device_properties(device_index).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(device_index), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(device_index), "pci_device_id", 0)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:                                   # noqa: BLE001  (no sysfs / no permission: leave the placement alone)
        return None
