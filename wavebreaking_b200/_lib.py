"""ctypes binding of libwbk.so (the C-ABI declared in include/wbk.h).

There is no CPU implementation behind this module: ``get()`` raises if the nvcc-built
library is missing or no CUDA device is visible.  (The CPU-only test-suite exercises the
kernels' integer logic through ``tests/emu`` -- the same sources compiled against a SIMT
emulation shim -- by calling :func:`use_library` explicitly; nothing in the package does.)
"""

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int64, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_PATH = os.path.join(HERE, "libwbk.so")

OK, ERR_INVALID, ERR_CUDA, ERR_CAPACITY, ERR_NODEVICE = 0, -1, -2, -3, -4
F32, F64, I16 = 0, 1, 2
ROUND_NONE, ROUND_FIRST, ROUND_ALL = 0, 1, 2
SMOOTH_MAX_FUSED = 8

ST_SEG_OVERFLOW = 1
ST_CONTOUR_OVERFLOW = 2
ST_LATTICE_VERTEX = 4
ST_PAIR_OVERFLOW = 8
ST_EVENT_OVERFLOW = 16
ST_SEL_OVERFLOW = 32
ST_WIDTH_OVERFLOW = 64
ST_PACK_OVERFLOW = 128
ST_FETCH_OVERFLOW = 256
ST_SPLIT_CHAINS = 512


class WbkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libwbk error {}: {}".format(code, msg))
        self.code = code


class CapacityError(WbkError):
    pass


class Caps(ctypes.Structure):
    """wbk_caps (include/wbk.h)."""

    _fields_ = [("max_jobs", c_int), ("seg_cap", c_int), ("contour_cap", c_int), ("sel_cap", c_int),
                ("pair_cap", c_int), ("event_cap", c_int)]


class SmoothOpts(ctypes.Structure):
    """wbk_smooth_opts (include/wbk.h): storage orientation / CF packing of the input field."""

    _fields_ = [("flip_lat", c_int), ("flip_lon", c_int), ("scale", c_double), ("offset", c_double),
                ("has_fill", c_int), ("fill", c_int)]


def smooth_opts(flip_lat=False, flip_lon=False, scale=1.0, offset=0.0, fill=None):
    return SmoothOpts(int(bool(flip_lat)), int(bool(flip_lon)), float(scale), float(offset),
                      int(fill is not None), int(fill) if fill is not None else 0)


class IndexParams(ctypes.Structure):
    """wbk_index_params (include/wbk.h)."""

    _fields_ = [("do_streamers", c_int), ("do_overturnings", c_int), ("do_cutoffs", c_int), ("gmax_nx", c_int),
                ("dlon", c_double), ("dlat", c_double), ("geo_dis", c_double), ("cont_dis", c_double),
                ("range_group", c_double), ("ot_min_exp", c_double), ("co_min_exp", c_double)]


EV_STREAMER, EV_OVERTURNING, EV_CUTOFF = 0, 1, 2
EV_INTS, EV_F64 = 10, 6
NEAR_CAP = 4096

_SIGNATURES = {
    "wbk_index_run": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p,
                              c_void_p, POINTER(IndexParams), c_void_p]),
    "wbk_events_raster": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int,
                                  POINTER(SmoothOpts), c_int, c_void_p, POINTER(IndexParams), c_void_p]),
    "wbk_split_clip": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "wbk_split_fetch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "wbk_pack_flags": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_void_p]),
    "wbk_flag_counts": (c_int, [c_void_p, c_int, c_int, ctypes.c_longlong, c_void_p, c_int, c_void_p, c_void_p]),
    "wbk_near_list": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "wbk_events_counts": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), c_void_p]),
    "wbk_events_fetch": (c_int, [c_void_p, c_int, c_int, POINTER(c_int), POINTER(c_double), POINTER(c_int), c_void_p]),
    "wbk_rasterize_rings": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "wbk_rasterize_rings_grid": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double,
                                         c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "wbk_workspace_bytes": (c_size_t, [POINTER(Caps), c_int, c_int, c_int]),
    "wbk_create": (c_int, [POINTER(c_void_p), POINTER(Caps), c_int, c_int, c_int, c_void_p, c_size_t]),
    "wbk_destroy": (c_int, [c_void_p]),
    "wbk_contours": (c_int, [c_void_p, c_void_p, c_int, c_int, POINTER(c_double), c_int, c_void_p]),
    "wbk_smooth_contours": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, POINTER(c_double), c_int,
                                    POINTER(SmoothOpts), c_void_p]),
    "wbk_tune_smooth_halves": (None, [c_int]),
    "wbk_orient": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, POINTER(SmoothOpts), c_void_p]),
    "wbk_contours_counts": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int), c_void_p]),
    "wbk_contours_pack": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p]),
    "wbk_contours_pack_auto": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "wbk_batch_fetch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                c_int, c_void_p, c_void_p]),
    "wbk_track_overlap": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "wbk_track_candidates": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "wbk_track_overlap_exact": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "wbk_track_distance": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "wbk_track_append": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                 c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                 c_int64, c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "wbk_prof_enable": (c_int, [c_int]),
    "wbk_prof_reset": (c_int, []),
    "wbk_prof_read": (c_int, [POINTER(c_int), POINTER(c_double)]),
    "wbk_prof_name": (c_char_p, [c_int]),
    "wbk_launch_count": (ctypes.c_longlong, []),
    "wbk_last_error": (c_char_p, []),
    "wbk_version": (c_int, []),
    "wbk_device_count": (c_int, []),
    "wbk_smooth": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int,
                           POINTER(SmoothOpts), c_void_p]),
    "wbk_convolve2d": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, POINTER(c_double), c_int,
                               c_int, c_int, c_int, c_double, c_void_p]),
    "wbk_nan_border": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "wbk_mflux": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, POINTER(SmoothOpts),
                          c_void_p]),
    "wbk_flip": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "wbk_synth_pv": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_double, c_double, POINTER(c_double), c_int,
                             c_void_p]),
}


class Library:
    """A loaded libwbk plus the torch device its buffers live on."""

    def __init__(self, path, device):
        import torch

        self.path = path
        self.cdll = ctypes.CDLL(path)
        self.device = torch.device(device)
        self.is_cuda = self.device.type == "cuda"
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(self.cdll, name)
            fn.restype = res
            fn.argtypes = args

    def stream(self):
        if not self.is_cuda:
            return None
        import torch

        return c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def last_error(self):
        msg = self.cdll.wbk_last_error()
        return msg.decode() if msg else ""

    def check(self, rc):
        if rc == OK:
            return
        cls = CapacityError if rc == ERR_CAPACITY else WbkError
        raise cls(rc, self.last_error())

    def call(self, name, *args):
        self.check(getattr(self.cdll, name)(*args))


PROF_NKERNELS = 32


def prof_read(lib):
    """dict kernel name -> (launches, total ms) since the last reset."""
    n = (c_int * PROF_NKERNELS)()
    ms = (c_double * PROF_NKERNELS)()
    lib.call("wbk_prof_read", n, ms)
    out = {}
    for k in range(PROF_NKERNELS):
        if n[k]:
            out[lib.cdll.wbk_prof_name(k).decode()] = (int(n[k]), float(ms[k]))
    return out


_LIB = None


def get():
    """The process-wide library; loads wavebreaking_b200/libwbk.so on first use."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(DEFAULT_PATH):
            raise RuntimeError(
                "libwbk.so is not built (run `python -m wavebreaking_b200._build`); "
                "wavebreaking_b200 has no CPU fallback"
            )
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device visible; wavebreaking_b200 runs on sm_100a GPUs only (no CPU fallback)")
        lib = Library(DEFAULT_PATH, "cuda:{}".format(torch.cuda.current_device()))
        n = lib.cdll.wbk_device_count()
        if n <= 0:
            raise RuntimeError(lib.last_error())
        _LIB = lib
    return _LIB


def use_library(path, device):
    """TESTS ONLY: install an explicitly given library build (tests/emu) as the process-wide one."""
    global _LIB
    _LIB = Library(path, device) if path is not None else None
    return _LIB


def ptr(t):
    """Raw pointer of a torch tensor (or None)."""
    return None if t is None else c_void_p(t.data_ptr())


def dtype_code(torch_dtype):
    import torch

    if torch_dtype == torch.float32:
        return F32
    if torch_dtype == torch.float64:
        return F64
    if torch_dtype == torch.int16:
        return I16
    raise TypeError("only float32 / float64 fields are supported, got {}".format(torch_dtype))
