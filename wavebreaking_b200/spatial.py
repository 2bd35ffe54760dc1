"""Device-side spatial pre-processing (host wrappers over libwbk's stencil kernels).

Columnar core behind ``calculate_smoothed_field`` / ``calculate_momentum_flux``
(reference: wavebreaking/processing/spatial.py:27-128).  Inputs are numpy arrays or torch
tensors shaped [ntime, nlat, nlon]; results are torch tensors on the library's device.
"""

import ctypes

import numpy as np
import torch

from . import _lib

DEFAULT_WEIGHTS = np.array([[0, 1, 0], [1, 2, 1], [0, 1, 0]])
_MODES = {"wrap": 0, "grid-wrap": 0, "reflect": 1, "grid-mirror": 1, "mirror": 2, "nearest": 3, "constant": 4,
          "grid-constant": 4}


_STAGE_CHUNK = 32 << 20  # bytes per staging buffer
_STAGE_BUFS = 4
_stage = {}  # page-locked staging buffers + worker pool, created on first use


def _upload_pageable(a, device):
    """Contiguous numpy array in ordinary (pageable) memory -> device tensor through page-locked staging buffers.

    A plain ``tensor.to(device)`` of pageable memory is staged by the driver on one thread (about 10 GB/s for a
    1.2 GB field).  Here worker threads copy 32 MiB chunks into pinned buffers (numpy releases the GIL) while the
    previous chunks cross the link asynchronously, so the upload runs at the host's memcpy rate.
    """
    if not _stage:
        from concurrent.futures import ThreadPoolExecutor

        _stage["bufs"] = [torch.empty(_STAGE_CHUNK, dtype=torch.uint8, pin_memory=True) for _ in range(_STAGE_BUFS)]
        _stage["views"] = [b.numpy() for b in _stage["bufs"]]
        _stage["pool"] = ThreadPoolExecutor(max_workers=_STAGE_BUFS, thread_name_prefix="wbk-upload")
    bufs, views, pool = _stage["bufs"], _stage["views"], _stage["pool"]
    src = a.reshape(-1).view(np.uint8)
    out = torch.empty(a.shape, dtype=torch.float32 if a.dtype == np.float32 else torch.float64, device=device)
    dst = out.view(-1).view(torch.uint8)
    n = src.size
    events = [None] * _STAGE_BUFS
    pending = []  # (future, buffer, offset, length) in submission order

    def flush_one():
        fut, b, off, ln = pending.pop(0)
        fut.result()
        dst[off:off + ln].copy_(bufs[b][:ln], non_blocking=True)
        events[b] = torch.cuda.Event()
        events[b].record()

    for k, off in enumerate(range(0, n, _STAGE_CHUNK)):
        b = k % _STAGE_BUFS
        if len(pending) == _STAGE_BUFS:
            flush_one()  # the oldest chunk, which sits in buffer b
        if events[b] is not None:
            events[b].synchronize()  # its previous contents have left the buffer
        ln = min(_STAGE_CHUNK, n - off)
        pending.append((pool.submit(np.copyto, views[b][:ln], src[off:off + ln]), b, off, ln))
    while pending:
        flush_one()
    for ev in events:
        if ev is not None:
            ev.synchronize()  # the staging buffers are reused by the next upload
    return out


def to_device(a, lib=None):
    """numpy / torch -> contiguous float32/float64 torch tensor on the library device."""
    lib = lib or _lib.get()
    if isinstance(a, torch.Tensor):
        t = a
    else:
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        a = np.ascontiguousarray(a)
        if a.nbytes >= 4 * _STAGE_CHUNK and lib.is_cuda:
            return _upload_pageable(a, lib.device)
        t = torch.from_numpy(a)
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(torch.float64)
    return t.to(lib.device).contiguous()


def _numpy2():
    return int(np.__version__.split(".")[0]) >= 2


def smooth(data, passes, weights=DEFAULT_WEIGHTS, mode="wrap", numpy2_promotion=None):
    """``passes`` x [scipy.ndimage.convolve(weights, mode) / sum(weights)] + NaN border rows.

    Bit-identical to the reference loop (spatial.py:100-107).  ``numpy2_promotion`` selects
    the dtype behaviour of ``float32 / np.int64`` (float64 under NumPy >= 2, the default
    follows the installed NumPy).
    """
    lib = _lib.get()
    x = to_device(data, lib)
    if x.dim() != 3:
        raise ValueError("expected [ntime, nlat, nlon]")
    ntime, nlat, nlon = x.shape
    passes = int(passes) if float(passes) == int(passes) else passes
    if not isinstance(passes, int):
        raise TypeError("'float' object cannot be interpreted as an integer")
    weights = np.asarray(weights)
    if weights.ndim != 2:
        raise RuntimeError("filter weights array has incorrect shape.")
    if numpy2_promotion is None:
        numpy2_promotion = _numpy2()
    f32 = x.dtype == torch.float32
    border = int(weights.shape[0] / 2 + 0.5)
    default = (mode in ("wrap", "grid-wrap") and weights.shape == (3, 3)
               and np.array_equal(weights, DEFAULT_WEIGHTS) and nlat >= 4)
    st = lib.stream()
    if default:
        if passes == 0:
            out = torch.empty_like(x)
            lib.call("wbk_smooth", _lib.ptr(x), _lib.dtype_code(x.dtype), _lib.ptr(out), _lib.dtype_code(out.dtype),
                     None, ntime, nlat, nlon, 0, _lib.ROUND_NONE, None, st)
            return out
        if f32 and numpy2_promotion:
            out_dtype, rmode = torch.float64, _lib.ROUND_FIRST
        elif f32:
            out_dtype, rmode = torch.float32, _lib.ROUND_ALL
        else:
            out_dtype, rmode = torch.float64, _lib.ROUND_NONE
        out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
        tmp = torch.empty_like(out) if passes > _lib.SMOOTH_MAX_FUSED else None
        lib.call("wbk_smooth", _lib.ptr(x), _lib.dtype_code(x.dtype), _lib.ptr(out), _lib.dtype_code(out_dtype),
                 _lib.ptr(tmp), ntime, nlat, nlon, passes, rmode, None, st)
        return out
    # generic weights / mode: one launch per pass
    if mode not in _MODES:
        raise RuntimeError("boundary mode not supported")
    w = np.ascontiguousarray(weights, dtype=np.float64)
    wsum = np.sum(weights)
    promote = numpy2_promotion or not np.issubdtype(np.asarray(wsum).dtype, np.integer) or not f32
    cur = x
    for _ in range(passes):
        out_dtype = torch.float64 if (cur.dtype == torch.float64 or promote) else torch.float32
        out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
        lib.call("wbk_convolve2d", _lib.ptr(cur), _lib.dtype_code(cur.dtype), _lib.ptr(out), _lib.dtype_code(out_dtype),
                 ntime, nlat, nlon, w.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), w.shape[0], w.shape[1],
                 _MODES[mode], 1, float(wsum), st)
        cur = out
    if cur is x:
        cur = x.clone()
    lib.call("wbk_nan_border", _lib.ptr(cur), _lib.dtype_code(cur.dtype), ntime, nlat, nlon, min(border, nlat), st)
    return cur


def momentum_flux(u, v, lon_contiguous=True):
    """(u - zonal mean) * (v - zonal mean), NaN-skipping means (spatial.py:50-54), bit-identical to the reference's
    numpy arithmetic: ``lon_contiguous`` tells whether longitude is the fastest axis of the user's array (numpy then
    sums pairwise) or not (plain sequential sums)."""
    lib = _lib.get()
    a, b = to_device(u, lib), to_device(v, lib)
    if a.shape != b.shape or a.dim() != 3:
        raise ValueError("u and v must both be [ntime, nlat, nlon]")
    if a.dtype != b.dtype:
        a, b = a.to(torch.float64), b.to(torch.float64)
    out = torch.empty_like(a)
    ntime, nlat, nlon = a.shape
    lib.call("wbk_mflux", _lib.ptr(a), _lib.ptr(b), _lib.ptr(out), _lib.dtype_code(a.dtype), ntime, nlat, nlon,
             0 if lon_contiguous else 1, None, lib.stream())
    return out


def flip(x, flip_lat, flip_lon):
    """Re-orient a field to ascending latitude / longitude (data_utils.py:196-213)."""
    lib = _lib.get()
    x = to_device(x, lib)
    if not (flip_lat or flip_lon):
        return x
    out = torch.empty_like(x)
    ntime, nlat, nlon = x.shape
    lib.call("wbk_flip", _lib.ptr(x), _lib.ptr(out), _lib.dtype_code(x.dtype), ntime, nlat, nlon, int(flip_lat),
             int(flip_lon), lib.stream())
    return out


def synth_pv(ntime, nlat, nlon, hour0=0.0, hour_step=1.0, dtype=torch.float32, seed=None):
    """Synthetic PV generated directly in device memory (device mirror of synthetic.pv_field)."""
    from . import synthetic

    lib = _lib.get()
    blobs = np.ascontiguousarray(synthetic.blob_table(synthetic.SEED if seed is None else seed), dtype=np.float64)
    out = torch.empty((ntime, nlat, nlon), dtype=dtype, device=lib.device)
    lib.call("wbk_synth_pv", _lib.ptr(out), _lib.dtype_code(dtype), ntime, nlat, nlon, float(hour0), float(hour_step),
             blobs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), blobs.shape[1], lib.stream())
    return out
