"""Batched per-time-step detection pipeline (the benchmarked hot path).

One batch = ``T`` time steps of a raw field through what the reference does with
``calculate_smoothed_field`` -> ``calculate_contours`` -> ``calculate_streamers`` /
``calculate_overturnings`` / ``calculate_cutoffs`` -> ``to_xarray`` (x3):
columnar event tables (host) and the three int8 flag grids.  All arithmetic runs in libwbk's
CUDA kernels (including the meridian split of the events that straddle the date line).

A batch is *enqueued without any host synchronisation* (``submit``): smoothing, marching squares, linking,
device-side packing, the three indices, rasterisation and one gather of all results, then the asynchronous
device->host copies.  ``collect`` waits once and slices the tables.  Several slots (each with its own
context, buffers and CUDA stream) keep the GPU busy while the host handles the previous batch and let
host<->device copies overlap with kernels (``Detector.stream``).
"""

import ctypes
import logging
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, detect, spatial

logger = logging.getLogger(__name__)


@dataclass
class BatchResult:
    ntime: int
    contours: detect.ContourSet
    tables: dict              # kind -> detect.EventTable
    flags: torch.Tensor       # int8 [3, ntime, nlat, nlon] (device, or pinned host in the end-to-end path)
    gmax_nx: int
    n_split: int = 0
    # streamer pairs decided within 1e-9 of geo_dis / cont_dis, kept AND rejected ones (wbk_near_list):
    # int32 [m, 6] = time step, level index, contour, i, j, flags (1 kept, 2 geo in band, 4 cont in band)
    near: np.ndarray = None
    near_total: int = 0
    pieces: dict = None  # device-clipped pieces of the straddling events: ev (row in kind-major order), off, xy
    counts: tuple = None  # events per kind (streamers, overturnings, cutoffs)
    work: dict = None  # device work counters of the batch: marching-squares segments, candidate pairs, scan tiles
    flags_packed: torch.Tensor = None  # pinned uint8: the three grids, one bit per cell (unpack_flags restores them)


def packed_nbytes(ncells):
    """bytes of the bit-packed form of ``ncells`` flag cells (whole 32-bit words)."""
    return 4 * ((int(ncells) + 31) // 32)


def unpack_flags(packed, nt, nlat, nlon):
    """int8 [3, nt, nlat, nlon] flag grids from the bit-packed download (host numpy)."""
    ncells = 3 * nt * nlat * nlon
    buf = packed.numpy() if isinstance(packed, torch.Tensor) else np.asarray(packed)
    bits = np.unpackbits(buf[:packed_nbytes(ncells)], bitorder="little")[:ncells]
    return bits.view(np.int8).reshape(3, nt, nlat, nlon)


def _pinned(shape, dtype, lib):
    return torch.empty(shape, dtype=dtype, pin_memory=lib.is_cuda)


def _intensity_item(item, shape):
    """One intensity item of ``Detector.stream`` as the tuple ``(field,)`` or ``(u, v)``; raises ValueError unless its
    tensors are float32 / float64 and shaped like the batch (``shape``), and u and v agree in shape and dtype."""
    fields = tuple(item) if isinstance(item, (tuple, list)) else (item,)
    if len(fields) not in (1, 2) or not all(isinstance(f, torch.Tensor) for f in fields):
        raise ValueError("an intensity item is a tensor or a pair (u, v) of tensors")
    if len(fields) == 2 and (fields[0].shape != fields[1].shape or fields[0].dtype != fields[1].dtype):
        raise ValueError("u and v differ: shapes {} and {}, dtypes {} and {}".format(
            tuple(fields[0].shape), tuple(fields[1].shape), fields[0].dtype, fields[1].dtype))
    for f in fields:
        if f.dtype not in (torch.float32, torch.float64):
            raise ValueError("intensity has to be float32 or float64, got {} (packed int16 u / v are not "
                             "supported)".format(f.dtype))
        if tuple(f.shape) != tuple(shape):
            raise ValueError("an intensity item of shape {} for a batch of shape {}".format(tuple(f.shape),
                                                                                          tuple(shape)))
    return fields


class _Slot:
    """Context + device / pinned buffers + stream for one batch in flight."""

    def __init__(self, det, T, caps=None):
        lib = det.lib
        self.det, self.T = det, int(T)
        dev = lib.device
        L = len(det.levels)
        J = self.T * L
        self.J = J
        want = detect.default_caps(det.nlat, det.nlon, det.add, J)
        if caps:
            for k, v in caps.items():
                if k in want:  # (cap_c / cap_p / cap_e / cap_r size the slot's own buffers, below)
                    want[k] = max(want[k], int(v))
        self.ctx = detect.Context(det.nlat, det.nlon, det.add, want)
        self.cap_c = int(max(64 * J, 1024))
        self.cap_p = int(max(min(want["seg_cap"], 16384) * J, 1 << 16))
        self.cap_e = int(max(48 * J, 1024))
        self.cap_r = int(max(8192 * J, 1 << 16))
        if caps:
            self.cap_c = max(self.cap_c, int(caps.get("cap_c", 0)))
            self.cap_p = max(self.cap_p, int(caps.get("cap_p", 0)))
            self.cap_e = max(self.cap_e, int(caps.get("cap_e", 0)))
            self.cap_r = max(self.cap_r, int(caps.get("cap_r", 0)))
        shape = (self.T, det.nlat, det.nlon)
        i32, f64 = torch.int32, torch.float64
        self.sm = torch.empty(shape, dtype=f64, device=dev) if det.passes > 0 else None
        self.sm_f32 = None
        self.sm_tmp = torch.empty(shape, dtype=f64, device=dev) if det.passes > _lib.SMOOTH_MAX_FUSED else None
        self.raw_dev = None  # allocated on first host submit
        self.inten_dev = [None, None]  # uploads of host intensity items (the field, or u and v), on first use
        self.mflux = None  # momentum flux of (u, v) intensity items, on first use
        self.flipped = None
        self.job_off = torch.empty(J + 1, dtype=i32, device=dev)
        self.pt_off = torch.empty(self.cap_c + 1, dtype=i32, device=dev)
        self.meta = torch.empty((self.cap_c, 4), dtype=i32, device=dev)
        self.pts = torch.empty(self.cap_p, dtype=i32, device=dev)
        self.work = torch.empty(2 * self.cap_p, dtype=f64, device=dev)
        self.flags = None
        self.ev_int = torch.empty((self.cap_e, _lib.EV_INTS), dtype=i32, device=dev)
        self.ev_f64 = torch.empty((self.cap_e, _lib.EV_F64), dtype=f64, device=dev)
        self.ev_job = torch.empty(self.cap_e, dtype=i32, device=dev)
        self.ring_off = torch.empty(self.cap_e + 1, dtype=i32, device=dev)
        self.ring_pts = torch.empty(self.cap_r, dtype=i32, device=dev)
        self.summary = torch.zeros(16, dtype=i32, device=dev)
        self.h_summary = _pinned(16, i32, lib)
        # pieces of the events that straddle the last meridian (device clipper output, wbk_split_fetch)
        self.cap_sr = int(max(16 * J, 1024))
        self.cap_sv = int(max(4096 * J, 1 << 16))
        if caps:
            self.cap_sr = max(self.cap_sr, int(caps.get("cap_sr", 0)))
            self.cap_sv = max(self.cap_sv, int(caps.get("cap_sv", 0)))
        self.sp_ev = torch.zeros(self.cap_sr, dtype=i32, device=dev)
        self.sp_off = torch.zeros(self.cap_sr + 1, dtype=i32, device=dev)
        self.sp_xy = torch.zeros((self.cap_sv, 2), dtype=i32, device=dev)
        self.sp_cnt = torch.zeros(4, dtype=i32, device=dev)
        self.h_sp_ev = _pinned(self.cap_sr, i32, lib)
        self.h_sp_off = _pinned(self.cap_sr + 1, i32, lib)
        self.h_sp_xy = _pinned((self.cap_sv, 2), i32, lib)
        self.h_sp_cnt = _pinned(4, i32, lib)
        self.near = torch.zeros((_lib.NEAR_CAP, 4), dtype=i32, device=dev)
        self.near_cnt = torch.zeros(1, dtype=i32, device=dev)
        self.h_near = _pinned((_lib.NEAR_CAP, 4), i32, lib)
        self.h_near_cnt = _pinned(1, i32, lib)
        self.h_ev_int = _pinned((self.cap_e, _lib.EV_INTS), i32, lib)
        self.h_ev_f64 = _pinned((self.cap_e, _lib.EV_F64), f64, lib)
        self.h_ev_job = _pinned(self.cap_e, i32, lib)
        self.h_ring_off = _pinned(self.cap_e + 1, i32, lib)
        self.h_ring_pts = _pinned(self.cap_r, i32, lib)
        self.stream = torch.cuda.Stream(device=dev) if lib.is_cuda else None
        self.done = torch.cuda.Event() if lib.is_cuda else None
        self.pending = None   # (raw, ntime, flags_dev, flags_host, gmax)
        self.grow_seen = 0
        self.packed = None    # bit-packed flag grids (device), allocated on first use
        self.clim_group = None  # int32 [T] (device): groups of the batch's steps for FlagClimatology, on first use
        self.graphs = {}      # buffers key -> (torch.cuda.CUDAGraph, pending record)
        self.graph_seen = set()

    def close(self):
        self.graphs.clear()
        self.ctx.close()


class Detector:
    """Holds the grid, thresholds and the reusable slots of one detection configuration."""

    def __init__(self, lat, lon, levels=(2.0,), periodic_add=120, passes=5, which=detect.KINDS, geo_dis=800.0,
                 cont_dis=1500.0, range_group=5.0, ot_min_exp=5.0, co_min_exp=5.0, want_flags=True, fuse=True,
                 packing=None, graphs=False, nvtx=True, want_pieces=False):
        self.lib = _lib.get()
        self.lat = np.asarray(lat, dtype=np.float64)
        self.lon = np.asarray(lon, dtype=np.float64)
        # descending coordinates (ERA5 latitudes): batches are flipped on the device after the upload
        # (utils/data_utils.py:196-213); all results refer to the ascending orientation
        self.flip_lat = bool(len(self.lat) > 1 and self.lat[0] > self.lat[-1])
        self.flip_lon = bool(len(self.lon) > 1 and self.lon[0] > self.lon[-1])
        if self.flip_lat:
            self.lat = self.lat[::-1].copy()
        if self.flip_lon:
            self.lon = self.lon[::-1].copy()
        self.nlat, self.nlon = len(self.lat), len(self.lon)
        self.dlon = float(abs(self.lon[1] - self.lon[0]))
        self.dlat = float(abs(self.lat[1] - self.lat[0]))
        self.add = int(periodic_add / self.dlon)
        self.levels = np.ascontiguousarray(np.atleast_1d(np.asarray(levels, dtype=np.float64)))
        self.passes = int(passes)
        self.which = tuple(which)
        self.params = dict(geo_dis=geo_dis, cont_dis=cont_dis, range_group=range_group, ot_min_exp=ot_min_exp,
                           co_min_exp=co_min_exp)
        self.want_flags = want_flags
        if want_flags:
            detect.grid_ratio(self.dlon, self.dlat)  # flag grids need spacings wbk_events_raster can measure in
        # smoothing that also leaves the marching-squares bit planes (wbk_smooth_contours): the contour stage then
        # does not re-read the smoothed field.  fuse=False runs wbk_smooth + wbk_contours (same results).
        self.fuse = bool(fuse)
        # CF packing of int16 input (scale_factor, add_offset, _FillValue or None), decoded in the smoothing loads
        self.packing = tuple(packing) if packing is not None else (1.0, 0.0, None)
        # also download the device clipper's pieces of the events that straddle the last meridian (events_soup then
        # needs no host-side polygon clipping; used by the tracking leg)
        self.want_pieces = bool(want_pieces)
        self.graphs = bool(graphs)  # replay one captured CUDA graph per batch (see submit)
        self.graph_replays = 0
        self.graph_kernel_launches = 0
        self.nvtx = bool(nvtx)      # NVTX ranges per stage (upload / smooth+contours / indices / properties / download)
        self.coords = detect.coord_tables(self.lat, self.lon, self.dlon, self.dlat, self.lib)
        self._slots = {}
        self._grow = {}
        self._grow_version = 0

    # ------------------------------------------------------------------ slots
    def _slot(self, T, index=0):
        key = (int(T), int(index))
        s = self._slots.get(key)
        if s is not None and s.pending is None and s.grow_seen != self._grow_version:
            # another slot had to regrow its arenas: adopt the larger capacities before the next batch overflows too
            if self.lib.is_cuda:
                torch.cuda.synchronize()
            s.close()
            s = None
        if s is None:
            s = _Slot(self, T, self._grow)
            s.grow_seen = self._grow_version
            self._slots[key] = s
        return s

    def close(self):
        for s in self._slots.values():
            s.close()
        self._slots.clear()

    def _prm(self, gmax):
        p = self.params
        return _lib.IndexParams(
            do_streamers=int("streamers" in self.which), do_overturnings=int("overturnings" in self.which),
            do_cutoffs=int("cutoffs" in self.which), gmax_nx=int(gmax), dlon=self.dlon, dlat=self.dlat,
            geo_dis=float(p["geo_dis"]), cont_dis=float(p["cont_dis"]), range_group=float(p["range_group"]),
            ot_min_exp=float(p["ot_min_exp"]), co_min_exp=float(p["co_min_exp"]))

    # ------------------------------------------------------------------ enqueue / collect
    def _enqueue(self, slot, raw, flags_out, flags_host, gmax_nx, smoothed, intensity, packed_host):
        """All device work of one batch on the CURRENT stream; returns what ``collect`` needs.  Allocation-free in
        the steady state (so it can be captured into a CUDA graph)."""
        lib = self.lib
        nvtx = torch.cuda.nvtx if (lib.is_cuda and self.nvtx) else None
        nt = int(raw.shape[0])
        st = lib.stream()
        if nvtx:
            nvtx.range_push("wbk.upload")
        if raw.device != lib.device:  # host input: H2D on this slot's stream
            if slot.raw_dev is None or slot.raw_dev.dtype != raw.dtype:
                slot.raw_dev = torch.empty((slot.T, self.nlat, self.nlon), dtype=raw.dtype, device=lib.device)
            slot.raw_dev[:nt].copy_(raw, non_blocking=True)
            raw = slot.raw_dev[:nt]
        raw = raw.contiguous()
        raw_in = raw  # what the caller handed over (the regrow path re-submits exactly this)
        if isinstance(intensity, tuple):  # the field or (u, v) as stored: host items go to the slot's own buffers
            fields = []
            for k, f in enumerate(intensity):
                if f.device != lib.device:
                    if slot.inten_dev[k] is None or slot.inten_dev[k].dtype != f.dtype:
                        slot.inten_dev[k] = torch.empty((slot.T, self.nlat, self.nlon), dtype=f.dtype,
                                                        device=lib.device)
                    slot.inten_dev[k][:nt].copy_(f, non_blocking=True)
                    f = slot.inten_dev[k][:nt]
                fields.append(f.contiguous())
            intensity = tuple(fields)
        elif intensity is not None:
            intensity = intensity.to(lib.device).contiguous()
        if nvtx:
            nvtx.range_pop()
            nvtx.range_push("wbk.smooth+contours")
        h = slot.ctx.handle
        L = len(self.levels)
        lv = self.levels.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        # the stored orientation (descending ERA5 latitudes, utils/data_utils.py:196-213) and the CF packing of
        # int16 input are resolved inside the smoothing loads: no re-oriented / decoded copy of the batch
        opts = _lib.smooth_opts(self.flip_lat, self.flip_lon, *self.packing) if (
            self.flip_lat or self.flip_lon or raw.dtype == torch.int16) else None
        fused = False
        if smoothed is not None:
            sm = smoothed
        elif self.passes > 0:
            f32 = raw.dtype == torch.float32
            if f32 and not spatial._numpy2():
                if slot.sm_f32 is None:
                    slot.sm_f32 = torch.empty((slot.T, self.nlat, self.nlon), dtype=torch.float32, device=lib.device)
                sm, rmode = slot.sm_f32[:nt], _lib.ROUND_ALL
            else:
                sm, rmode = slot.sm[:nt], (_lib.ROUND_FIRST if f32 else _lib.ROUND_NONE)
            if self.fuse and sm.dtype == torch.float64 and self.passes <= _lib.SMOOTH_MAX_FUSED and self.nlat >= 4:
                lib.call("wbk_smooth_contours", h, _lib.ptr(raw), _lib.dtype_code(raw.dtype), _lib.ptr(sm), nt,
                         self.passes, lv, L, opts, st)
                fused = True
            else:
                lib.call("wbk_smooth", _lib.ptr(raw), _lib.dtype_code(raw.dtype), _lib.ptr(sm),
                         _lib.dtype_code(sm.dtype), _lib.ptr(slot.sm_tmp), nt, self.nlat, self.nlon, self.passes,
                         rmode, opts, st)
        else:
            if opts is not None:  # no smoothing: orientation / decode only
                want = torch.float64 if raw.dtype == torch.int16 else raw.dtype
                if slot.flipped is None or slot.flipped.dtype != want:
                    slot.flipped = torch.empty((slot.T, self.nlat, self.nlon), dtype=want, device=lib.device)
                lib.call("wbk_orient", _lib.ptr(raw), _lib.dtype_code(raw.dtype), _lib.ptr(slot.flipped), nt,
                         self.nlat, self.nlon, opts, st)
                raw = slot.flipped[:nt]
            sm = raw
        if not fused:
            lib.call("wbk_contours", h, _lib.ptr(sm), _lib.dtype_code(sm.dtype), nt, lv, L, st)
        lib.call("wbk_contours_pack_auto", h, _lib.ptr(slot.job_off), _lib.ptr(slot.pt_off), _lib.ptr(slot.meta),
                 _lib.ptr(slot.pts), slot.cap_c, slot.cap_p, st)
        if nvtx:
            nvtx.range_pop()
            nvtx.range_push("wbk.indices")
        if isinstance(intensity, torch.Tensor) and intensity.dtype != sm.dtype:
            intensity = intensity.to(sm.dtype)
        prm = self._prm(-1 if gmax_nx is None else gmax_nx)
        lib.call("wbk_index_run", h, nt * L, L, _lib.ptr(slot.job_off), _lib.ptr(slot.pt_off), _lib.ptr(slot.meta),
                 _lib.ptr(slot.pts), slot.cap_c, slot.cap_p, _lib.ptr(self.coords), _lib.ptr(slot.work),
                 ctypes.byref(prm), st)
        lib.call("wbk_near_list", h, _lib.ptr(slot.near), _lib.NEAR_CAP, _lib.ptr(slot.near_cnt), st)
        if nvtx:
            nvtx.range_pop()
            nvtx.range_push("wbk.properties+to_xarray")
        flags = None
        if self.want_flags:
            if flags_out is not None:
                flags = flags_out
            else:
                if slot.flags is None:
                    slot.flags = torch.empty((3, slot.T, self.nlat, self.nlon), dtype=torch.int8, device=lib.device)
                flags = slot.flags if nt == slot.T else torch.empty((3, nt, self.nlat, self.nlon), dtype=torch.int8,
                                                                    device=lib.device)
        # the rasteriser reads the intensity's member cells in their stored dtype and orientation
        inten, iflip = intensity, (0, 0)
        if isinstance(intensity, tuple):
            inten, iflip = intensity[0], (int(self.flip_lat), int(self.flip_lon))
            if len(intensity) == 2:
                # zonal means summed in the stored memory order (what numpy does on the user's array); longitude is
                # the contiguous axis of a batch
                u, v = intensity
                if slot.mflux is None or slot.mflux.dtype != u.dtype:
                    slot.mflux = torch.empty((slot.T, self.nlat, self.nlon), dtype=u.dtype, device=lib.device)
                inten = slot.mflux[:nt]
                lib.call("wbk_mflux", _lib.ptr(u), _lib.ptr(v), _lib.ptr(inten), _lib.dtype_code(u.dtype), nt,
                         self.nlat, self.nlon, 0, st)
        lib.call("wbk_events_raster", h, _lib.ptr(slot.job_off), _lib.ptr(slot.pt_off), _lib.ptr(slot.pts),
                 _lib.ptr(self.coords), _lib.ptr(sm), _lib.dtype_code(sm.dtype), _lib.ptr(inten),
                 _lib.dtype_code(sm.dtype if inten is None else inten.dtype), iflip[0], iflip[1], nt, _lib.ptr(flags),
                 ctypes.byref(prm), st)
        lib.call("wbk_batch_fetch", h, _lib.ptr(slot.pt_off), _lib.ptr(slot.pts), _lib.ptr(slot.ev_int),
                 _lib.ptr(slot.ev_f64), _lib.ptr(slot.ev_job), _lib.ptr(slot.ring_off), _lib.ptr(slot.ring_pts),
                 slot.cap_e, slot.cap_r, _lib.ptr(slot.summary), st)
        if flags is not None and self.want_pieces:
            lib.call("wbk_split_fetch", h, _lib.ptr(slot.sp_ev), _lib.ptr(slot.sp_off), _lib.ptr(slot.sp_xy), slot.cap_sr,
                     slot.cap_sv, _lib.ptr(slot.sp_cnt), st)
            slot.h_sp_cnt.copy_(slot.sp_cnt, non_blocking=True)
            slot.h_sp_ev.copy_(slot.sp_ev, non_blocking=True)
            slot.h_sp_off.copy_(slot.sp_off, non_blocking=True)
            slot.h_sp_xy.copy_(slot.sp_xy, non_blocking=True)
        if nvtx:
            nvtx.range_pop()
            nvtx.range_push("wbk.download")
        # asynchronous read-back of everything the host needs (tables are small; flags only on request)
        slot.h_summary.copy_(slot.summary, non_blocking=True)
        slot.h_near_cnt.copy_(slot.near_cnt, non_blocking=True)
        slot.h_near.copy_(slot.near, non_blocking=True)
        slot.h_ev_int.copy_(slot.ev_int, non_blocking=True)
        slot.h_ev_f64.copy_(slot.ev_f64, non_blocking=True)
        slot.h_ev_job.copy_(slot.ev_job, non_blocking=True)
        slot.h_ring_off.copy_(slot.ring_off, non_blocking=True)
        slot.h_ring_pts.copy_(slot.ring_pts, non_blocking=True)
        if flags_host is not None and flags is not None:
            flags_host[:, :nt].copy_(flags[:, :nt] if flags.shape[1] != nt else flags, non_blocking=True)
        if packed_host is not None and flags is not None:
            # one bit per cell on the wire (wbk_pack_flags); unpack_flags() restores the int8 grids on the host
            ncells = 3 * nt * self.nlat * self.nlon
            if slot.packed is None:
                slot.packed = torch.empty(packed_nbytes(3 * slot.T * self.nlat * self.nlon), dtype=torch.uint8,
                                          device=lib.device)
            fl = flags if flags.shape[1] == nt and flags.is_contiguous() else flags[:, :nt].contiguous()
            lib.call("wbk_pack_flags", _lib.ptr(fl), _lib.ptr(slot.packed), ncells, st)
            nb = packed_nbytes(ncells)
            packed_host[:nb].copy_(slot.packed[:nb], non_blocking=True)
        if nvtx:
            nvtx.range_pop()
        # (inten keeps the buffer a captured graph writes the momentum flux to alive)
        return dict(raw=raw_in, nt=nt, flags=flags, flags_host=flags_host, gmax=gmax_nx, smoothed=smoothed, sm=sm,
                    intensity=intensity, inten=inten, packed_host=packed_host)

    def submit(self, slot, raw, flags_out=None, flags_host=None, gmax_nx=None, smoothed=None, stream=None,
               intensity=None, packed_host=None):
        """Enqueue one batch on the slot's stream (or ``stream``).  ``raw``: device tensor or (pinned) host
        tensor [T' <= T, nlat, nlon].  No host synchronisation happens here.

        With ``Detector(graphs=True)`` the whole batch (uploads, ~25 kernels and memsets, downloads) is captured into
        ONE CUDA graph per (slot, buffers) the second time the same buffers are submitted and replayed afterwards: one
        launch per batch instead of ~40 driver calls, which is what limits several ranks sharing one host.

        ``intensity``: a device tensor [T', nlat, nlon] in the ascending orientation, converted to the smoothed
        field's dtype (as in ``detect.run_indices``; not captured in a graph), or a tuple ``(field,)`` / ``(u, v)``
        in the form of :meth:`stream`'s items (stored orientation, own dtype, captured with the batch)."""
        lib = self.lib
        nt = int(raw.shape[0])
        if nt > slot.T:
            raise ValueError("batch of {} time steps exceeds the slot size {}".format(nt, slot.T))
        if isinstance(intensity, tuple):
            intensity = _intensity_item(intensity, raw.shape)
        use_stream = stream if stream is not None else slot.stream
        args = (slot, raw, flags_out, flags_host, gmax_nx, smoothed, intensity, packed_host)
        if use_stream is None:  # emulator
            slot.pending = dict(self._enqueue(*args), stream=None)
            return slot
        graphable = self.graphs and smoothed is None and not isinstance(intensity, torch.Tensor)
        key = None
        if graphable:
            key = (raw.data_ptr(), raw.dtype, nt, None if flags_out is None else flags_out.data_ptr(),
                   None if flags_host is None else flags_host.data_ptr(),
                   None if packed_host is None else packed_host.data_ptr(), gmax_nx, use_stream.cuda_stream,
                   None if intensity is None else tuple((f.data_ptr(), f.dtype, f.device.type) for f in intensity))
        with torch.cuda.stream(use_stream):
            use_stream.wait_stream(torch.cuda.default_stream(lib.device))
            if key is not None and key in slot.graphs:
                g, pend, nk = slot.graphs[key]
                g.replay()
                self.graph_replays += 1
                self.graph_kernel_launches += nk  # kernels inside the graph (the library only counts direct launches)
                slot.pending = pend
            elif key is not None and key in slot.graph_seen:
                # second submission of these buffers: everything is allocated, capture the batch
                use_stream.synchronize()
                g = torch.cuda.CUDAGraph()
                n0 = lib.cdll.wbk_launch_count()
                with torch.cuda.graph(g, stream=use_stream, capture_error_mode="relaxed"):
                    pend = self._enqueue(*args)
                nk = int(lib.cdll.wbk_launch_count() - n0)
                slot.graphs[key] = (g, pend, nk)
                g.replay()
                self.graph_replays += 1
                self.graph_kernel_launches += nk
                slot.pending = pend
            else:
                slot.pending = self._enqueue(*args)
                if key is not None:
                    slot.graph_seen.add(key)
            slot.pending = dict(slot.pending, stream=use_stream)  # (a replayed graph's record is shared: copy it)
            slot.done.record()
        return slot

    def collect(self, slot, climatology=None, trackers=()):
        """Wait for the slot's batch and return its BatchResult (re-runs it with larger arenas on overflow).

        ``climatology``: a :class:`FlagClimatology` that the batch's flag grids are added to; ``trackers``: a list of
        :class:`EventTracker` that link the batch's events.  Both happen here, after every check that can make the batch
        run again has passed, so each batch is counted exactly once."""
        pend = slot.pending
        if pend is None:
            raise RuntimeError("nothing was submitted on this slot")
        if slot.done is not None:
            slot.done.synchronize()
        s = slot.h_summary.numpy()
        C, P, ns, no, nc, status, max_nx, n_split = (int(v) for v in s[:8])
        work = dict(segments=int(s[8]), pairs=int(s[9]), tiles=int(s[11]))
        bad = status & (_lib.ST_SEG_OVERFLOW | _lib.ST_CONTOUR_OVERFLOW | _lib.ST_PAIR_OVERFLOW | _lib.ST_EVENT_OVERFLOW
                        | _lib.ST_SEL_OVERFLOW | _lib.ST_PACK_OVERFLOW | _lib.ST_FETCH_OVERFLOW)
        if status & _lib.ST_SPLIT_CHAINS:
            raise _lib.WbkError(_lib.ERR_INVALID, "an event crosses the last meridian too often for the device clipper; "
                                                  "its cells would be missing from the flag grids")
        if bad:
            return self._regrow_and_rerun(slot, status, climatology, trackers)
        slot.pending = None
        nt = pend["nt"]
        L = len(self.levels)
        counts = (ns, no, nc)
        tables, o = {}, 0
        ring_off = slot.h_ring_off.numpy()
        ring_pts = slot.h_ring_pts.numpy().view(np.uint32)
        for kind, n in zip(detect.KINDS, counts):
            ints = slot.h_ev_int.numpy()[o:o + n].copy()
            f64 = slot.h_ev_f64.numpy()[o:o + n].copy()
            job = slot.h_ev_job.numpy()[o:o + n].copy()
            rings = None
            if kind != "overturnings":
                ro = ring_off[o:o + n + 1].copy()
                rings = detect.LazyRings(ro, ring_pts[ro[0]:ro[-1]].copy())
            tab = detect.EventTable(kind=kind, job=job, contour=ints[:, 0].copy(), ind1=ints[:, 1].copy(),
                                    ind2=ints[:, 2].copy(), box=ints[:, 3:7].copy(), orientation=ints[:, 7].copy(),
                                    split=ints[:, 8].copy(), near=ints[:, 9].copy(), sums=f64)
            tab.rings = rings
            tables[kind] = tab
            o += n
        cs = detect.ContourSet(
            njobs=nt * L, nlevels=L, nlat=self.nlat, nlon=self.nlon, add=self.add, levels=self.levels,
            job_off=slot.job_off[:nt * L + 1], pt_off=slot.pt_off[:C + 1], meta=slot.meta[:C], pts=slot.pts[:P],
            status=np.full(nt * L, status, dtype=np.int32), max_nx=max_nx, h_ncontours=None, h_npoints=None)
        flags = pend["flags_host"] if pend["flags_host"] is not None else pend["flags"]
        packed = pend.get("packed_host")
        n_sp = int(sum(int((t.split == 1).sum()) for t in tables.values()))
        pieces = None
        if self.want_pieces and pend["flags"] is not None:
            npc, nvx, clip_over = (int(v) for v in slot.h_sp_cnt.numpy()[:3])
            if npc > slot.cap_sr or nvx > slot.cap_sv:
                grow = dict(self._grow)
                grow["cap_sr"], grow["cap_sv"] = max(2 * slot.cap_sr, 2 * npc), max(2 * slot.cap_sv, 2 * nvx)
                self._grow = grow
                slot.pending = pend  # the re-run submits the batch again from its pending record
                return self._regrow_and_rerun(slot, 0, climatology, trackers)
            off = slot.h_sp_off.numpy()[:npc + 1].astype(np.int64)
            pieces = dict(ev=slot.h_sp_ev.numpy()[:npc].copy(), off=off, xy=slot.h_sp_xy.numpy()[:nvx].copy(),
                          overflow=bool(clip_over))
        n_near = int(slot.h_near_cnt[0]) if "streamers" in self.which else 0
        rec = slot.h_near.numpy()[:min(n_near, _lib.NEAR_CAP)]
        near = np.c_[rec[:, 0] // L, rec[:, 0] % L, rec[:, 1], rec[:, 2], rec[:, 3] & 0x0FFFFFFF, (rec[:, 3] >> 28) & 7]
        if climatology is not None:
            climatology._add(slot, pend)
        for tr in trackers or ():
            tr._add(slot, pend, tables, counts)
        return BatchResult(ntime=nt, contours=cs, tables=tables, flags=flags,
                           gmax_nx=max_nx if pend["gmax"] is None else int(pend["gmax"]), n_split=n_sp,
                           near=near.astype(np.int32), near_total=n_near, flags_packed=packed, work=work, pieces=pieces,
                           counts=(ns, no, nc))

    def _regrow_and_rerun(self, slot, status, climatology=None, trackers=()):
        pend = slot.pending
        caps = dict(slot.ctx.caps)
        grow = dict(self._grow)
        if status & _lib.ST_SEG_OVERFLOW:
            grow["seg_cap"] = caps["seg_cap"] * 2
        if status & _lib.ST_CONTOUR_OVERFLOW:
            grow["contour_cap"] = caps["contour_cap"] * 2
        if status & _lib.ST_PAIR_OVERFLOW:
            grow["pair_cap"] = caps["pair_cap"] * 4
        if status & _lib.ST_EVENT_OVERFLOW:
            grow["event_cap"] = caps["event_cap"] * 4
        if status & _lib.ST_SEL_OVERFLOW:
            grow["sel_cap"] = caps["sel_cap"] * 4
        # the summary record holds the true totals of the batch: size the buffers for them (with headroom) in one go
        C, P, ns, no, nc = (int(v) for v in slot.h_summary.numpy()[:5])
        if status & _lib.ST_PACK_OVERFLOW:
            grow["cap_c"] = max(slot.cap_c * 2, int(1.3 * C))
            grow["cap_p"] = max(slot.cap_p * 2, int(1.3 * P))
        if status & _lib.ST_FETCH_OVERFLOW:
            grow["cap_e"] = max(slot.cap_e * 2, int(1.3 * (ns + no + nc)))
            grow["cap_r"] = slot.cap_r * 2
        self._grow = grow
        self._grow_version += 1
        if len(grow) and max(grow.values()) > (1 << 28):
            raise _lib.WbkError(_lib.ERR_CAPACITY, "arenas still overflow after repeated regrowth (status {})".format(status))
        key = next(k for k, v in self._slots.items() if v is slot)
        if self.lib.is_cuda:
            torch.cuda.synchronize()
        slot.close()
        new = _Slot(self, slot.T, grow)
        new.grow_seen = self._grow_version
        self._slots[key] = new
        self.submit(new, pend["raw"], flags_out=pend["flags"], flags_host=pend["flags_host"], gmax_nx=pend["gmax"],
                    smoothed=pend["smoothed"], intensity=pend["intensity"], packed_host=pend.get("packed_host"))
        return self.collect(new, climatology, trackers)

    # ------------------------------------------------------------------ convenience
    def run_batch(self, raw, gmax_nx=None, smoothed=None, intensity=None):
        """Synchronous: raw device tensor [T, nlat, nlon] -> BatchResult (flags and contour set are private
        copies, valid after further calls)."""
        nt = int(raw.shape[0])
        slot = self._slot(nt)
        flags = None
        if self.want_flags:
            flags = torch.empty((3, nt, self.nlat, self.nlon), dtype=torch.int8, device=self.lib.device)
        self.submit(slot, raw, flags_out=flags, gmax_nx=gmax_nx, smoothed=smoothed, intensity=intensity)
        res = self.collect(slot)
        cs = res.contours
        cs.job_off, cs.pt_off, cs.meta, cs.pts = cs.job_off.clone(), cs.pt_off.clone(), cs.meta.clone(), cs.pts.clone()
        return res

    def run_batch_host(self, raw_host, flags_host=None):
        """Synchronous end-to-end: (pinned) host input -> tables + flag grids in (pinned) host memory."""
        nt = int(raw_host.shape[0])
        slot = self._slot(nt)
        if self.want_flags and flags_host is None:
            flags_host = _pinned((3, nt, self.nlat, self.nlon), torch.int8, self.lib)
        self.submit(slot, raw_host, flags_host=flags_host)
        return self.collect(slot)

    def stream(self, batches, depth=3, flags_host=None, shared_stream=False, gmax_nx="full", packed_host=None,
               climatology=None, trackers=None, intensity=None):
        """Pipelined execution: yields one BatchResult per input batch, in order.

        ``batches``: iterable of device or pinned-host tensors of (at most) equal length.  ``depth`` batches are
        in flight at once, each on its own CUDA stream, so uploads, kernels, downloads and the host-side table
        handling overlap.  With ``shared_stream`` all slots enqueue on ONE side stream: kernels of different
        batches do not overlap each other, the host merely runs ahead (device-resident inputs).
        ``flags_host``: optional list of pinned int8 buffers, one per slot.
        ``packed_host``: optional list of pinned uint8 buffers (``packed_nbytes(3 * T * nlat * nlon)`` bytes), one per
        slot: the flag grids come back bit-packed (8x less device -> host traffic; ``unpack_flags`` restores them).
        ``gmax_nx``: the global ``exp_lon.max()`` in columns.  The reference takes it over ALL dates of a call
        (streamer_index.py:106, overturning_index.py:105, cutoff_index.py:90), a stream only sees one batch at a
        time, so the default ``"full"`` uses the width of the extended grid, ``nlon + periodic_add / dlon``: the value
        the maximum has as soon as ANY date of the record holds a circumglobal contour (a batch without one then yields
        no streamers / overturnings, exactly like those dates do in the reference).  If no batch at all reaches the full
        width a warning is logged with the maximum that was seen -- re-run with ``gmax_nx=<that value>`` to get the
        reference's result for such a record.  ``None`` = every batch uses its own maximum; an int = that value.
        The flag grids / contour set of a result are only valid until its slot is reused (``depth`` batches later).
        ``climatology``: a :class:`FlagClimatology`; the flag grids of every batch are added to its counters on the
        device (the batches take consecutive time steps of its group array, from its cursor on).
        ``trackers``: a list of :class:`EventTracker` (for example one per kind); every batch's events are linked to the
        events of the last ``time_range`` hours, whose polygons stay on the device.
        ``intensity``: an iterable consumed in step with ``batches``; its item for a batch is a device or pinned-host
        tensor shaped like the batch, float32 or float64, in the batch's stored orientation, or a pair ``(u, v)`` of
        such tensors whose momentum flux (``wbk_mflux``, the reference's ``calculate_momentum_flux``) is computed on
        the device.  Every event gets the area-weighted mean of it over its cells (the ``intensity`` column), the same
        field for every contour level; without it that column is 0.  Host items are uploaded into the slot's own
        buffers, so the batch, the upload and the momentum flux included, is captured in its CUDA graph.  A batch is
        (time, lat, lon) with longitude contiguous, so the zonal means of the momentum flux are summed pairwise, as
        ``spatial.momentum_flux(u, v, lon_contiguous=True)`` does.
        """
        inten_it = iter(intensity) if intensity is not None else None
        if climatology is not None:
            climatology._check_detector(self)
        trackers = list(trackers or ())
        for tr in trackers:
            tr._check_detector(self)
        common = None
        if shared_stream and self.lib.is_cuda:
            if getattr(self, "_shared", None) is None:
                self._shared = torch.cuda.Stream(device=self.lib.device)
            common = self._shared
        full = self.nlon + self.add
        assumed = gmax_nx == "full"
        if assumed:
            gmax_nx = full
        seen_max = 0
        inflight = []
        i = 0
        starts, submitted = [tr.cursor for tr in trackers], 0
        for raw in batches:
            idx = i % depth
            if len(inflight) == depth:
                res = self.collect(inflight.pop(0), climatology, trackers)
                seen_max = max(seen_max, res.contours.max_nx)
                yield res
            item = None
            if inten_it is not None:  # checked before any device work on the batch
                item = next(inten_it, None)
                if item is None:
                    raise ValueError("the intensity iterable ended before the batches (batch {})".format(i))
                item = _intensity_item(item, raw.shape)
            for tr, start in zip(trackers, starts):  # before any device work on a batch the dates do not cover
                tr._check_steps(start + submitted, int(raw.shape[0]))
            submitted += int(raw.shape[0])
            slot = self._slot(int(raw.shape[0]), idx)
            fh = flags_host[idx] if flags_host is not None else None
            ph = packed_host[idx] if packed_host is not None else None
            inflight.append(self.submit(slot, raw, flags_host=fh, stream=common, gmax_nx=gmax_nx, packed_host=ph,
                                        intensity=item))
            i += 1
        while inflight:
            res = self.collect(inflight.pop(0), climatology, trackers)
            seen_max = max(seen_max, res.contours.max_nx)
            yield res
        if assumed and i > 0 and seen_max < full:
            logger.warning("no contour of the %d batches spans the extended grid (%d columns; widest: %d): the "
                           "reference's exp_lon.max() would be %d columns, re-run with gmax_nx=%d", i, full, seen_max,
                           seen_max, seen_max)


GROUPINGS = ("all", "month", "season")


def groups_from_dates(dates, by):
    """int32 group of every date for :class:`FlagClimatology`: ``by="all"`` puts every step in group 0, ``"month"``
    gives January = 0 .. December = 11, ``"season"`` gives DJF = 0, MAM = 1, JJA = 2, SON = 3 (December counts with
    the following January and February).  Missing dates (NaT) get -1, i.e. are not counted."""
    if by not in GROUPINGS:
        raise ValueError("by has to be one of {}, got {!r}".format(GROUPINGS, by))
    d = np.asarray(dates)
    if not np.issubdtype(d.dtype, np.datetime64):
        raise ValueError("dates have to be datetime64 values, got dtype {}".format(d.dtype))
    month = d.astype("datetime64[M]").astype(np.int64) % 12
    if by == "all":
        g = np.zeros(d.shape, dtype=np.int32)
    elif by == "month":
        g = month.astype(np.int32)
    else:
        g = ((month + 1) // 3 % 4).astype(np.int32)
    g[np.isnat(d)] = -1
    return g


def _percent(counts, steps):
    """100 * counts / steps (float64) over the leading group axis; NaN for groups without steps."""
    c = np.asarray(counts, dtype=np.float64)
    s = np.asarray(steps, dtype=np.float64).reshape((-1,) + (1,) * (c.ndim - 1))
    with np.errstate(invalid="ignore", divide="ignore"):
        out = 100.0 * c / s
    out[np.broadcast_to(s == 0, out.shape)] = np.nan
    return out


class FlagClimatology:
    """Flag-frequency climatology accumulated on the device while ``Detector.stream`` runs.

    ``groups``: int array over the global time axis of the record: the group of every time step in [0, ngroups), or
    -1 for a step that is not counted (``groups_from_dates`` makes monthly / seasonal ones).  ``ngroups`` defaults to
    ``max(groups) + 1``.  ``t0``: the time step of the record the first batch starts at (the start of a rank's shard
    in a sharded run, ``sharding.shard_range``).  The counters, uint32 ``[ngroups, 3, nlat, nlon]`` (streamers,
    overturnings, cutoffs), live on the device and are zeroed once; every batch adds the number of its steps in which a
    cell is flagged, in the group of that step, without any flag grid leaving the device.
    """

    def __init__(self, det, groups, ngroups=None, t0=0):
        if not det.want_flags:
            raise ValueError("a flag climatology needs the flag grids: the Detector has want_flags=False")
        g = np.asarray(groups)
        if g.ndim != 1 or not (np.issubdtype(g.dtype, np.integer) or g.size == 0):
            raise ValueError("groups has to be a 1-D integer array over the time axis")
        g = np.ascontiguousarray(g, dtype=np.int64)
        if ngroups is None:
            ngroups = int(g.max()) + 1 if g.size and g.max() >= 0 else 1
        ngroups = int(ngroups)
        if ngroups < 1:
            raise ValueError("ngroups has to be positive, got {}".format(ngroups))
        if g.size and (g.min() < -1 or g.max() >= ngroups):
            raise ValueError("groups has values outside [-1, {}): {}..{}".format(ngroups, int(g.min()), int(g.max())))
        if not 0 <= int(t0) <= len(g):
            raise ValueError("t0 = {} is outside the group array (length {})".format(t0, len(g)))
        self.lib = det.lib
        self.nlat, self.nlon = det.nlat, det.nlon
        self.groups = g.astype(np.int32)
        self.ngroups = ngroups
        self.cursor = int(t0)
        self._steps = np.zeros(ngroups, dtype=np.int64)
        # uint32 counters, held in an int32 tensor (the bits are read back as uint32)
        self._counts = torch.zeros((ngroups, 3, self.nlat, self.nlon), dtype=torch.int32, device=self.lib.device)

    def _check_detector(self, det):
        if not det.want_flags:
            raise ValueError("a flag climatology needs the flag grids: the Detector has want_flags=False")
        if (det.nlat, det.nlon) != (self.nlat, self.nlon):
            raise ValueError("the climatology is for a {} x {} grid, the Detector's is {} x {}".format(
                self.nlat, self.nlon, det.nlat, det.nlon))

    def _add(self, slot, pend):
        """Add the flag grids of one collected batch, on the stream the batch ran on."""
        nt, flags = int(pend["nt"]), pend["flags"]
        if self.cursor + nt > len(self.groups):
            raise ValueError("the batch covers time steps {}..{} of the record, the group array has {}".format(
                self.cursor, self.cursor + nt - 1, len(self.groups)))
        g = self.groups[self.cursor:self.cursor + nt]
        add = np.bincount(g[g >= 0], minlength=self.ngroups)
        if (self._steps + add > 0xFFFFFFFF).any():
            raise ValueError("a group would count more than 2**32 - 1 time steps")
        lib = self.lib
        st = pend.get("stream")
        with torch.cuda.stream(st) if st is not None else _null():
            if slot.clim_group is None:
                slot.clim_group = torch.empty(slot.T, dtype=torch.int32, device=lib.device)
            slot.clim_group[:nt].copy_(torch.from_numpy(g), non_blocking=True)
            # the grids as the rasteriser wrote them: kind stride nt * nlat * nlon (also for a partial last batch)
            lib.call("wbk_flag_counts", _lib.ptr(flags), 3, nt, self.nlat * self.nlon, _lib.ptr(slot.clim_group),
                     self.ngroups, _lib.ptr(self._counts), lib.stream())
        self._steps += add
        self.cursor += nt

    def counts(self):
        """uint32 ``[ngroups, 3, nlat, nlon]`` on the host (ascending coordinates, like the Detector's flag grids)."""
        if self.lib.is_cuda:
            torch.cuda.synchronize(self.lib.device)
        return self._counts.cpu().numpy().view(np.uint32)

    @property
    def steps(self):
        """int64 ``[ngroups]``: time steps counted in every group."""
        return self._steps.copy()

    def frequency(self):
        """float64 ``[ngroups, 3, nlat, nlon]``: percent of the group's time steps in which a cell is flagged (NaN for
        groups without steps)."""
        return _percent(self.counts(), self._steps)


TRACK_METHODS = ("by_overlap", "by_distance")


class EventTracker:
    """``track_events`` (events.py:151-241, ``buffer=0``) of one kind of event while ``Detector.stream`` runs.

    ``dates``: the date of every time step of the record (datetime64 or numbers, increasing); an event of a batch that
    starts at step ``cursor`` has the date ``dates[cursor + job // nlevels]``.  ``t0``: the step the first batch
    starts at (the start of a rank's shard in a sharded run, ``sharding.shard_range``).  ``time_range`` (hours) is
    required: the reference's default, the smallest positive gap between event dates, is only known at the end.

    Only the polygons of the last ``time_range`` hours are kept, on the device, in the layout of
    ``wbk_track_overlap_exact`` (``wbk_track_append`` builds them from the batch's device buffers, exactly as
    :func:`events_soup` does on the host).  Every batch is linked against that window with the kernels and the
    decision of :func:`tracking.link_events`; the links are kept as event ids on the host.  After the last batch
    :meth:`labels` gives the labels of all events of the kind in the order of the concatenated batch tables, equal to
    ``tracking.track_columnar`` on the whole record; :func:`sharding.finish_tracks` does the same for a sharded run.
    """

    def __init__(self, det, dates, kind, time_range, method="by_overlap", overlap=0, distance=1000, t0=0):
        from . import tracking

        if kind not in detect.KINDS:
            raise ValueError("kind has to be one of {}, got {!r}".format(detect.KINDS, kind))
        if method not in TRACK_METHODS:
            raise ValueError("'{}' not supported as method! Supported methods are 'by_overlap' and 'by_distance'"
                             .format(method))
        if time_range is None:
            raise ValueError("time_range (hours) is required for tracking in a stream")
        self.kind, self.method = kind, method
        self.overlap, self.distance, self.time_range = float(overlap), float(distance), time_range
        self.lib = det.lib
        self.nlat, self.nlon, self.nlevels = det.nlat, det.nlon, len(det.levels)
        self.lat, self.lon = det.lat.copy(), det.lon.copy()
        self._check_detector(det)
        d = np.asarray(dates)
        if d.ndim != 1:
            raise ValueError("dates has to be a 1-D array over the time axis")
        self.keys, window = tracking.time_keys(d)
        if len(d) > 1 and not np.all(self.keys[1:] - self.keys[:-1] > 0):
            raise ValueError("dates have to increase from one time step to the next")
        if not 0 <= int(t0) <= len(d):
            raise ValueError("t0 = {} is outside the dates array (length {})".format(t0, len(d)))
        self.win = window(time_range)
        self.cursor = int(t0)
        self.n_events = 0
        self.stats = dict(pairs_in_range=0, candidates=0, links=0, near=0)
        self.host_ms = []  # host time of every batch's tracking step
        self._links, self._near = [], []
        # the head: events within time_range of the previous shard's last step (linked by the earlier ranks)
        self._prev = self.keys[self.cursor - 1] if self.cursor > 0 else None
        self._head = None if self._prev is not None else {}
        # the window: device polygons + host keys / event ids / per-polygon ring and vertex counts
        self._wkeys = self.keys[:0].copy()
        self._wgid = np.zeros(0, dtype=np.int64)
        self._wrad = np.zeros((0, 2))
        self._wnr = np.zeros(0, dtype=np.int64)
        self._wnv = np.zeros(0, dtype=np.int64)
        self._nv = self._nr = 0
        self._buf = None  # edges, vsign, ring_off, poly_off, bbox
        # the tracker's own stream: its read-backs wait for its own work only, not for the batches queued behind the
        # collected one (with shared_stream=True they would wait for the whole pipeline)
        self._stream = torch.cuda.Stream(device=self.lib.device) if self.lib.is_cuda else None
        self._done = torch.cuda.Event() if self.lib.is_cuda else None

    def _on_stream(self):
        return torch.cuda.stream(self._stream) if self._stream is not None else _null()

    def _check_steps(self, first, nt):
        """Refuse a batch of nt steps starting at step ``first`` that runs past the dates array."""
        if first + nt > len(self.keys):
            raise ValueError("the batch covers time steps {}..{} of the record, the dates array has {}".format(
                first, first + nt - 1, len(self.keys)))

    def _check_detector(self, det):
        if self.method == "by_overlap" and not (det.want_flags and det.want_pieces):
            raise ValueError("a by_overlap tracker needs the device clipper's pieces: build the Detector with "
                             "want_flags=True and want_pieces=True")
        if ((det.nlat, det.nlon) != (self.nlat, self.nlon) or len(det.levels) != self.nlevels
                or not np.array_equal(det.lat, self.lat) or not np.array_equal(det.lon, self.lon)):
            raise ValueError("the tracker is for a {} x {} grid with {} level(s), the Detector has a different grid "
                             "({} x {}, {} level(s))".format(self.nlat, self.nlon, self.nlevels, det.nlat, det.nlon,
                                                            len(det.levels)))

    # ------------------------------------------------------------------ device window
    def _reserve(self, nv, nr, npoly):
        """Room for nv more vertices, nr more rings and npoly more polygons (grown by doubling)."""
        need = (self._nv + nv, self._nr + nr + 1, len(self._wkeys) + npoly + 1)
        b = self._buf
        if b is not None and need[0] <= len(b[0]) and need[1] <= len(b[2]) and need[2] <= len(b[3]):
            return
        dev = self.lib.device
        cap = [max(2 * c, 1024) for c in need]
        if b is not None:
            cap = [max(c, len(x)) for c, x in zip(cap, (b[0], b[2], b[3]))]
        i32 = torch.int32
        new = (torch.empty((cap[0], 4), dtype=i32, device=dev), torch.empty(cap[0], dtype=i32, device=dev),
               torch.zeros(cap[1], dtype=i32, device=dev), torch.zeros(cap[2], dtype=i32, device=dev),
               torch.empty((cap[2], 4), dtype=i32, device=dev))
        if b is not None:
            np_ = len(self._wkeys)
            new[0][:self._nv].copy_(b[0][:self._nv])
            new[1][:self._nv].copy_(b[1][:self._nv])
            new[2][:self._nr + 1].copy_(b[2][:self._nr + 1])
            new[3][:np_ + 1].copy_(b[3][:np_ + 1])
            new[4][:np_].copy_(b[4][:np_])
            if self.lib.is_cuda:
                torch.cuda.current_stream(dev).synchronize()  # nothing reads the old window any more
        self._buf = new

    def _push(self, keys, gid, rad, nr, nv):
        self._wkeys = np.concatenate([self._wkeys, keys])
        self._wgid = np.concatenate([self._wgid, gid])
        self._wrad = np.concatenate([self._wrad, rad])
        self._wnr = np.concatenate([self._wnr, nr])
        self._wnv = np.concatenate([self._wnv, nv])
        self._nr += int(nr.sum())
        self._nv += int(nv.sum())

    def _evict(self, m):
        """Drop the first m window events (their dates can no longer link to a later date)."""
        if m == 0:
            return
        dr, dv = int(self._wnr[:m].sum()), int(self._wnv[:m].sum())
        np_ = len(self._wkeys)
        if self.method == "by_overlap" and self._buf is not None:
            e, vs, ro, po, bb = self._buf
            kv, kr, kp = self._nv - dv, self._nr - dr, np_ - m
            e[:kv].copy_(e[dv:self._nv].clone())
            vs[:kv].copy_(vs[dv:self._nv].clone())
            ro[:kr + 1].copy_(ro[dr:self._nr + 1] - dv)
            po[:kp + 1].copy_(po[m:np_ + 1] - dr)
            bb[:kp].copy_(bb[m:np_].clone())
        self._wkeys, self._wgid, self._wrad = self._wkeys[m:], self._wgid[m:], self._wrad[m:]
        self._wnr, self._wnv = self._wnr[m:], self._wnv[m:]
        self._nr -= dr
        self._nv -= dv

    def _snapshot(self, m):
        """Host copy of the first m window events (the head of a shard)."""
        dr, dv = int(self._wnr[:m].sum()), int(self._wnv[:m].sum())
        h = dict(keys=self._wkeys[:m].copy(), gid=self._wgid[:m].copy(), rad=self._wrad[:m].copy(),
                 nr=self._wnr[:m].copy(), nv=self._wnv[:m].copy())
        if self.method == "by_overlap" and m:
            e, vs, ro, po, bb = self._buf
            h.update(edges=e[:dv].cpu().numpy(), vsign=vs[:dv].cpu().numpy(), ring_off=ro[:dr + 1].cpu().numpy(),
                     poly_off=po[:m + 1].cpu().numpy(), bbox=bb[:m].cpu().numpy())
        return h

    def _append_host(self, h, gid):
        """Append polygons given on the host (a published head) to the window."""
        m = len(h["keys"])
        if self.method == "by_overlap" and m:
            self._reserve(int(h["nv"].sum()), int(h["nr"].sum()), m)
            e, vs, ro, po, bb = self._buf
            np_, dv = len(self._wkeys), len(h["edges"])
            dev = self.lib.device
            e[self._nv:self._nv + dv].copy_(torch.from_numpy(h["edges"]).to(dev))
            vs[self._nv:self._nv + dv].copy_(torch.from_numpy(h["vsign"]).to(dev))
            ro[self._nr:self._nr + len(h["ring_off"])].copy_(torch.from_numpy(h["ring_off"] + self._nv).to(dev))
            po[np_:np_ + m + 1].copy_(torch.from_numpy(h["poly_off"] + self._nr).to(dev))
            bb[np_:np_ + m].copy_(torch.from_numpy(h["bbox"]).to(dev))
        self._push(h["keys"], gid, h["rad"], h["nr"], h["nv"])

    # ------------------------------------------------------------------ linking
    def _link(self, W, owned):
        """Link the window events [0, owned) to the events [W, len) appended last.  Returns (pairs in range, links as
        window positions)."""
        from . import tracking

        lib = self.lib
        n = len(self._wkeys)
        lo, hi = tracking.windows(self._wkeys, self.win)
        lo[:W] = np.maximum(lo[:W], W)
        lo[owned:] = hi[owned:]
        hi = np.maximum(hi, lo)
        n_in = int((hi - lo).sum())
        empty = np.zeros((0, 2), dtype=np.int32)
        if n_in == 0:
            return 0, empty, empty
        dev = lib.device
        st = lib.stream()
        d_lo, d_hi = torch.from_numpy(lo).to(dev), torch.from_numpy(hi).to(dev)
        d_pairs = torch.empty((n_in, 2), dtype=torch.int32, device=dev)
        d_count = torch.zeros(1, dtype=torch.int32, device=dev)
        box = self._buf[4] if self.method == "by_overlap" and self.overlap >= 0 else None
        lib.call("wbk_track_candidates", _lib.ptr(d_lo), _lib.ptr(d_hi), _lib.ptr(box), n, _lib.ptr(d_pairs), n_in,
                 _lib.ptr(d_count), st)
        m = int(d_count.cpu()[0])
        pairs = d_pairs[:m].cpu().numpy()
        if self.method == "by_distance":
            links, near = tracking.decide_pairs(pairs, "by_distance", distance=self.distance, rad=self._wrad,
                                                dist=lambda p: tracking.pair_distances(self._wrad, p))
        else:
            e, vs, ro, po, _ = self._buf

            def exact(p):
                d_p = torch.from_numpy(np.ascontiguousarray(p, dtype=np.int32)).to(dev)
                out = torch.empty(len(p), dtype=torch.int32, device=dev)
                lib.call("wbk_track_overlap_exact", _lib.ptr(e), _lib.ptr(vs), _lib.ptr(ro), _lib.ptr(po),
                         _lib.ptr(d_p), len(p), _lib.ptr(out), lib.stream())
                return out.cpu().numpy()

            def areas(p):
                if len(p) == 0:
                    return np.zeros((0, 3))
                xy = e[:self._nv, :2].to(torch.float64).contiguous()
                d_p = torch.from_numpy(np.ascontiguousarray(p, dtype=np.int32)).to(dev)
                out = torch.empty((len(p), 3), dtype=torch.float64, device=dev)
                lib.call("wbk_track_overlap", _lib.ptr(xy), _lib.ptr(ro), _lib.ptr(po), _lib.ptr(d_p), len(p),
                         _lib.ptr(out), lib.stream())
                return out.cpu().numpy()

            links, near = tracking.decide_pairs(pairs, "by_overlap", self.overlap, exact=exact, areas=areas)
        self.stats["pairs_in_range"] += n_in
        self.stats["candidates"] += len(pairs)
        self.stats["links"] += len(links)
        self.stats["near"] += len(near)
        return n_in, links, near

    def _add(self, slot, pend, tables, counts):
        """Append and link the events of one collected batch, on the stream the batch ran on."""
        import time

        tick = time.perf_counter()
        nt = int(pend["nt"])
        self._check_steps(self.cursor, nt)
        st = pend.get("stream")
        with self._on_stream():
            if st is not None:
                self._stream.wait_event(slot.done)  # the batch's buffers (final: collect has waited for this event)
            self._add_batch(slot, tables, counts, nt)
            if st is not None:
                # the slot's next batch overwrites the buffers wbk_track_append reads
                self._done.record(self._stream)
                st.wait_event(self._done)
        self.cursor += nt
        self.host_ms.append(1e3 * (time.perf_counter() - tick))

    def _add_batch(self, slot, tables, counts, nt):
        from . import tracking

        k = detect.KINDS.index(self.kind)
        tab = tables[self.kind]
        n, first = len(tab), int(sum(counts[:k]))
        keys = self.keys[self.cursor + tab.job.astype(np.int64) // self.nlevels]
        gid = self.n_events + np.arange(n, dtype=np.int64)
        rad = np.zeros((n, 2))
        nr = np.zeros(n, dtype=np.int64)
        nv = np.zeros(n, dtype=np.int64)
        W = len(self._wkeys)
        if n and self.method == "by_distance":
            # the reference feeds (lon, lat) where haversine expects (lat, lon) (events.py:189-195); kept
            props = detect.finish_properties(tab, self.lon, self.lat, self.nlon)
            rad = np.radians(np.asarray(props["com"], dtype=np.float64).reshape(-1, 2))
        elif n:
            npc, _, clip_over = (int(v) for v in slot.h_sp_cnt.numpy()[:3])
            if clip_over:
                raise _lib.WbkError(_lib.ERR_CAPACITY, "the device clipper's arenas overflowed: the pieces of the events "
                                                       "that straddle the last meridian are incomplete")
            split = tab.split == 1
            is_box = self.kind == "overturnings"
            ro = slot.h_ring_off.numpy()
            nv[:] = 4 if is_box else np.diff(ro[first:first + n + 1])
            nr[:] = 1
            pev = slot.h_sp_ev.numpy()[:npc].astype(np.int64) - first
            plen = np.diff(slot.h_sp_off.numpy()[:npc + 1]).astype(np.int64)
            mine = (pev >= 0) & (pev < n)
            mine[mine] = split[pev[mine]]
            nr[split] = np.bincount(pev[mine], minlength=n)[split]
            nv[split] = np.bincount(pev[mine], weights=plen[mine], minlength=n).astype(np.int64)[split]
            self._reserve(int(nv.sum()), int(nr.sum()), n)
            e, vs, wro, wpo, bb = self._buf
            lib = self.lib
            lib.call("wbk_track_append", _lib.ptr(slot.ev_int), _lib.ptr(slot.ring_off), _lib.ptr(slot.ring_pts),
                     _lib.ptr(slot.sp_ev), _lib.ptr(slot.sp_off), _lib.ptr(slot.sp_xy), npc, first, n, int(is_box),
                     self.nlon, int(nr.sum()), int(nv.sum()), _lib.ptr(e), _lib.ptr(vs), _lib.ptr(wro), _lib.ptr(wpo),
                     _lib.ptr(bb), self._nv, self._nr, W, len(e), len(wro), len(wpo), lib.stream())
        self._push(keys, gid, rad, nr, nv)
        self.n_events += n
        if n:
            _, links, near = self._link(W, len(self._wkeys))
            self._links.append(self._wgid[links.astype(np.int64)].reshape(-1, 2))
            self._near.append(self._wgid[near.astype(np.int64)].reshape(-1, 2))
        # the head of a shard is complete once the next date lies beyond time_range of the previous shard's last step
        end = self.cursor + nt
        nxt = self.keys[end] if end < len(self.keys) else None
        if self._head is None and (nxt is None or not nxt - self._prev <= self.win):
            self._head = self._snapshot(self._head_size())
        if nxt is None:
            self._evict(len(self._wkeys))
        else:
            self._evict(int(np.count_nonzero(~(nxt - self._wkeys <= self.win))))

    def _head_size(self):
        return int(np.count_nonzero(self._wkeys - self._prev <= self.win))

    # ------------------------------------------------------------------ results
    def _pairs(self, parts):
        out = np.concatenate(parts) if parts else np.zeros((0, 2), dtype=np.int64)
        return out[np.lexsort((out[:, 1], out[:, 0]))] if len(out) else out

    @property
    def links(self):
        """int64 [m, 2]: the linked event pairs (event ids in the order of the concatenated batch tables)."""
        return self._pairs(self._links)

    @property
    def near(self):
        """int64 [m, 2]: the pairs decided within ``tracking.NEAR_REL`` of a threshold (event ids, sorted)."""
        return self._pairs(self._near)

    def labels(self):
        """int64 labels of all events tracked so far (``track_events``' ``label`` column in the order of the
        concatenated batch tables).  Raises ValueError when no pair of events was in range, like the reference."""
        from . import tracking

        if self.stats["pairs_in_range"] == 0:
            raise ValueError("No events detected in the time range: {}".format(self.time_range))
        return tracking.labels_from_links(self.n_events, self.links)


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def summarize(res):
    """Small dict of counts (used by the benchmark's result read-back and the tests)."""
    return dict(
        ntime=res.ntime, contours=res.contours.ncontours, points=res.contours.npoints,
        streamers=len(res.tables["streamers"]), overturnings=len(res.tables["overturnings"]),
        cutoffs=len(res.tables["cutoffs"]), split=res.n_split, near=res.near_total,
        segments=(res.work or {}).get("segments", 0), pairs=(res.work or {}).get("pairs", 0),
    )


def events_soup(res, kind, det):
    """Lattice polygons of the events of one kind of a BatchResult, as ``track_events`` sees them after
    ``transform_polygons`` (utils/index_utils.py:129-184): index coordinates of the REAL grid, folded with
    ``x % nlon``, events that straddle the last meridian split into their pieces (a multipolygon).
    Returns ``(tracking.PolygonSoup, com)`` with ``com`` the (lon, lat) centre-of-mass column."""
    from . import geometry, tracking

    tab = res.tables[kind]
    n = len(tab)
    nlon = det.nlon
    if kind == "overturnings":
        x0, y0, x1, y1 = (tab.box[:, k].astype(np.int64) for k in range(4))
        xy = np.stack([np.c_[x1, y0], np.c_[x1, y1], np.c_[x0, y1], np.c_[x0, y0]], axis=1).reshape(-1, 2)
        off = np.arange(n + 1, dtype=np.int64) * 4
    else:
        off = tab.rings.off - tab.rings.off[0]
        p = tab.rings.packed
        xy = np.c_[(p & 0xFFFF).astype(np.int64), (p >> 16).astype(np.int64)]
    straddle = np.nonzero(tab.split == 1)[0]
    if len(straddle) == 0:
        xy[:, 0] %= nlon
        soup = tracking.PolygonSoup(xy.astype(np.int32), off, np.arange(n + 1), True)
    elif res.pieces is not None and not res.pieces["overflow"]:
        # pieces from the device clipper (wbk_split_fetch): everything stays vectorised.  Rows of this kind start at
        # `first` in the kind-major gather order of the batch
        first = int(sum(res.counts[:detect.KINDS.index(kind)]))
        allxy, ring_off, poly_off = geometry.interleave_pieces(xy, off, tab.split, res.pieces, first, nlon)
        soup = tracking.PolygonSoup(allxy.astype(np.int32), ring_off, poly_off, True)
    else:
        # only the few events that straddle the meridian are rebuilt one by one
        ring_xy, ring_len, poly_nr = [], [], np.ones(n, dtype=np.int64)
        prev = 0
        for e in straddle:
            a, b = off[prev], off[e]
            if b > a:
                seg = xy[a:b].copy()
                seg[:, 0] %= nlon
                ring_xy.append(seg)
                ring_len.extend(np.diff(off[prev:e + 1]).tolist())
            pieces = geometry.transform_ring(xy[off[e]:off[e + 1]], nlon)
            poly_nr[e] = len(pieces)
            for pc in pieces:
                ring_xy.append(np.asarray(pc, dtype=np.int64).reshape(-1, 2))
                ring_len.append(len(pc))
            prev = e + 1
        if off[n] > off[prev]:
            seg = xy[off[prev]:off[n]].copy()
            seg[:, 0] %= nlon
            ring_xy.append(seg)
            ring_len.extend(np.diff(off[prev:n + 1]).tolist())
        allxy = np.concatenate(ring_xy) if ring_xy else np.zeros((0, 2), dtype=np.int64)
        soup = tracking.PolygonSoup(allxy.astype(np.int32), np.r_[0, np.cumsum(ring_len)], np.r_[0, np.cumsum(poly_nr)],
                                    True)
    props = detect.finish_properties(tab, det.lon, det.lat, nlon)
    return soup, np.asarray(props["com"], dtype=np.float64).reshape(-1, 2)
