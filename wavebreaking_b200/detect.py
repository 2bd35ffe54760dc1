"""Batched detection core: device contexts, contour sets and the index kernels' host wrappers.

Columnar layer under the drop-in API (``wavebreaking_b200.api``).  A *job* is one
(time step, contour level); jobs are ordered time-outer, level-inner like the reference's
``iterate_time_dimension`` / ``iterate_contour_levels`` loops (utils/index_utils.py:217-258).
"""

import ctypes
from dataclasses import dataclass
from fractions import Fraction

import numpy as np
import torch

from . import _lib


def _iptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int))


def default_caps(nlat, nlon, add, njobs):
    """Arena capacities that fit smooth geophysical fields with headroom (regrown on overflow)."""
    W = nlon + add
    p2 = lambda v: 1 << max(4, int(np.ceil(np.log2(max(v, 2)))))
    return dict(max_jobs=int(njobs), seg_cap=p2(8 * (W + nlat)), contour_cap=p2(max(256, W // 2)), sel_cap=2,
                pair_cap=p2(48 * W), event_cap=256)


class Context:
    """Owns a wbk_ctx and its torch-allocated device workspace."""

    def __init__(self, nlat, nlon, add, caps):
        self.lib = _lib.get()
        self.nlat, self.nlon, self.add = int(nlat), int(nlon), int(add)
        self.caps = dict(caps)
        c = _lib.Caps(**self.caps)
        need = self.lib.cdll.wbk_workspace_bytes(ctypes.byref(c), self.nlat, self.nlon, self.add)
        if need == 0:
            raise ValueError("invalid capacities / grid for wbk_create: {}".format(self.caps))
        self.workspace = torch.empty(need + 256, dtype=torch.uint8, device=self.lib.device)
        base = self.workspace.data_ptr()
        aligned = (base + 255) & ~255
        self.handle = ctypes.c_void_p()
        self.lib.call("wbk_create", ctypes.byref(self.handle), ctypes.byref(c), self.nlat, self.nlon, self.add,
                      ctypes.c_void_p(aligned), need)

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle:
            self.lib.cdll.wbk_destroy(self.handle)
            self.handle = None
            self.workspace = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_CTX_CACHE = {}


def get_context(nlat, nlon, add, njobs, min_caps=None):
    """A cached context for this grid whose capacities cover ``njobs`` (and ``min_caps``)."""
    key = (int(nlat), int(nlon), int(add), _lib.get().path)
    want = default_caps(nlat, nlon, add, njobs)
    if min_caps:
        for k, v in min_caps.items():
            want[k] = max(want[k], int(v))
    ctx = _CTX_CACHE.get(key)
    if ctx is not None and all(ctx.caps[k] >= want[k] for k in want):
        return ctx
    if ctx is not None:
        for k in want:
            want[k] = max(want[k], ctx.caps[k])
        ctx.close()
    ctx = Context(nlat, nlon, add, want)
    _CTX_CACHE[key] = ctx
    return ctx


def clear_contexts():
    for ctx in _CTX_CACHE.values():
        ctx.close()
    _CTX_CACHE.clear()


@dataclass
class ContourSet:
    """Packed contours of a batch (device tensors) in index coordinates of the extended grid."""

    njobs: int
    nlevels: int
    nlat: int
    nlon: int
    add: int
    levels: np.ndarray
    job_off: torch.Tensor   # int32 [njobs + 1]
    pt_off: torch.Tensor    # int32 [C + 1]
    meta: torch.Tensor      # int32 [C, 4]: closed, nx, sum_y, job
    pts: torch.Tensor       # uint32-as-int32 [P]: x | y << 16
    status: np.ndarray      # int32 [njobs]
    max_nx: int
    h_ncontours: np.ndarray
    h_npoints: np.ndarray
    _host: dict = None

    @property
    def ncontours(self):
        return int(self.pt_off.shape[0]) - 1

    @property
    def npoints(self):
        return int(self.pts.shape[0])

    def host(self):
        """Host copies: dict(job_off, pt_off, closed, nx, sum_y, job, x, y)."""
        if self._host is None:
            meta = self.meta.cpu().numpy().reshape(-1, 4)
            pts = self.pts.cpu().numpy().view(np.uint32)
            self._host = dict(
                job_off=self.job_off.cpu().numpy(), pt_off=self.pt_off.cpu().numpy(),
                closed=meta[:, 0].astype(bool), nx=meta[:, 1].copy(), sum_y=meta[:, 2].copy(), job=meta[:, 3].copy(),
                x=(pts & 0xFFFF).astype(np.int64), y=(pts >> 16).astype(np.int64),
            )
        return self._host

    def contour_points(self, c):
        h = self.host()
        a, b = h["pt_off"][c], h["pt_off"][c + 1]
        return np.c_[h["x"][a:b], h["y"][a:b]]


def contours(field, levels, add, caps=None):
    """Contours of every (time step, level) of ``field`` [ntime, nlat, nlon] (device tensor).

    contour_index.py:86-175 with ``original_coordinates=False``.  Retries with larger arenas
    when a job overflows its capacity.
    """
    lib = _lib.get()
    if field.dim() != 3:
        raise ValueError("expected [ntime, nlat, nlon]")
    field = field.contiguous()
    ntime, nlat, nlon = (int(v) for v in field.shape)
    levels = np.ascontiguousarray(np.atleast_1d(np.asarray(levels, dtype=np.float64)))
    nlevels = len(levels)
    njobs = ntime * nlevels
    grow = dict(caps or {})
    for _attempt in range(8):
        ctx = get_context(nlat, nlon, add, max(njobs, 1), grow)
        lib.call("wbk_contours", ctx.handle, _lib.ptr(field), _lib.dtype_code(field.dtype), ntime,
                 levels.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), nlevels, lib.stream())
        nc = np.zeros(max(njobs, 1), dtype=np.int32)
        npnt = np.zeros(max(njobs, 1), dtype=np.int32)
        status = np.zeros(max(njobs, 1), dtype=np.int32)
        max_nx = ctypes.c_int(0)
        try:
            lib.call("wbk_contours_counts", ctx.handle, _iptr(nc), _iptr(npnt), _iptr(status), ctypes.byref(max_nx),
                     lib.stream())
            break
        except _lib.CapacityError:
            if status.max() & _lib.ST_SEG_OVERFLOW or np.any(status & _lib.ST_SEG_OVERFLOW):
                grow["seg_cap"] = ctx.caps["seg_cap"] * 2
            if np.any(status & _lib.ST_CONTOUR_OVERFLOW):
                grow["contour_cap"] = ctx.caps["contour_cap"] * 2
    else:
        raise _lib.WbkError(_lib.ERR_CAPACITY, "contour arenas still overflow after 8 regrowths")
    nc, npnt, status = nc[:njobs], npnt[:njobs], status[:njobs]
    C, Pn = int(nc.sum()), int(npnt.sum())
    dev = lib.device
    job_off = torch.empty(njobs + 1, dtype=torch.int32, device=dev)
    pt_off = torch.zeros(C + 1, dtype=torch.int32, device=dev)
    meta = torch.empty((C, 4), dtype=torch.int32, device=dev)
    pts = torch.empty(Pn, dtype=torch.int32, device=dev)
    if njobs > 0:
        lib.call("wbk_contours_pack", ctx.handle, _iptr(nc), _iptr(npnt), _lib.ptr(job_off), _lib.ptr(pt_off),
                 _lib.ptr(meta) if C else _lib.ptr(job_off), _lib.ptr(pts) if Pn else _lib.ptr(job_off), lib.stream())
    else:
        job_off.zero_()
    return ContourSet(njobs=njobs, nlevels=nlevels, nlat=nlat, nlon=nlon, add=int(add), levels=levels,
                      job_off=job_off, pt_off=pt_off, meta=meta, pts=pts, status=status.copy(),
                      max_nx=int(max_nx.value), h_ncontours=nc.copy(), h_npoints=npnt.copy())


# --------------------------------------------------------------------------------------------- index stage
KINDS = ("streamers", "overturnings", "cutoffs")


def cell_area_km2(dlon, dlat):
    """Equatorial cell area used by calculate_properties (utils/index_utils.py:58-60)."""
    return np.round(6371 * 2 * np.pi / (360 / ((dlon + dlat) / 2))) ** 2


def coord_tables(lat, lon, dlon, dlat, lib=None):
    """Device doubles [lat_deg | lat_rad | cos(lat_rad) | cell area | lon_rad] (wbk_index_run's d_coords).

    Built on the host with the calls the reference makes (np.radians, np.cos for the areas) and
    libm's cos for the haversine factor (what sklearn's C code evaluates).
    """
    import math

    lib = lib or _lib.get()
    lat = np.asarray(lat, dtype=np.float64)
    lon = np.asarray(lon, dtype=np.float64)
    lat_rad = np.radians(lat)
    cos_lat = np.array([math.cos(v) for v in lat_rad])
    area = np.cos(np.radians(lat)) * cell_area_km2(dlon, dlat)
    tab = np.concatenate([lat, lat_rad, cos_lat, area, np.radians(lon)])
    return torch.from_numpy(tab).to(lib.device)


class LazyRings:
    """Ragged ring vertices of the events of one table; ring e is built on access as an (n, 2) int array."""

    def __init__(self, off, packed):
        self.off = np.asarray(off, dtype=np.int64)
        self.packed = np.asarray(packed).view(np.uint32)

    def __len__(self):
        return len(self.off) - 1

    def __getitem__(self, e):
        if isinstance(e, slice):
            return [self[i] for i in range(*e.indices(len(self)))]
        if e < 0:
            e += len(self)
        p = self.packed[self.off[e] - self.off[0]: self.off[e + 1] - self.off[0]]
        return np.c_[(p & 0xFFFF).astype(np.int64), (p >> 16).astype(np.int64)]

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    @property
    def nbytes(self):
        return self.packed.nbytes + self.off.nbytes


@dataclass
class EventTable:
    """Events of one index in reference row order (host arrays)."""

    kind: str
    job: np.ndarray        # [n]
    contour: np.ndarray    # [n] index into the contour set
    ind1: np.ndarray
    ind2: np.ndarray
    box: np.ndarray        # [n, 4]: x0, y0, x1, y1 (overturning box / bounding box)
    orientation: np.ndarray  # 0 cyclonic, 1 anticyclonic (overturnings)
    split: np.ndarray      # 0 on the real grid, 1 straddles the last meridian, 2 entirely in the extension
    near: np.ndarray       # streamers: base-point decision within 1e-9 of a threshold
    sums: np.ndarray       # [n, 6]: sum a, sum a*data, sum a*intensity, sum a*x, sum a*y, member count
    rings: object = None   # LazyRings: index-space ring of every streamer / cutoff event (fetched with the batch)

    def __len__(self):
        return len(self.job)


def run_indices(cs, data, coords, dlon, dlat, intensity=None, which=KINDS, gmax_nx=None, geo_dis=800.0,
                cont_dis=1500.0, range_group=5.0, ot_min_exp=5.0, co_min_exp=5.0, want_flags=False, min_caps=None,
                want_pieces=False):
    """Streamers / overturnings / cutoffs + properties (+ to_xarray flags) for a contour set.

    ``data`` / ``intensity``: device tensors [ntime, nlat, nlon].  Returns ``(tables, flags)`` where
    tables maps kind -> EventTable and flags is an int8 tensor [3, ntime, nlat, nlon] or None.
    Events that straddle the last meridian (split == 1) are clipped and rasterised on the device too.
    ``want_pieces``: returns ``(tables, flags, pieces)`` with the device clipper's pieces of those events
    (``geometry.interleave_pieces``), or None for pieces when the clipper's arenas overflowed.
    """
    lib = _lib.get()
    ntime = int(data.shape[0])
    nlevels = cs.nlevels
    prm = _lib.IndexParams(
        do_streamers=int("streamers" in which), do_overturnings=int("overturnings" in which),
        do_cutoffs=int("cutoffs" in which), gmax_nx=int(cs.max_nx if gmax_nx is None else gmax_nx),
        dlon=float(dlon), dlat=float(dlat), geo_dis=float(geo_dis), cont_dis=float(cont_dis),
        range_group=float(range_group), ot_min_exp=float(ot_min_exp), co_min_exp=float(co_min_exp))
    work = torch.empty(2 * max(cs.npoints, 1), dtype=torch.float64, device=lib.device)
    flags = None
    if want_flags:
        flags = torch.empty((3, ntime, cs.nlat, cs.nlon), dtype=torch.int8, device=lib.device)
    data = data.contiguous()
    if intensity is not None:
        intensity = intensity.contiguous().to(data.dtype)
    grow = dict(min_caps or {})
    counts = np.zeros((3, max(cs.njobs, 1)), dtype=np.int32)
    status = np.zeros(max(cs.njobs, 1), dtype=np.int32)
    for _attempt in range(8):
        ctx = get_context(cs.nlat, cs.nlon, cs.add, max(cs.njobs, 1), grow)
        lib.call("wbk_index_run", ctx.handle, cs.njobs, nlevels, _lib.ptr(cs.job_off), _lib.ptr(cs.pt_off),
                 _lib.ptr(cs.meta), _lib.ptr(cs.pts), cs.ncontours, cs.npoints, _lib.ptr(coords), _lib.ptr(work),
                 ctypes.byref(prm), lib.stream())
        lib.call("wbk_events_raster", ctx.handle, _lib.ptr(cs.job_off), _lib.ptr(cs.pt_off), _lib.ptr(cs.pts),
                 _lib.ptr(coords), _lib.ptr(data), _lib.dtype_code(data.dtype), _lib.ptr(intensity),
                 _lib.dtype_code(data.dtype), 0, 0, ntime, _lib.ptr(flags), ctypes.byref(prm), lib.stream())
        try:
            lib.call("wbk_events_counts", ctx.handle, _iptr(counts), _iptr(status), lib.stream())
            break
        except _lib.CapacityError:
            if np.any(status & _lib.ST_PAIR_OVERFLOW):
                grow["pair_cap"] = ctx.caps["pair_cap"] * 4
            if np.any(status & _lib.ST_EVENT_OVERFLOW):
                grow["event_cap"] = ctx.caps["event_cap"] * 4
            if np.any(status & _lib.ST_SEL_OVERFLOW):
                grow["sel_cap"] = ctx.caps["sel_cap"] * 4
    else:
        raise _lib.WbkError(_lib.ERR_CAPACITY, "index arenas still overflow after 8 regrowths")
    counts = counts.reshape(3, -1)[:, :cs.njobs] if cs.njobs else counts[:, :0]
    tables = {}
    for kind_id, kind in enumerate(KINDS):
        n = int(counts[kind_id].sum()) if cs.njobs else 0
        ints = np.zeros((n, _lib.EV_INTS), dtype=np.int32)
        f64 = np.zeros((n, _lib.EV_F64), dtype=np.float64)
        job = np.zeros(n, dtype=np.int32)
        if n:
            lib.call("wbk_events_fetch", ctx.handle, kind_id, n, _iptr(ints),
                     f64.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), _iptr(job), lib.stream())
        tables[kind] = EventTable(kind=kind, job=job, contour=ints[:, 0].copy(), ind1=ints[:, 1].copy(),
                                  ind2=ints[:, 2].copy(), box=ints[:, 3:7].copy(), orientation=ints[:, 7].copy(),
                                  split=ints[:, 8].copy(), near=ints[:, 9].copy(), sums=f64)
    if not want_pieces:
        return tables, flags
    pieces = None
    if any(int((t.split == 1).sum()) for t in tables.values()):
        pieces = _fetch_pieces(lib, ctx, cs)
    return tables, flags, pieces


def _fetch_pieces(lib, ctx, cs):
    """Pieces of the straddling events from the device clipper (wbk_split_clip + wbk_split_fetch)."""
    lib.call("wbk_split_clip", ctx.handle, _lib.ptr(cs.pt_off), _lib.ptr(cs.pts), lib.stream())
    cap_r, cap_v = 4096, 1 << 18
    for _attempt in range(6):
        ev = torch.empty(cap_r, dtype=torch.int32, device=lib.device)
        off = torch.empty(cap_r + 1, dtype=torch.int32, device=lib.device)
        xy = torch.empty((cap_v, 2), dtype=torch.int32, device=lib.device)
        cnt = torch.zeros(4, dtype=torch.int32, device=lib.device)
        lib.call("wbk_split_fetch", ctx.handle, _lib.ptr(ev), _lib.ptr(off), _lib.ptr(xy), cap_r, cap_v, _lib.ptr(cnt),
                 lib.stream())
        npc, nvx, over = (int(v) for v in cnt.cpu().numpy()[:3])
        if over:
            return None  # the clipper's own arenas were too small: the caller clips these events on the host
        if npc <= cap_r and nvx <= cap_v:
            return dict(ev=ev[:npc].cpu().numpy(), off=off[:npc + 1].cpu().numpy().astype(np.int64),
                        xy=xy[:nvx].cpu().numpy(), overflow=False)
        cap_r, cap_v = max(cap_r, 2 * npc), max(cap_v, 2 * nvx)
    return None


def event_rings(cs, table):
    """Index-space ring (n, 2) of every event of a table (host)."""
    if table.kind != "overturnings" and table.rings is not None:
        return list(table.rings)
    rings = []
    h = cs.host() if table.kind != "overturnings" else None
    for e in range(len(table)):
        if table.kind == "overturnings":
            x0, y0, x1, y1 = (int(v) for v in table.box[e])
            rings.append(np.array([[x1, y0], [x1, y1], [x0, y1], [x0, y0]], dtype=np.int64))
        else:
            a = h["pt_off"][table.contour[e]]
            rings.append(np.c_[h["x"][a + table.ind1[e]: a + table.ind2[e] + 1],
                               h["y"][a + table.ind1[e]: a + table.ind2[e] + 1]])
    return rings


def grid_ratio(dlon, dlat):
    """``dlon : dlat`` as the reduced ratio ``(p, q)`` that the to_xarray buffer of an anisotropic grid is measured
    in (the rule of ``wbk_events_raster`` / ``wbk_rasterize_rings_grid``; raises ``ValueError`` on grids they refuse).

    Spacings within 1e-9 (relative) of each other are the isotropic grid ``(1, 1)``.  Otherwise ``dlon / dlat`` must
    be exactly ``p / q`` with ``p, q <= 64`` (the integer products of the membership test stay exact) and
    ``max(dlon, dlat) / min(dlon, dlat) < 3`` (the buffer discs around vertices hold no other grid point)."""
    dlon, dlat = float(dlon), float(dlat)
    if not (np.isfinite(dlon) and np.isfinite(dlat) and dlon > 0 and dlat > 0):
        raise ValueError("grid spacings dlon={!r}, dlat={!r} must be positive and finite".format(dlon, dlat))
    if abs(dlon - dlat) <= 1e-9 * abs(dlon):
        return 1, 1
    ratio = Fraction(dlon) / Fraction(dlat)
    p, q = ratio.numerator, ratio.denominator
    if p > 64 or q > 64:
        raise ValueError("flag grids need dlon / dlat to be an exact ratio p/q of integers <= 64; "
                         "dlon={!r}, dlat={!r}".format(dlon, dlat))
    if max(p, q) >= 3 * min(p, q):
        raise ValueError("flag grids need an aspect ratio max(dlon, dlat) / min(dlon, dlat) < 3; "
                         "dlon={!r}, dlat={!r}".format(dlon, dlat))
    return p, q


def rasterize_rings(rings, ring_t, nlat, nlon, ntime, r_cells=None, out_i8=None, values=None, spacing=None):
    """OR lattice rings into an int8 grid (or write ``values`` into a float64 grid, last ring wins).

    The buffer is ``r_cells`` grid cells, or with ``spacing=(dlon, dlat)`` the to_xarray buffer
    ``(dlon + dlat) / 4`` measured in degrees (``wbk_rasterize_rings_grid``; see :func:`grid_ratio`)."""
    if (r_cells is None) == (spacing is None):
        raise ValueError("rasterize_rings: give exactly one of r_cells and spacing")
    if spacing is not None:
        grid_ratio(*spacing)
        fn, radius = "wbk_rasterize_rings_grid", [float(spacing[0]), float(spacing[1])]
    else:
        fn, radius = "wbk_rasterize_rings", [float(r_cells) ** 2]
    lib = _lib.get()
    dev = lib.device
    n = len(rings)
    if out_i8 is None and values is None:
        out_i8 = torch.zeros((ntime, nlat, nlon), dtype=torch.int8, device=dev)
    if n == 0:
        return out_i8
    off = np.zeros(n + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(r) for r in rings])
    xy = np.ascontiguousarray(np.concatenate([np.asarray(r, dtype=np.int32).reshape(-1, 2) for r in rings]),
                              dtype=np.int32)
    d_xy = torch.from_numpy(xy).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    d_t = torch.from_numpy(np.ascontiguousarray(ring_t, dtype=np.int32)).to(dev)
    if values is None:
        lib.call(fn, _lib.ptr(d_xy), _lib.ptr(d_off), _lib.ptr(d_t), None, n, nlat, nlon, ntime, *radius,
                 _lib.ptr(out_i8), None, None, lib.stream())
        return out_i8
    out, vals = values
    d_val = torch.from_numpy(np.ascontiguousarray(vals, dtype=np.float64)).to(dev)
    owner = torch.empty((ntime, nlat, nlon), dtype=torch.int32, device=dev)
    lib.call(fn, _lib.ptr(d_xy), _lib.ptr(d_off), _lib.ptr(d_t), _lib.ptr(d_val), n, nlat, nlon, ntime, *radius,
             None, _lib.ptr(out), _lib.ptr(owner), lib.stream())
    return out


def finish_properties(table, lon, lat, nlon):
    """com / mean_var / intensity / event_area columns from the device sums (index_utils.py:105-120).

    ``com_near_integer`` marks the events whose area-weighted mean index lies within 1e-12 (relative) of an integer:
    the reference truncates the quotient of two pandas (Kahan) sums (``.astype("int")``, index_utils.py:105-106), and
    for an event that is symmetric about a grid line -- a single column of cells, say -- the exact quotient IS an
    integer, so the last bit of the summation decides between two neighbouring grid points.  The device sums are
    exact (double-double); in that case the reference may name the neighbouring point."""
    s = table.sums
    with np.errstate(divide="ignore", invalid="ignore"):
        qx = s[:, 3] / s[:, 0] if len(s) else np.zeros(0)
        qy = s[:, 4] / s[:, 0] if len(s) else np.zeros(0)
        xi = qx.astype("int") % nlon
        yi = qy.astype("int")
        mean_var = np.round(s[:, 1] / s[:, 0], 2)
        intensity = np.round(s[:, 2] / s[:, 0], 2)
        near = (np.abs(qx - np.rint(qx)) <= 1e-12 * np.maximum(np.abs(qx), 1.0)) | \
               (np.abs(qy - np.rint(qy)) <= 1e-12 * np.maximum(np.abs(qy), 1.0))
    com = list(map(tuple, np.c_[np.asarray(lon)[xi], np.asarray(lat)[yi]]))
    return dict(com=com, mean_var=mean_var, intensity=intensity, event_area=np.round(s[:, 0], 2), com_near_integer=near)
