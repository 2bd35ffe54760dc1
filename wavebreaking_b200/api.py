"""Drop-in API of the detection path (same names, arguments and error behaviour as the reference).

Mirrors ``wavebreaking/__init__.py:19-34``: ``calculate_smoothed_field``, ``calculate_momentum_flux``,
``calculate_contours``, ``calculate_streamers``, ``calculate_overturnings``, ``calculate_cutoffs``,
``to_xarray`` and ``track_events`` (alias ``event_tracking``), plus the decorator "runtime" of
``wavebreaking/utils/data_utils.py`` (argument type checks, dimension discovery with ``key=value``
overrides) and ``utils/index_utils.py`` (``combine_shared``).  Inputs are ``xarray.DataArray`` (or the
:class:`wavebreaking_b200.compat.Field` stand-in when xarray is not installed); outputs are
``geopandas.GeoDataFrame`` / ``xarray.DataArray`` when those packages are importable and pandas
DataFrames with lightweight geometry objects / ``Field`` otherwise.  All arithmetic runs in libwbk.
"""

import functools
import logging

import numpy as np
import pandas as pd
import torch

from . import _lib, compat, detect, geometry, spatial, tracking

logger = logging.getLogger(__name__)

__all__ = [
    "calculate_smoothed_field", "calculate_momentum_flux", "calculate_contours", "calculate_streamers",
    "calculate_overturnings", "calculate_cutoffs", "to_xarray", "track_events", "event_tracking", "combine_shared",
    "check_argument_types", "get_dimension_attributes", "check_empty_dataframes", "flag_frequency",
]

_FIELD = "field"
_FRAME = "frame"
_PANDAS = "pandas"


# ------------------------------------------------------------------------------------------- data_utils.py
def _type_ok(value, kind):
    if kind == _FIELD:
        return compat.is_field(value)
    if kind in (_FRAME, _PANDAS):
        return compat.is_frame(value)
    return isinstance(value, kind)


def _type_name(kind):
    if kind == _FIELD:
        return compat.field_type_name()
    if kind == _FRAME:
        return compat.frame_type_name()
    if kind == _PANDAS:
        return "pandas.core.frame.DataFrame"
    return str(kind)[8:-2]


def check_argument_types(arguments, types):
    """decorator to check the type of function arguments (utils/data_utils.py:28-50)"""

    def decorator(func):
        @functools.wraps(func)
        def wrapper(*args, **kwargs):
            for (arg_index, arg_name), arg_type in zip(enumerate(arguments), types):
                value = kwargs[arg_name] if arg_name in kwargs else args[arg_index]
                if not _type_ok(value, arg_type):
                    raise TypeError(arg_name + " has to be a " + _type_name(arg_type) + "!")
            return func(*args, **kwargs)

        return wrapper

    return decorator


def check_empty_dataframes(func):
    """decorator to check if there is an empty DataFrame (utils/data_utils.py:53-73)"""

    @functools.wraps(func)
    def wrapper(*args, **kwargs):
        for item in args:
            if compat.is_frame(item) and item.empty:
                raise ValueError("geopandas.GeoDataFrame is empty!")
        for key, item in kwargs.items():
            if compat.is_frame(item) and item.empty:
                raise ValueError(key + " geopandas.GeoDataFrame is empty!")
        return func(*args, **kwargs)

    return wrapper


def get_time_name(data):
    """utils/data_utils.py:76-93"""
    for dim in data.dims:
        values, attrs, encoding = compat.coord_info(data, dim)
        if (
            ("units" in attrs and "since" in attrs["units"])
            or ("units" in encoding and "since" in encoding["units"])
            or (values.dtype == np.dtype("datetime64[ns]"))
            or (dim in ["time"])
        ):
            return dim
    raise ValueError("'time' dimension (dtype='datetime64[ns]') not found."
                     " Add time dimension with xarray.DataArray.expand_dims('time').")


def get_lon_name(data):
    """utils/data_utils.py:96-109"""
    for dim in data.dims:
        _, attrs, _ = compat.coord_info(data, dim)
        if ("units" in attrs and attrs["units"] in ["degree_east", "degrees_east"]) or dim in ["lon", "longitude", "x"]:
            return dim
    raise ValueError("'longitude' dimension (units='degrees_east') not found.")


def get_lat_name(data):
    """utils/data_utils.py:112-126"""
    for dim in data.dims:
        _, attrs, _ = compat.coord_info(data, dim)
        if ("units" in attrs and attrs["units"] in ["degree_north", "degrees_north"]) or dim in ["lat", "latitude", "y"]:
            return dim
    raise ValueError("latitude' dimension (units='degrees_north') not found.")


def get_spatial_resolution(data, dim):
    """utils/data_utils.py:129-144"""
    values = compat.coord_info(data, dim)[0]
    delta = abs(np.unique((values[1:] - values[:-1])))
    if len(delta) > 1:
        raise ValueError("No regular grid found for dimension {}.".format(dim))
    elif delta[0] == 0:
        raise ValueError("Two equivalent coordinates found for dimension {}.".format(dim))
    return delta[0]


def get_dimension_attributes(arg_name):
    """decorator to get the dimension, size and resolution of the input data (utils/data_utils.py:147-193)"""

    def decorator(func):
        @functools.wraps(func)
        def wrapper(*args, **kwargs):
            data = kwargs[arg_name] if arg_name in kwargs else args[0]
            names = ["time_name", "lon_name", "lat_name"]
            sizes = ["ntime", "nlon", "nlat"]
            resolutions = ["dlon", "dlat"]
            get_dims = [get_time_name, get_lon_name, get_lat_name]
            for name, get_dim in zip(names, get_dims):
                if name not in kwargs:
                    kwargs[name] = get_dim(data)
            for size, name in zip(sizes, names):
                if size not in kwargs:
                    kwargs[size] = len(data[kwargs[name]])
            for res, name in zip(resolutions, names[1:]):
                if res not in kwargs:
                    kwargs[res] = get_spatial_resolution(data, kwargs[name])
            if len(data.dims) > 3:
                err_dims = [dim for dim in data.dims if dim not in [kwargs[name] for name in names]]
                raise ValueError("Unexpected dimension(s): {}. Select dimensions first.".format(err_dims))
            return func(*args, **kwargs)

        return wrapper

    return decorator


def combine_shared(lst):
    """utils/index_utils.py:187-214 (connected components of index lists, first-appearance order)."""
    return tracking.combine_shared(lst)


# ------------------------------------------------------------------------------------------- helpers
_CANON_CACHE = []  # [(key, _Canon)], most recent last; the device copy of `data` is reused by the three index calls


def _canon(data, kwargs, need_values=True, orient=True):
    """Cached :class:`_Canon`: ``calculate_streamers / overturnings / cutoffs / contours`` of one analysis are called
    on the same DataArray, so its upload (and re-orientation) happens once.  The key holds the identity of the
    value buffer, its shape / strides and the dimension names; the cache keeps the two most recent fields."""
    lazy = getattr(data, "_lazy", None)
    if (lazy is not None and lazy.device is not None and need_values and getattr(data, "_values", None) is None
            and lazy.device_meta == (tuple(data.dims), bool(orient))):
        c = _Canon(data, kwargs, need_values=False, orient=orient)
        c.tensor = lazy.device  # result of an earlier API call that is still on the device: no upload
        return c
    values = data.values
    iface = getattr(values, "__array_interface__", None)
    key = None
    if iface is not None and need_values:
        key = (iface["data"][0], values.shape, values.strides, str(values.dtype), tuple(data.dims), bool(orient),
               tuple(sorted((k, str(v)) for k, v in kwargs.items() if k.endswith("_name"))))
        for k, c in _CANON_CACHE:
            if k == key and c.tensor is not None and c.owner() is values:
                return c
    c = _Canon(data, kwargs, need_values, orient)
    if key is not None:
        import weakref

        try:
            c.owner = weakref.ref(values)
        except TypeError:
            c.owner = lambda: None
        _CANON_CACHE.append((key, c))
        del _CANON_CACHE[:-2]
    return c


class _Canon:
    """``data`` as a device tensor [time, lat, lon] with ascending lat / lon (data_utils.py:196-213)."""

    def __init__(self, data, kwargs, need_values=True, orient=True):
        self.time_name, self.lon_name, self.lat_name = kwargs["time_name"], kwargs["lon_name"], kwargs["lat_name"]
        self.time = compat.coord_info(data, self.time_name)[0]
        lon = compat.coord_info(data, self.lon_name)[0]
        lat = compat.coord_info(data, self.lat_name)[0]
        self.flip_lat = bool(np.average(np.diff(lat)) < 0) if (orient and len(lat) > 1) else False
        self.flip_lon = bool(np.average(np.diff(lon)) < 0) if (orient and len(lon) > 1) else False
        self.lat = lat[::-1].copy() if self.flip_lat else lat
        self.lon = lon[::-1].copy() if self.flip_lon else lon
        self.nlon, self.nlat, self.ntime = kwargs["nlon"], kwargs["nlat"], kwargs["ntime"]
        self.dlon, self.dlat = kwargs["dlon"], kwargs["dlat"]
        self.order = [data.dims.index(self.time_name), data.dims.index(self.lat_name), data.dims.index(self.lon_name)]
        self.dims = tuple(data.dims)
        self.tensor = None
        if need_values:
            values = np.asarray(data.values)
            if values.dtype not in (np.float32, np.float64):
                values = values.astype(np.float64)
            values = np.ascontiguousarray(np.transpose(values, self.order))
            t = spatial.to_device(values)
            self.tensor = spatial.flip(t, self.flip_lat, self.flip_lon)

    def to_input_layout(self, arr):
        """[time, lat, lon] (ascending) numpy array -> the input's dim order and orientation."""
        if self.flip_lat:
            arr = arr[:, ::-1, :]
        if self.flip_lon:
            arr = arr[:, :, ::-1]
        inv = np.argsort(self.order)
        return np.transpose(arr, inv)


def _to_host(dev):
    """Device tensor -> numpy array backed by page-locked memory (one asynchronous copy at link speed; a plain
    ``.cpu()`` lands in freshly allocated pageable memory at a fraction of it).  torch recycles the pinned block
    when the array is released."""
    lib = _lib.get()
    if not lib.is_cuda:
        return dev.cpu().numpy()
    host = torch.empty(dev.shape, dtype=dev.dtype, pin_memory=True)
    host.copy_(dev, non_blocking=True)
    torch.cuda.current_stream(lib.device).synchronize()
    return host.numpy()


def _as_levels(contour_levels):
    try:
        iter(contour_levels)
    except Exception:
        contour_levels = [contour_levels]
    return list(contour_levels)


# ------------------------------------------------------------------------------------------- spatial.py
@check_argument_types(["u", "v"], [_FIELD, _FIELD])
@get_dimension_attributes("u")
def calculate_momentum_flux(u, v, *args, **kwargs):
    """Momentum flux u'v' from the deviations of both wind components from the zonal mean
    (processing/spatial.py:27-57)."""
    cu = _canon(u, kwargs)
    vk = dict(kwargs)
    cv = _canon(v, vk)
    # numpy sums pairwise along a contiguous axis and sequentially along a strided one: follow the user's layout
    lon_last = tuple(u.dims)[-1] == kwargs["lon_name"] and tuple(v.dims)[-1] == kwargs["lon_name"]
    out = spatial.momentum_flux(cu.tensor, cv.tensor, lon_contiguous=lon_last).cpu().numpy()
    return compat.like(u, cu.to_input_layout(out), u.dims, name="mflux")


@check_argument_types(["data"], [_FIELD])
@get_dimension_attributes("data")
def calculate_smoothed_field(data, passes, weights=np.array([[0, 1, 0], [1, 2, 1], [0, 1, 0]]), mode="wrap", *args,
                             **kwargs):
    """``passes`` x 5-point smoothing (scipy.ndimage.convolve semantics), latitude border rows NaN
    (processing/spatial.py:60-128).  The result has dims (time, lat, lon) like the reference's."""
    c = _canon(data, kwargs, orient=False)  # the reference convolves the (lat, lon) slices as they are stored
    out = spatial.smooth(c.tensor, passes, np.asarray(weights), mode)
    dims = (c.time_name, c.lat_name, c.lon_name)
    attrs = dict(getattr(data, "attrs", {}) or {})
    attrs["smooth_passes"] = passes
    # the smoothed field stays on the device until its values are read; the index functions take the device tensor
    # (re-oriented to ascending coordinates if the input is stored descending) without another upload
    lat = compat.coord_info(data, c.lat_name)[0]
    lon = compat.coord_info(data, c.lon_name)[0]
    fl = bool(len(lat) > 1 and np.average(np.diff(lat)) < 0)
    fo = bool(len(lon) > 1 and np.average(np.diff(lon)) < 0)
    canonical = out if not (fl or fo) else None  # (descending input: the next call re-orients its own copy)
    lazy = compat.LazyValues(tuple(out.shape), np.float64 if out.dtype == torch.float64 else np.float32,
                             lambda: _to_host(out), device=canonical, device_meta=(dims, True))
    return compat.like(data, lazy, dims, name="smooth_" + str(data.name), attrs=attrs)


# ------------------------------------------------------------------------------------------- contours
class _DeviceContours:
    """Device-resident contours of a frame returned by ``calculate_contours(original_coordinates=False)``."""

    def __init__(self, batches, canon, levels, periodic_add):
        self.batches = batches  # list of (t0, ContourSet)
        self.key = (tuple(canon.time.tolist()), canon.nlat, canon.nlon, tuple(levels), periodic_add)


# frame.attrs only carries a small integer token: pandas deep-copies attrs into every derived frame and serialises
# them (to_parquet), which must not duplicate or choke on device buffers.  The buffers live here, most recent last.
_DEVICE_CONTOURS = {}
_DEVICE_TOKEN = [0]


def _remember_device_contours(frame, dev):
    _DEVICE_TOKEN[0] += 1
    token = _DEVICE_TOKEN[0]
    _DEVICE_CONTOURS[token] = dev
    for old in sorted(_DEVICE_CONTOURS)[:-4]:
        del _DEVICE_CONTOURS[old]
    frame.attrs["_wbk_device_token"] = token


def _batch_size(nlat, nlon, nlevels):
    """Time steps per launch: fill the GPU (>= 2 jobs per SM) without excessive arena memory."""
    per_job = max(nlat * nlon, 1)
    return int(max(1, min(296 // max(nlevels, 1) + 1, (1 << 28) // per_job)))


def _contour_batches(c, levels, periodic_add):
    add = int(periodic_add / c.dlon)
    tb = _batch_size(c.nlat, c.nlon, len(levels))
    out = []
    for t0 in range(0, c.ntime, tb):
        cs = detect.contours(c.tensor[t0:t0 + tb], levels, add)
        out.append((t0, cs))
    return out


def _contour_frame(c, batches, levels, original_coordinates):
    """Frame of all contours (contour_index.py:149-194), built from the ragged host arrays of the batches: no
    per-contour numpy work except the float mean of the original-coordinate latitudes (numpy's own summation order)."""
    nlev = len(levels)
    xs, ys, lens, tsteps, lidx, closed, nx, sumy = [], [], [], [], [], [], [], []
    for t0, cs in batches:
        h = cs.host()
        xs.append(h["x"])
        ys.append(h["y"])
        lens.append(np.diff(h["pt_off"]))
        tsteps.append(t0 + h["job"] // nlev)
        lidx.append(h["job"] % nlev)
        closed.append(h["closed"])
        nx.append(h["nx"])
        sumy.append(h["sum_y"])
    cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dtype=dt)
    x, y, lens = cat(xs, np.int64), cat(ys, np.int64), cat(lens, np.int64)
    tsteps, lidx = cat(tsteps, np.int64), cat(lidx, np.int64)
    n = len(lens)
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    rows = dict(date=np.asarray(c.time)[tsteps], level=np.asarray(levels, dtype=object)[lidx] if n else [],
                closed=cat(closed, bool))
    if not original_coordinates:
        rows["exp_lon"] = cat(nx, np.int64) * c.dlon
        # mean of the integer rows: the float64 sum of ints < 2^53 is exact in any order
        rows["mean_lat"] = np.round(cat(sumy, np.int64) / np.maximum(lens, 1), 2)
        geoms = compat.linestrings_from_ragged(np.c_[x, y], off)
    else:
        # contour_index.py:179-191: map to coordinates, drop repeated points (keep first) within every contour
        cid = np.repeat(np.arange(n, dtype=np.int64), lens)
        xm = x % c.nlon
        key = (cid * c.nlon + xm) * c.nlat + y
        _, first = np.unique(key, return_index=True)
        keep = np.zeros(len(key), dtype=bool)
        keep[first] = True
        lon_v, lat_v = np.asarray(c.lon, dtype=np.float64)[xm[keep]], np.asarray(c.lat, dtype=np.float64)[y[keep]]
        klens = np.bincount(cid[keep], minlength=n).astype(np.int64)
        koff = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(klens, out=koff[1:])
        ncol = np.bincount(np.unique(cid * c.nlon + xm) // c.nlon, minlength=n)
        rows["exp_lon"] = ncol * c.dlon
        rows["mean_lat"] = np.array([np.round(lat_v[a:b].mean(), 2) for a, b in zip(koff[:-1], koff[1:])]) if n else []
        geoms = compat.linestrings_from_ragged(np.c_[lon_v, lat_v], koff)
    return compat.make_frame(rows, geoms)


@check_argument_types(["data"], [_FIELD])
@get_dimension_attributes("data")
def calculate_contours(data, contour_levels, periodic_add=120, original_coordinates=True, *args, **kwargs):
    """Contour lines for a set of levels on the periodically extended grid
    (indices/contour_index.py:45-194; time / level loops of utils/index_utils.py:217-258 batched)."""
    c = _canon(data, kwargs)
    levels = _as_levels(contour_levels)
    batches = _contour_batches(c, levels, periodic_add)
    frame = _contour_frame(c, batches, levels, original_coordinates)
    if not original_coordinates:
        _remember_device_contours(frame, _DeviceContours(batches, c, levels, periodic_add))
    return frame


def _contours_from_frame(contours, c, levels, periodic_add):
    """Contour sets for the index stage: the device-resident ones of ``calculate_contours`` when the frame is the
    one it returned, else the user's frame uploaded as ONE packed contour set.  Like the reference
    (streamer_index.py:104-108, contour_index.py:221-231) every contour of the frame takes part, whatever its level;
    levels missing from ``contour_levels`` are appended to the level list."""
    token = contours.attrs.get("_wbk_device_token") if hasattr(contours, "attrs") else None
    dev = _DEVICE_CONTOURS.get(token)
    key = (tuple(c.time.tolist()), c.nlat, c.nlon, tuple(levels), periodic_add)
    if dev is not None and dev.key == key and sum(cs.ncontours for _, cs in dev.batches) == len(contours):
        return dev.batches, levels
    lib = _lib.get()
    levels = list(levels)
    for lv in pd.unique(contours.level):
        if float(lv) not in [float(v) for v in levels]:
            levels.append(lv)
    level_index = {float(l): i for i, l in enumerate(levels)}
    nlev = len(levels)
    dates = contours.date.values
    if np.issubdtype(c.time.dtype, np.datetime64):
        dates = dates.astype(c.time.dtype)
    tpos = pd.Index(c.time).get_indexer(pd.Index(dates))
    if (tpos < 0).any():
        raise KeyError(contours.date.values[np.argmax(tpos < 0)])
    lpos = np.array([level_index[float(v)] for v in contours.level.values], dtype=np.int64)
    coords = [compat.line_coords(g) for g in contours.geometry]
    lens = np.array([len(a) for a in coords], dtype=np.int64)
    allxy = np.concatenate(coords).astype(np.int64) if coords else np.zeros((0, 2), dtype=np.int64)
    jobs = tpos.astype(np.int64) * nlev + lpos
    order = np.argsort(jobs, kind="stable")
    njobs = c.ntime * nlev
    job_arr = jobs[order]
    job_off = np.searchsorted(job_arr, np.arange(njobs + 1)).astype(np.int32)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    from .tracking import _ranges

    sel = _ranges(off[:-1][order], lens[order])
    px, py = allxy[sel, 0], allxy[sel, 1]
    cid = np.repeat(np.arange(len(lens), dtype=np.int64), lens[order])
    pt_off = np.zeros(len(lens) + 1, dtype=np.int32)
    pt_off[1:] = np.cumsum(lens[order])
    nxc = np.bincount(np.unique(cid * 65536 + px) // 65536, minlength=len(lens)) if len(lens) else np.zeros(0, dtype=np.int64)
    sumy = np.bincount(cid, weights=py, minlength=len(lens)).astype(np.int64) if len(lens) else np.zeros(0, dtype=np.int64)
    meta = np.c_[contours.closed.values.astype(np.int64)[order], nxc, sumy, job_arr].astype(np.int32)
    allp = (px | (py << 16)).astype(np.uint32)
    dev_t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(lib.device)
    cs = detect.ContourSet(
        njobs=njobs, nlevels=nlev, nlat=c.nlat, nlon=c.nlon, add=int(periodic_add / c.dlon),
        levels=np.asarray(levels, dtype=np.float64), job_off=dev_t(job_off), pt_off=dev_t(pt_off),
        meta=dev_t(meta.reshape(-1, 4)), pts=dev_t(allp.view(np.int32)), status=np.zeros(njobs, dtype=np.int32),
        max_nx=int(nxc.max()) if len(nxc) else 0, h_ncontours=np.diff(job_off), h_npoints=None)
    return [(0, cs)], levels


def decorator_contour_calculation(func):
    """wrap the contour calculation around the index functions (indices/contour_index.py:197-249)"""

    @functools.wraps(func)
    def wrapper(data, contour_levels, periodic_add=120, *args, **kwargs):
        if "contours" not in kwargs:
            kwargs["contours"] = calculate_contours(data, contour_levels, periodic_add, original_coordinates=False)
        else:
            if not compat.is_frame(kwargs["contours"]):
                raise TypeError("contours has to be a geopandas.GeoDataFrame!")
            if kwargs["contours"].empty:
                raise ValueError("contours geopandas.GeoDataFrame is empty!")
            levels = _as_levels(contour_levels)
            check_levels = [i for i in levels if i not in set(kwargs["contours"].level)]
            if len(check_levels) > 0:
                logger.warning("\n The contour levels {} are not present in 'contours'".format(check_levels))
            coords = compat.line_coords(kwargs["contours"].iloc[0].geometry)
            check_int = (coords.astype("int") == coords).all()
            check_zero = (coords[:, 0] >= 0).all()
            if not (check_int and check_zero):
                raise ValueError("Original coordinates not supported for the index calculation. "
                                 "Use original_coordinates=False in the contour calculation.")
        return func(data, contour_levels, periodic_add=periodic_add, *args, **kwargs)

    return wrapper


# ------------------------------------------------------------------------------------------- indices
_EVENT_COLUMNS = ["date", "level", "com", "mean_var", "intensity", "event_area"]


def _event_rings(cs, tab):
    """Ragged index-space rings of the events of one table (vectorised): (xy int64 [N, 2], off [n + 1])."""
    from .tracking import _ranges

    n = len(tab)
    if tab.kind == "overturnings":
        x0, y0, x1, y1 = (tab.box[:, k].astype(np.int64) for k in range(4))
        xy = np.stack([np.c_[x1, y0], np.c_[x1, y1], np.c_[x0, y1], np.c_[x0, y0]], axis=1).reshape(-1, 2)
        return xy, np.arange(n + 1, dtype=np.int64) * 4
    h = cs.host()
    start = h["pt_off"][tab.contour].astype(np.int64) + tab.ind1.astype(np.int64)
    lens = (tab.ind2.astype(np.int64) - tab.ind1.astype(np.int64) + 1) if n else np.zeros(0, dtype=np.int64)
    idx = _ranges(start, lens)
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    return np.c_[h["x"][idx], h["y"][idx]], off


def _fold_and_split(xy, off, split, nlon, pieces=None, first=0):
    """``transform_polygons`` (utils/index_utils.py:129-184) on ragged rings: fold with ``x % nlon``; the few events
    that straddle the last meridian (split == 1) are cut into their pieces (taken from the device clipper when
    ``pieces`` is given, else clipped on the host).  Returns (xy, ring_off, poly_off)."""
    n = len(off) - 1
    straddle = np.nonzero(np.asarray(split) == 1)[0]
    if len(straddle) == 0:
        out = xy.copy()
        out[:, 0] %= nlon
        return out, off, np.arange(n + 1, dtype=np.int64)
    if pieces is not None:
        return geometry.interleave_pieces(xy, off, split, pieces, first, nlon)
    parts, ring_len, poly_nr = [], [], np.ones(n, dtype=np.int64)
    prev = 0
    for e in straddle:
        if off[e] > off[prev]:
            seg = xy[off[prev]:off[e]].copy()
            seg[:, 0] %= nlon
            parts.append(seg)
            ring_len.extend(np.diff(off[prev:e + 1]).tolist())
        pieces = geometry.transform_ring(xy[off[e]:off[e + 1]], nlon)
        poly_nr[e] = len(pieces)
        for pc in pieces:
            parts.append(np.asarray(pc, dtype=np.int64).reshape(-1, 2))
            ring_len.append(len(pc))
        prev = e + 1
    if off[n] > off[prev]:
        seg = xy[off[prev]:off[n]].copy()
        seg[:, 0] %= nlon
        parts.append(seg)
        ring_len.extend(np.diff(off[prev:n + 1]).tolist())
    allxy = np.concatenate(parts) if parts else np.zeros((0, 2), dtype=np.int64)
    return allxy, np.r_[0, np.cumsum(ring_len)].astype(np.int64), np.r_[0, np.cumsum(poly_nr)].astype(np.int64)


def _run_index(kind, data, contour_levels, contours, intensity, periodic_add, kwargs, **params):
    c = _canon(data, kwargs)
    levels = _as_levels(contour_levels)
    inten = None
    if intensity is not None:
        if not compat.is_field(intensity):
            raise TypeError("intensity has to be a " + compat.field_type_name() + "!")
        inten = _canon(intensity, dict(kwargs)).tensor
    batches, levels = _contours_from_frame(contours, c, levels, periodic_add)
    # exp_lon.max() is global over all dates and levels (streamer_index.py:106)
    gmax = max([cs.max_nx for _, cs in batches] + [0])
    if len(contours):
        gmax = max(gmax, int(round(float(np.max(contours.exp_lon)) / c.dlon)))
    coords = detect.coord_tables(c.lat, c.lon, c.dlon, c.dlat)
    cols = {k: [] for k in _EVENT_COLUMNS}
    orient, xy_parts, ring_offs, poly_offs = [], [], [], []
    nlev = len(levels)
    lon_v, lat_v = np.asarray(c.lon, dtype=np.float64), np.asarray(c.lat, dtype=np.float64)
    for t0, cs in batches:
        nt = cs.njobs // nlev
        field = c.tensor[t0:t0 + nt]
        tables, _, pieces = detect.run_indices(cs, field, coords, c.dlon, c.dlat,
                                               intensity=None if inten is None else inten[t0:t0 + nt], which=(kind,),
                                               gmax_nx=gmax, want_flags=False, want_pieces=True, **params)
        tab = tables[kind]
        if len(tab) == 0:
            continue
        props = detect.finish_properties(tab, c.lon, c.lat, c.nlon)
        t, l = np.divmod(tab.job.astype(np.int64), nlev)
        cols["date"].append(np.asarray(c.time)[t0 + t])
        cols["level"].append(np.asarray(levels, dtype=object)[l])
        for k in ("mean_var", "intensity", "event_area"):
            cols[k].append(np.asarray(props[k]))
        cols["com"].extend(props["com"])
        orient.append(np.where(tab.orientation != 0, "anticyclonic", "cyclonic"))
        xy, off = _event_rings(cs, tab)
        pxy, roff, poff = _fold_and_split(xy, off, tab.split, c.nlon, pieces)
        xy_parts.append(np.c_[lon_v[pxy[:, 0]], lat_v[pxy[:, 1]]])
        ring_offs.append(roff)
        poly_offs.append(poff)
    if not xy_parts:
        return compat.empty_frame()
    # one ragged geometry column for all batches
    vo = ro = 0
    r_all, p_all = [np.zeros(1, dtype=np.int64)], [np.zeros(1, dtype=np.int64)]
    for xyp, roff, poff in zip(xy_parts, ring_offs, poly_offs):
        r_all.append(roff[1:] + vo)
        p_all.append(poff[1:] + ro)
        vo += len(xyp)
        ro += len(roff) - 1
    geoms = compat.polygons_from_ragged(np.concatenate(xy_parts), np.concatenate(r_all), np.concatenate(p_all))
    frame_cols = {k: (np.concatenate(v) if k != "com" else v) for k, v in cols.items()}
    if kind == "overturnings":
        frame_cols["orientation"] = np.concatenate(orient)
    return compat.make_frame(frame_cols, geoms)


@check_argument_types(["data"], [_FIELD])
@get_dimension_attributes("data")
@decorator_contour_calculation
def calculate_streamers(data, contour_level, contours=None, geo_dis=800, cont_dis=1500, intensity=None,
                        periodic_add=120, *args, **kwargs):
    """Streamer index of Wernli and Sprenger (2007) (indices/streamer_index.py:44-289)."""
    if contours is None:
        contours = kwargs["contours"]
    return _run_index("streamers", data, contour_level, contours, intensity, periodic_add, kwargs,
                      geo_dis=geo_dis, cont_dis=cont_dis)


@check_argument_types(["data"], [_FIELD])
@get_dimension_attributes("data")
@decorator_contour_calculation
def calculate_overturnings(data, contour_levels, contours=None, range_group=5, min_exp=5, intensity=None,
                           periodic_add=120, *args, **kwargs):
    """Overturning index of Barnes and Hartmann (2012) (indices/overturning_index.py:40-232)."""
    if contours is None:
        contours = kwargs["contours"]
    return _run_index("overturnings", data, contour_levels, contours, intensity, periodic_add, kwargs,
                      range_group=range_group, ot_min_exp=min_exp)


@check_argument_types(["data"], [_FIELD])
@get_dimension_attributes("data")
@decorator_contour_calculation
def calculate_cutoffs(data, contour_level, contours=None, min_exp=5, intensity=None, periodic_add=120, *args,
                      **kwargs):
    """Cutoff index: closed contours shorter than the full longitudinal extent (indices/cutoff_index.py:33-104)."""
    if contours is None:
        contours = kwargs["contours"]
    return _run_index("cutoffs", data, contour_level, contours, intensity, periodic_add, kwargs, co_min_exp=min_exp)


# ------------------------------------------------------------------------------------------- events.py
@check_argument_types(["data", "events"], [_FIELD, _FRAME])
@check_empty_dataframes
@get_dimension_attributes("data")
def to_xarray(data, events, flag="ones", name="flag", *args, **kwargs):
    """Flag the grid cells covered by events (processing/events.py:37-110)."""
    c = _Canon(data, kwargs, need_values=False)
    # the buffer of events.py:75-78 is measured in degrees: ValueError before any device work for spacings the
    # rasteriser cannot measure it in exactly
    detect.grid_ratio(c.dlon, c.dlat)
    if flag != "ones":
        try:
            set_val = np.asarray(events[flag].values, dtype=np.float64)
        except KeyError:
            raise KeyError("{} is not a column of the events geopandas.GeoDataFrame.".format(flag))
    # ragged extraction of all rings, then ONE vectorised snap to grid indices
    dates = np.asarray(events["date"].values)
    if np.issubdtype(c.time.dtype, np.datetime64):
        dates = dates.astype(c.time.dtype)
    tpos = pd.Index(c.time).get_indexer(pd.Index(dates))
    if (tpos < 0).any():
        raise KeyError(events["date"].values[int(np.argmax(tpos < 0))])
    per_event = [compat.geometry_rings(g) for g in events["geometry"]]
    nring = np.array([len(r) for r in per_event], dtype=np.int64)
    flat = [np.asarray(r, dtype=np.float64).reshape(-1, 2) for rr in per_event for r in rr]
    rings, ring_t, ring_v = [], [], []
    if flat:
        lens = np.array([len(r) for r in flat], dtype=np.int64)
        allxy = np.concatenate(flat)
        idx = np.c_[(allxy[:, 0] - c.lon[0]) / c.dlon, (allxy[:, 1] - c.lat[0]) / c.dlat]
        snapped = np.rint(idx)
        if not np.allclose(idx, snapped, atol=1e-6):
            raise ValueError("to_xarray: event vertices must lie on grid points of `data`")
        snapped = snapped.astype(np.int32)
        cuts = np.cumsum(lens)[:-1]
        rings = np.split(snapped, cuts)
        ev_of_ring = np.repeat(np.arange(len(per_event)), nring)
        ring_t = tpos[ev_of_ring].tolist()
        ring_v = (np.ones(len(flat)) if flag == "ones" else set_val[ev_of_ring]).tolist()
    lib = _lib.get()
    if flag == "ones":
        dev = detect.rasterize_rings(rings, ring_t, c.nlat, c.nlon, c.ntime, spacing=(c.dlon, c.dlat))
        out_dtype = np.dtype(np.int8)
    else:
        grid = torch.zeros((c.ntime, c.nlat, c.nlon), dtype=torch.float64, device=lib.device)
        dev = detect.rasterize_rings(rings, ring_t, c.nlat, c.nlon, c.ntime, spacing=(c.dlon, c.dlat),
                                     values=(grid, ring_v))
        out_dtype = np.dtype(data.dtype)
    shape = tuple(len(data[d]) for d in data.dims)
    # the grid stays on the device until its values are read (a DataArray result is downloaded at once).  The int8
    # grid is also offered as `device` (flag_frequency counts it there); without device_meta no index function takes it
    lazy = compat.LazyValues(shape, out_dtype,
                             lambda: np.ascontiguousarray(c.to_input_layout(_to_host(dev)).astype(out_dtype, copy=False)),
                             device=dev if flag == "ones" else None)
    res = compat.like(data, lazy, data.dims, name=name, attrs=dict(getattr(data, "attrs", {}) or {}))
    res.attrs["long_name"] = "flag wave breaking"
    return res


@check_argument_types(["flag_data"], [_FIELD])
@get_dimension_attributes("flag_data")
def flag_frequency(flag_data, months=None, *args, **kwargs):
    """Flag frequency: the percentage of time steps in which each grid cell is flagged.

    ``flag_data``: the int8 output of ``to_xarray(..., flag="ones")`` (any other dtype raises TypeError); a result of
    ``to_xarray`` that still lives on the device is counted there, without a download.  ``months``: count only the
    time steps whose month (1-12, from the time coordinate, which then has to be datetime64) is in this list.
    Returns a (lat, lon) array in ``flag_data``'s dimension order and orientation, float64 percent (NaN when no time
    step is selected).  No smoothing is applied (``calculate_smoothed_field`` can be called on the result).

    This is the frequency the reference's ``plot_clim`` draws, as this project defines it: 100 * (number of selected
    steps with a nonzero flag) / (number of selected steps).  The reference's own formula could not be compared here
    (it is not installed), so small differences in its normalisation are possible.
    """
    if np.dtype(flag_data.dtype) != np.int8:
        raise TypeError("flag_data has to be the int8 output of to_xarray(..., flag='ones'), got dtype {}".format(
            np.dtype(flag_data.dtype)))
    c = _Canon(flag_data, kwargs, need_values=False)
    if months is None:
        group = np.zeros(c.ntime, dtype=np.int32)
    else:
        if not np.issubdtype(c.time.dtype, np.datetime64):
            raise ValueError("months needs a datetime64 time coordinate, got dtype {}".format(c.time.dtype))
        month = c.time.astype("datetime64[M]").astype(np.int64) % 12 + 1
        group = np.where(np.isin(month, np.asarray(months, dtype=np.int64).ravel()), 0, -1).astype(np.int32)
    lib = _lib.get()
    lazy = getattr(flag_data, "_lazy", None)
    if lazy is not None and lazy.device is not None and getattr(flag_data, "_values", None) is None:
        grid = lazy.device  # int8 [time, lat, lon], ascending coordinates: counted where it is
    else:
        host = np.transpose(np.asarray(flag_data.values), c.order)
        host = host[:, ::-1 if c.flip_lat else 1, ::-1 if c.flip_lon else 1]
        grid = torch.from_numpy(np.ascontiguousarray(host)).to(lib.device)
    counts = torch.zeros((c.nlat, c.nlon), dtype=torch.int32, device=lib.device)
    dev_group = torch.from_numpy(group).to(lib.device)
    lib.call("wbk_flag_counts", _lib.ptr(grid), 1, c.ntime, c.nlat * c.nlon, _lib.ptr(dev_group), 1, _lib.ptr(counts),
             lib.stream())
    from . import pipeline

    freq = pipeline._percent(_to_host(counts).view(np.uint32)[None], [int((group == 0).sum())])
    freq = c.to_input_layout(freq)  # [1, lat, lon] -> the input's dimension order, with a time axis of length 1
    dims = tuple(d for d in flag_data.dims if d != c.time_name)
    values = np.ascontiguousarray(freq.reshape([freq.shape[i] for i, d in enumerate(flag_data.dims) if d != c.time_name]))
    return compat.like(flag_data, values, dims, name="flag_frequency",
                       attrs={"long_name": "flag frequency", "units": "%"})


@check_argument_types(["events"], [_PANDAS])
@check_empty_dataframes
def track_events(events, time_range=None, method="by_overlap", buffer=0, overlap=0, distance=1000):
    """Temporal tracking of events (processing/events.py:113-241)."""
    return tracking.track_events(events, time_range, method, buffer, overlap, distance)


event_tracking = track_events
