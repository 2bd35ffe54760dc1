"""Stand-ins for xarray / geopandas / shapely objects when those packages are not installed.

The drop-in API (:mod:`wavebreaking_b200.api`) takes ``xarray.DataArray`` and returns
``geopandas.GeoDataFrame`` / ``xarray.DataArray`` whenever those packages can be imported.  The build
and test image of this repository has neither (no network), so the same API also accepts and returns
the minimal containers below; they carry exactly what the detection path needs (values, dimension names,
coordinates / coordinate rings) and convert to the real types on demand.
"""

import numpy as np

try:  # pragma: no cover - not available in the build image
    import xarray as _xr
except Exception:  # noqa: BLE001
    _xr = None
try:  # pragma: no cover
    import geopandas as _gpd
    import shapely as _shapely
except Exception:  # noqa: BLE001
    _gpd = None
    _shapely = None


def have_xarray():
    return _xr is not None


def have_geopandas():
    return _gpd is not None


class _Coord:
    """One coordinate axis (values + attrs), the part of xarray's IndexVariable the path reads."""

    def __init__(self, values, attrs=None, encoding=None):
        self.values = np.asarray(values)
        self.data = self.values
        self.attrs = dict(attrs or {})
        self.encoding = dict(encoding or {})

    @property
    def dtype(self):
        return self.values.dtype

    def __len__(self):
        return len(self.values)

    def __iter__(self):
        return iter(self.values)

    def __getitem__(self, i):
        return self.values[i]


class LazyValues:
    """Values that still live on the device: ``load()`` brings them to the host (once) as a numpy array in the
    Field's dimension order.  ``device`` is the canonical device tensor [time, lat, lon] (ascending lat / lon) that
    the next API call can use without any upload; the index functions take it only when ``device_meta`` matches
    (``to_xarray``'s int8 grid has none and is read by ``flag_frequency`` alone)."""

    def __init__(self, shape, dtype, load, device=None, device_meta=None):
        self.shape, self.dtype, self._load = tuple(shape), np.dtype(dtype), load
        self.device, self.device_meta = device, device_meta


class Field:
    """Minimal labelled array: ``values`` with named ``dims`` and 1-D ``coords`` (DataArray stand-in).

    ``values`` may be a :class:`LazyValues`: results of ``calculate_smoothed_field`` / ``to_xarray`` stay on the
    device until ``.values`` is read, and the index functions take the device tensor directly (a DataArray result
    cannot be lazy; with xarray installed the values are downloaded at once)."""

    def __init__(self, values, dims, coords, name=None, attrs=None):
        self._lazy = values if isinstance(values, LazyValues) else None
        self._values = None if self._lazy is not None else np.asarray(values)
        self.dims = tuple(dims)
        shape = self._lazy.shape if self._lazy is not None else self._values.shape
        if len(self.dims) != len(shape):
            raise ValueError("dims do not match the array rank")
        self.coords = {}
        for d in self.dims:
            c = coords[d]
            self.coords[d] = c if isinstance(c, _Coord) else _Coord(c)
            if len(self.coords[d]) != shape[self.dims.index(d)]:
                raise ValueError("coordinate {} does not match the array shape".format(d))
        for k, v in coords.items():  # scalar / extra coordinates (e.g. a level) are carried along
            if k not in self.coords:
                self.coords[k] = v if isinstance(v, _Coord) else _Coord(np.atleast_1d(v))
        self.name = name
        self.attrs = dict(attrs or {})

    @property
    def values(self):
        if self._values is None:
            self._values = np.asarray(self._lazy._load())
        return self._values

    def __getitem__(self, dim):
        return self.coords[dim]

    @property
    def shape(self):
        return self._lazy.shape if self._values is None else self._values.shape

    @property
    def dtype(self):
        return self._lazy.dtype if self._values is None else self._values.dtype

    def to_xarray(self):  # pragma: no cover
        if _xr is None:
            raise ImportError("xarray is not installed")
        return _xr.DataArray(self.values, dims=self.dims, coords={d: self.coords[d].values for d in self.dims},
                             name=self.name, attrs=self.attrs)


def is_field(obj):
    return isinstance(obj, Field) or (_xr is not None and isinstance(obj, _xr.DataArray))


def field_type_name():
    return "xarray.core.dataarray.DataArray"


def coord_info(data, dim):
    """(values, attrs, encoding) of a dimension coordinate of a Field or DataArray."""
    c = data[dim]
    values = np.asarray(c.values)
    return values, dict(getattr(c, "attrs", {}) or {}), dict(getattr(c, "encoding", {}) or {})


def like(data, values, dims, name=None, attrs=None):
    """A new labelled array of the same flavour as ``data`` (DataArray in, DataArray out).  ``values`` may be a
    :class:`LazyValues` (kept lazy in a Field, downloaded at once for a DataArray)."""
    coords = {d: np.asarray(data[d].values) for d in dims}
    if _xr is not None and isinstance(data, _xr.DataArray):  # pragma: no cover
        if isinstance(values, LazyValues):
            values = values._load()
        return _xr.DataArray(values, dims=dims, coords=coords, name=name, attrs=attrs or {})
    return Field(values, dims, coords, name=name, attrs=attrs)


# --------------------------------------------------------------------------------------------- geometries
class LineString:
    """Ordered vertices (n, 2); ``.coords.xy`` / ``np.asarray(.coords)`` like shapely."""

    geom_type = "LineString"

    def __init__(self, coords):
        self._xy = np.asarray(coords, dtype=np.float64).reshape(-1, 2)

    @classmethod
    def from_view(cls, xy):
        """No-copy construction from a float64 (n, 2) slice of a shared coordinate array."""
        obj = cls.__new__(cls)
        obj._xy = xy
        return obj

    class _Coords:
        def __init__(self, xy):
            self._xy = xy

        @property
        def xy(self):
            return self._xy[:, 0].copy(), self._xy[:, 1].copy()

        def __array__(self, dtype=None, copy=None):
            return self._xy if dtype is None else self._xy.astype(dtype)

        def __len__(self):
            return len(self._xy)

        def __iter__(self):
            return iter(map(tuple, self._xy))

    @property
    def coords(self):
        return LineString._Coords(self._xy)

    @property
    def bounds(self):
        return (self._xy[:, 0].min(), self._xy[:, 1].min(), self._xy[:, 0].max(), self._xy[:, 1].max())

    @property
    def is_empty(self):
        return len(self._xy) == 0

    @property
    def wkt(self):
        return "LINESTRING ({})".format(", ".join("{:g} {:g}".format(x, y) for x, y in self._xy))

    def __repr__(self):
        return "<LineString n={}>".format(len(self._xy))

    def to_shapely(self):  # pragma: no cover
        return _shapely.LineString(self._xy)


class Polygon:
    """A single exterior ring (closed on output like shapely: first vertex repeated)."""

    geom_type = "Polygon"

    def __init__(self, shell=None):
        xy = np.zeros((0, 2)) if shell is None else np.asarray(shell, dtype=np.float64).reshape(-1, 2)
        if len(xy) and not np.array_equal(xy[0], xy[-1]):
            xy = np.concatenate([xy, xy[:1]])
        self._xy = xy

    @classmethod
    def from_closed_view(cls, xy):
        """No-copy construction from a float64 (n + 1, 2) slice whose last vertex repeats the first."""
        obj = cls.__new__(cls)
        obj._xy = xy
        return obj

    @property
    def exterior(self):
        return LineString(self._xy)

    @property
    def is_empty(self):
        return len(self._xy) == 0

    @property
    def geoms(self):
        return [self]

    @property
    def bounds(self):
        return self.exterior.bounds

    @property
    def area(self):
        x, y = self._xy[:, 0], self._xy[:, 1]
        return 0.0 if len(x) < 4 else abs(float(np.sum(x[:-1] * y[1:] - x[1:] * y[:-1]))) / 2.0

    @property
    def wkt(self):
        if self.is_empty:
            return "POLYGON EMPTY"
        return "POLYGON (({}))".format(", ".join("{:g} {:g}".format(x, y) for x, y in self._xy))

    def __repr__(self):
        return "<Polygon n={}>".format(max(len(self._xy) - 1, 0))

    def rings(self):
        """Open rings (n, 2) of this geometry."""
        return [] if self.is_empty else [self._xy[:-1]]

    def to_shapely(self):  # pragma: no cover
        return _shapely.Polygon(self._xy) if len(self._xy) else _shapely.Polygon()


class MultiPolygon:
    geom_type = "MultiPolygon"

    def __init__(self, polygons):
        self.geoms = [p if isinstance(p, Polygon) else Polygon(p) for p in polygons]

    @classmethod
    def from_parts(cls, polygons):
        obj = cls.__new__(cls)
        obj.geoms = polygons
        return obj

    @property
    def is_empty(self):
        return len(self.geoms) == 0

    @property
    def area(self):
        return sum(p.area for p in self.geoms)

    @property
    def wkt(self):
        return "MULTIPOLYGON ({})".format(", ".join(p.wkt[len("POLYGON "):] for p in self.geoms))

    def __repr__(self):
        return "<MultiPolygon parts={}>".format(len(self.geoms))

    def rings(self):
        return [r for p in self.geoms for r in p.rings()]

    def to_shapely(self):  # pragma: no cover
        return _shapely.MultiPolygon([p.to_shapely() for p in self.geoms])


def geometry_rings(geom):
    """Open exterior rings (list of (n, 2) arrays) of a compat or shapely (Multi)Polygon."""
    if isinstance(geom, (Polygon, MultiPolygon)):
        return geom.rings()
    if geom is None or getattr(geom, "is_empty", False):
        return []
    parts = list(geom.geoms) if hasattr(geom, "geoms") else [geom]
    out = []
    for p in parts:
        xy = np.asarray(p.exterior.coords)
        out.append(xy[:-1] if len(xy) > 1 and np.array_equal(xy[0], xy[-1]) else xy)
    return out


def line_coords(geom):
    """(n, 2) vertex array of a compat or shapely LineString."""
    return np.asarray(geom.coords, dtype=np.float64).reshape(-1, 2)


def make_frame(columns, geometry):
    """GeoDataFrame when geopandas is importable, else a pandas DataFrame with a ``geometry`` column."""
    import pandas as pd

    if _gpd is not None:  # pragma: no cover
        geoms = [g.to_shapely() if hasattr(g, "to_shapely") else g for g in geometry]
        return _gpd.GeoDataFrame(pd.DataFrame(columns), geometry=geoms)
    df = pd.DataFrame(columns)
    df["geometry"] = pd.Series(list(geometry), index=df.index, dtype=object)
    return df


def empty_frame():
    import pandas as pd

    if _gpd is not None:  # pragma: no cover
        return _gpd.GeoDataFrame()
    return pd.DataFrame()


def is_frame(obj):
    import pandas as pd

    return isinstance(obj, pd.DataFrame)


def frame_type_name():
    return "geopandas.geodataframe.GeoDataFrame"


# --------------------------------------------------------------------------------------------- ragged construction
def linestrings_from_ragged(xy, off):
    """Geometry column of LineStrings from one (N, 2) float64 coordinate array and offsets [n + 1]: shapely's
    vectorised ``from_ragged_array`` when shapely is installed, no-copy views otherwise."""
    xy = np.ascontiguousarray(xy, dtype=np.float64)
    off = np.asarray(off, dtype=np.int64)
    if _shapely is not None:  # pragma: no cover
        return list(_shapely.from_ragged_array(_shapely.GeometryType.LINESTRING, xy, (off,)))
    return [LineString.from_view(xy[a:b]) for a, b in zip(off[:-1], off[1:])]


def polygons_from_ragged(xy, ring_off, poly_off):
    """Geometry column of (Multi)Polygons: polygon p = rings [poly_off[p], poly_off[p+1]) (0 rings: the empty
    ``Polygon()``, 1: Polygon, more: MultiPolygon), ring r = OPEN vertices [ring_off[r], ring_off[r+1]) of ``xy``.
    The rings are closed once, vectorised (first vertex appended), and the geometries are views into that array."""
    xy = np.ascontiguousarray(xy, dtype=np.float64)
    ring_off = np.asarray(ring_off, dtype=np.int64)
    poly_off = np.asarray(poly_off, dtype=np.int64)
    nr = len(ring_off) - 1
    lens = np.diff(ring_off)
    # closed copy: ring r occupies [ring_off[r] + r, ring_off[r+1] + r + 1)
    closed = np.empty((len(xy) + nr, 2), dtype=np.float64)
    src = np.arange(len(xy), dtype=np.int64)
    shift = np.repeat(np.arange(nr, dtype=np.int64), lens)
    closed[src + shift] = xy
    if nr:
        closed[ring_off[1:] + np.arange(nr)] = xy[np.minimum(ring_off[:-1], max(len(xy) - 1, 0))]
    coff = ring_off + np.arange(nr + 1)
    if _shapely is not None:  # pragma: no cover
        polys = _shapely.from_ragged_array(_shapely.GeometryType.POLYGON, closed, (coff, np.arange(nr + 1)))
        out = []
        for a, b in zip(poly_off[:-1], poly_off[1:]):
            out.append(_shapely.Polygon() if b == a else polys[a] if b - a == 1 else _shapely.MultiPolygon(list(polys[a:b])))
        return out
    rings = [Polygon.from_closed_view(closed[a:b]) for a, b in zip(coff[:-1], coff[1:])]
    out = []
    for a, b in zip(poly_off[:-1], poly_off[1:]):
        out.append(Polygon() if b == a else rings[a] if b - a == 1 else MultiPolygon.from_parts(rings[a:b]))
    return out
