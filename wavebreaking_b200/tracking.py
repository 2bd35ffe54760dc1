"""Temporal tracking of events: candidate pairs, exact overlap / distance tests and labels.

Reference: wavebreaking/processing/events.py:113-241 (``track_events``) and
wavebreaking/utils/index_utils.py:187-214 (``combine_shared``).

The columnar core (:func:`link_events`) works on events sorted by date:

* the pairs ``(i, j)`` with ``0 < date_j - date_i <= time_range`` (events.py:160-181) are an index window per
  event (two vectorised searches); ``wbk_track_candidates`` expands the windows on the device and drops the pairs
  whose bounding boxes are disjoint;
* ``by_overlap``: event polygons are lattice polygons (their vertices are grid points), so "the intersection has
  a positive area" is decided EXACTLY in integer arithmetic by ``wbk_track_overlap_exact``; only for
  ``overlap > 0`` the float64 areas of the overlapping pairs are evaluated (``wbk_track_overlap``);
* ``by_distance``: sklearn's haversine on the device, pairs within 1e-9 of the threshold are re-decided with
  libm in the reference's operand order (they are returned as the *near* list);
* labels: connected components, label = dense rank of the smallest member index (events.py:225-238).

:func:`track_sharded` runs the same on time-sharded ranks with a halo of ``time_range`` hours of events.
"""

import math

import numpy as np
import pandas as pd
import torch

from . import _lib, compat


def combine_shared(lst):
    """Connected components of index lists that share elements.

    Components come out in order of first appearance (like the reference's sweep over ``lst``);
    the members of a component are returned in ascending order (the reference returns them in
    Python-set iteration order, which is ascending for the small non-negative ints it is used with).
    """
    parent = {}

    def find(a):
        root = a
        while parent[root] != root:
            root = parent[root]
        while parent[a] != root:
            parent[a], a = root, parent[a]
        return root

    order = []
    for item in lst:
        item = [int(v) if isinstance(v, (np.integer,)) else v for v in item]
        for v in item:
            if v not in parent:
                parent[v] = v
                order.append(v)
        for v in item[1:]:
            ra, rb = find(item[0]), find(v)
            if ra != rb:
                parent[rb] = ra
    groups, seen = {}, []
    for v in order:
        r = find(v)
        if r not in groups:
            groups[r] = []
            seen.append(r)
        groups[r].append(v)
    return [sorted(groups[r]) for r in seen]


# ------------------------------------------------------------------------------------------------ polygons
class PolygonSoup:
    """Columnar (multi)polygons: polygon p = rings [poly_off[p], poly_off[p+1]), ring r = vertices
    [ring_off[r], ring_off[r+1]) of ``xy`` (open rings, no repeated closing vertex).  ``lattice`` tells whether
    ``xy`` holds exact integer lattice coordinates (int32, all in [0, 4096)): only then the exact test applies."""

    def __init__(self, xy, ring_off, poly_off, lattice):
        self.xy = np.ascontiguousarray(xy)
        self.ring_off = np.ascontiguousarray(ring_off, dtype=np.int32)
        self.poly_off = np.ascontiguousarray(poly_off, dtype=np.int32)
        self.lattice = bool(lattice)

    def __len__(self):
        return len(self.poly_off) - 1

    def take(self, idx):
        """Sub-soup of the polygons ``idx`` (in that order)."""
        idx = np.asarray(idx, dtype=np.int64)
        r0, r1 = self.poly_off[idx].astype(np.int64), self.poly_off[idx + 1].astype(np.int64)
        nr = r1 - r0
        rings = _ranges(r0, nr)
        v0, v1 = self.ring_off[rings].astype(np.int64), self.ring_off[rings + 1].astype(np.int64)
        nv = v1 - v0
        verts = _ranges(v0, nv)
        return PolygonSoup(self.xy[verts], np.r_[0, np.cumsum(nv)], np.r_[0, np.cumsum(nr)], self.lattice)

    @staticmethod
    def concat(soups):
        soups = [s for s in soups if s is not None]
        xy = np.concatenate([s.xy for s in soups]) if soups else np.zeros((0, 2), dtype=np.int32)
        ro, po, vo, rr = [np.zeros(1, dtype=np.int64)], [np.zeros(1, dtype=np.int64)], 0, 0
        for s in soups:
            ro.append(s.ring_off[1:].astype(np.int64) + vo)
            po.append(s.poly_off[1:].astype(np.int64) + rr)
            vo += len(s.xy)
            rr += len(s.ring_off) - 1
        return PolygonSoup(xy, np.concatenate(ro), np.concatenate(po), all(s.lattice for s in soups))

    def bounds(self):
        """int/float [n, 4] x0, y0, x1, y1 per polygon; empty polygons get an empty box (x0 > x1)."""
        n = len(self)
        v0 = self.ring_off[self.poly_off[:-1]].astype(np.int64)
        v1 = self.ring_off[self.poly_off[1:]].astype(np.int64)
        out = np.zeros((n, 4), dtype=self.xy.dtype)
        out[:, 0] = out[:, 1] = 1
        ok = v1 > v0
        if ok.any() and len(self.xy):
            starts = v0[ok]
            # reduceat over [v0, v1): polygons are contiguous and in order, empty ones are skipped
            mins = np.minimum.reduceat(self.xy, starts, axis=0)
            maxs = np.maximum.reduceat(self.xy, starts, axis=0)
            out[ok, 0:2] = mins
            out[ok, 2:4] = maxs
        return out


def _ranges(start, count):
    """Concatenated aranges start[i] .. start[i] + count[i] (vectorised)."""
    count = np.asarray(count, dtype=np.int64)
    total = int(count.sum())
    if total == 0:
        return np.zeros(0, dtype=np.int64)
    offs = np.repeat(np.cumsum(count) - count, count)
    return np.repeat(np.asarray(start, dtype=np.int64), count) + (np.arange(total, dtype=np.int64) - offs)


def _latticise(vals):
    """Map coordinate values onto an integer lattice ``(v - v0) / q`` if they all sit on one (q = smallest
    positive gap of the sorted unique values); returns the int array or None."""
    if len(vals) == 0:
        return np.zeros(0, dtype=np.int32)
    u = np.unique(vals)
    if len(u) == 1:
        return np.zeros(len(vals), dtype=np.int32)
    q = np.diff(u).min()
    idx = (vals - u[0]) / q
    snapped = np.rint(idx)
    if not np.allclose(idx, snapped, rtol=0, atol=1e-6) or snapped.max() >= 4096:
        return None
    return snapped.astype(np.int32)


def soup_from_geometries(geoms):
    """(Multi)Polygon geometries (shapely or wavebreaking_b200.compat) -> PolygonSoup.  Coordinates that sit on
    a regular lattice (events of a regular grid always do) are converted to exact integers."""
    xy, ring_len, poly_nr = [], [], []
    for g in geoms:
        rings = compat.geometry_rings(g)
        poly_nr.append(len(rings))
        for ring in rings:
            ring = np.asarray(ring, dtype=np.float64).reshape(-1, 2)
            xy.append(ring)
            ring_len.append(len(ring))
    allxy = np.concatenate(xy) if xy else np.zeros((0, 2))
    ring_off = np.r_[0, np.cumsum(ring_len)].astype(np.int64)
    poly_off = np.r_[0, np.cumsum(poly_nr)].astype(np.int64)
    ix, iy = _latticise(allxy[:, 0]), _latticise(allxy[:, 1])
    if ix is not None and iy is not None:
        return PolygonSoup(np.c_[ix, iy].astype(np.int32), ring_off, poly_off, True)
    return PolygonSoup(allxy, ring_off, poly_off, False)


# ------------------------------------------------------------------------------------------------ windows
def _hours_of(diff_ns):
    """pandas ``Series.dt.total_seconds() / 3600`` of an int64 nanosecond difference (events.py:165)."""
    return (np.int64(diff_ns) / 1e9) / 3600


def time_keys(dates):
    """(keys, window(time_range)) for the date column: int64 nanoseconds for datetimes (the window is the largest
    nanosecond difference whose ``total_seconds() / 3600`` is still <= time_range), float64 otherwise."""
    dates = np.asarray(dates)
    if np.issubdtype(dates.dtype, np.datetime64):
        keys = dates.astype("datetime64[ns]").astype(np.int64)

        def window(time_range):
            lo, hi = 0, 1 << 62
            while lo < hi:  # monotone: rounded division twice
                mid = (lo + hi + 1) >> 1
                if _hours_of(mid) <= time_range:
                    lo = mid
                else:
                    hi = mid - 1
            return np.int64(lo)

        return keys, window
    keys = dates.astype(np.float64)
    return keys, (lambda time_range: float(time_range))


def windows(keys_sorted, win):
    """lo, hi (int32) per event: events j in [lo, hi) satisfy 0 < key_j - key_i <= win."""
    k = keys_sorted
    lo = np.searchsorted(k, k, side="right")
    if k.dtype == np.int64:
        hi = np.searchsorted(k, k + win, side="right")
    else:
        hi = np.searchsorted(k, k + win, side="right")
        n = len(k)
        # the reference compares the rounded difference: fix the boundary cases of the rounded sum
        for _ in range(4):
            up = (hi < n) & (k[np.minimum(hi, n - 1)] - k <= win)
            dn = (hi > lo) & (k[np.maximum(hi - 1, 0)] - k > win)
            if not (up.any() or dn.any()):
                break
            hi = hi + up - dn
    hi = np.maximum(hi, lo)
    return lo.astype(np.int32), hi.astype(np.int32)


# ------------------------------------------------------------------------------------------------ device steps
def _dev(a, lib):
    return torch.from_numpy(np.ascontiguousarray(a)).to(lib.device)


def candidate_pairs(lo, hi, bbox=None, first=0, last=None):
    """Pairs (i, j), j in [lo[i], hi[i]), whose integer bounding boxes intersect; i restricted to [first, last).
    Returns an (m, 2) int32 array in no particular order."""
    lib = _lib.get()
    n = len(lo)
    last = n if last is None else last
    lo = np.asarray(lo, dtype=np.int32).copy()
    hi = np.asarray(hi, dtype=np.int32).copy()
    lo[:first], hi[:first] = 0, 0
    lo[last:], hi[last:] = 0, 0
    out = []
    cnt = (hi - lo).astype(np.int64)
    d_bbox = _dev(np.asarray(bbox, dtype=np.int32), lib) if bbox is not None else None
    chunk_cap = 1 << 26
    # chunks of events whose windows hold at most chunk_cap pairs
    cum = np.cumsum(cnt)
    start = 0
    while start < n:
        base = cum[start - 1] if start else 0
        end = int(np.searchsorted(cum, base + chunk_cap, side="right"))
        end = max(end, start + 1)
        cap = int(cum[end - 1] - base)
        if cap > 0:
            l2, h2 = lo.copy(), hi.copy()
            l2[:start], h2[:start] = 0, 0
            l2[end:], h2[end:] = 0, 0
            d_pairs = torch.empty((cap, 2), dtype=torch.int32, device=lib.device)
            d_count = torch.zeros(1, dtype=torch.int32, device=lib.device)
            d_lo, d_hi = _dev(l2, lib), _dev(h2, lib)  # (named: the buffers must outlive the launch)
            lib.call("wbk_track_candidates", _lib.ptr(d_lo), _lib.ptr(d_hi), _lib.ptr(d_bbox), n,
                     _lib.ptr(d_pairs), cap, _lib.ptr(d_count), lib.stream())
            m = int(d_count.item())
            out.append(d_pairs[:m].cpu().numpy())
        start = end
    return np.concatenate(out) if out else np.zeros((0, 2), dtype=np.int32)


def _edge_table(soup):
    """Per vertex: its edge (x0, y0, x1, y1) to the next vertex of the ring, and the ring's orientation sign."""
    xy = soup.xy.astype(np.int64)
    nv = np.diff(soup.ring_off).astype(np.int64)
    V = len(xy)
    nxt = np.arange(V, dtype=np.int64) + 1
    ends = soup.ring_off[1:].astype(np.int64)[nv > 0] - 1
    nxt[ends] = soup.ring_off[:-1].astype(np.int64)[nv > 0]
    edges = np.c_[xy, xy[nxt]] if V else np.zeros((0, 4), dtype=np.int64)
    cross = edges[:, 0] * edges[:, 3] - edges[:, 2] * edges[:, 1]
    area2 = np.add.reduceat(cross, soup.ring_off[:-1].astype(np.int64)[nv > 0]) if V else np.zeros(0, dtype=np.int64)
    ring_sign = np.zeros(len(nv), dtype=np.int32)
    ring_sign[nv > 0] = np.sign(area2).astype(np.int32)
    vsign = np.repeat(ring_sign, nv)
    return edges.astype(np.int32), vsign.astype(np.int32)


def overlap_exact(soup, pairs):
    """int32 [m]: bit 0 = the polygons of the pair overlap in a region of positive area (exact), bit 1 = the
    boundaries touch without crossing (decided by the piecewise rule)."""
    lib = _lib.get()
    pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
    if len(pairs) == 0:
        return np.zeros(0, dtype=np.int32)
    if not soup.lattice:
        raise ValueError("overlap_exact needs lattice polygons")
    if len(soup.xy) == 0:
        return np.zeros(len(pairs), dtype=np.int32)
    # edge table (x0, y0, x1, y1 per vertex) and ring orientation signs, built ON the device from the uploaded vertices
    # (tens of millions of vertices for a decade of events: numpy would dominate the whole tracking step)
    dev = lib.device
    xy = torch.from_numpy(np.ascontiguousarray(soup.xy, dtype=np.int32)).to(dev)
    ring_off = torch.from_numpy(soup.ring_off.astype(np.int64)).to(dev)
    V = xy.shape[0]
    nv = ring_off[1:] - ring_off[:-1]
    nxt = torch.arange(1, V + 1, device=dev, dtype=torch.int64)
    live = nv > 0
    nxt[ring_off[1:][live] - 1] = ring_off[:-1][live]
    edges = torch.cat([xy, xy[nxt]], dim=1).contiguous()  # int32 [V, 4]
    e64 = edges.to(torch.int64)
    cross = e64[:, 0] * e64[:, 3] - e64[:, 2] * e64[:, 1]
    csum = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(cross, 0)])
    area2 = csum[ring_off[1:]] - csum[ring_off[:-1]]
    vsign = torch.repeat_interleave(torch.sign(area2).to(torch.int32), nv).contiguous()
    out = torch.empty(len(pairs), dtype=torch.int32, device=dev)
    bufs = [edges, vsign, _dev(soup.ring_off, lib), _dev(soup.poly_off, lib), _dev(pairs, lib)]  # alive until the read
    lib.call("wbk_track_overlap_exact", *[_lib.ptr(b) for b in bufs], len(pairs), _lib.ptr(out), lib.stream())
    return out.cpu().numpy()


def overlap_areas(geoms_or_soup, pairs):
    """(area A, area B, area A n B) in float64 for every pair, computed by wbk_track_overlap."""
    lib = _lib.get()
    soup = geoms_or_soup if isinstance(geoms_or_soup, PolygonSoup) else soup_from_geometries(list(geoms_or_soup))
    pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
    if len(pairs) == 0:
        return np.zeros((0, 3))
    xy = np.ascontiguousarray(soup.xy, dtype=np.float64)
    if len(xy) == 0:
        return np.zeros((len(pairs), 3))
    out = torch.empty((len(pairs), 3), dtype=torch.float64, device=lib.device)
    bufs = [_dev(a, lib) for a in (xy, soup.ring_off, soup.poly_off, pairs)]  # alive until the result is read
    lib.call("wbk_track_overlap", *[_lib.ptr(b) for b in bufs], len(pairs), _lib.ptr(out), lib.stream())
    return out.cpu().numpy()


def _haversine_libm(p1, p2):
    """sklearn DistanceMetric('haversine') of two (lat, lon)-radian points with libm, operand order of
    sklearn/metrics/_dist_metrics.pyx.tp:2641-2656."""
    s0 = math.sin(0.5 * (p1[0] - p2[0]))
    s1 = math.sin(0.5 * (p1[1] - p2[1]))
    return 2 * math.asin(math.sqrt(s0 * s0 + math.cos(p1[0]) * math.cos(p2[0]) * s1 * s1))


def pair_distances(rad, pairs):
    """Haversine (radians on the unit sphere) for the pairs of rows of ``rad`` [n, 2] on the device."""
    lib = _lib.get()
    pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
    if len(pairs) == 0:
        return np.zeros(0)
    out = torch.empty(len(pairs), dtype=torch.float64, device=lib.device)
    d_rad, d_pairs = _dev(np.asarray(rad, dtype=np.float64), lib), _dev(pairs, lib)  # alive until the result is read
    lib.call("wbk_track_distance", _lib.ptr(d_rad), _lib.ptr(d_pairs), len(pairs), _lib.ptr(out), lib.stream())
    return out.cpu().numpy()


# ------------------------------------------------------------------------------------------------ linking
NEAR_REL = 1e-9


def decide_pairs(pairs, method, overlap=0, distance=1000, exact=None, areas=None, dist=None, rad=None):
    """The linking decision of events.py:187-217 for candidate pairs of lattice polygons (``by_overlap``) or of centres
    of mass (``by_distance``).  ``exact(pairs)``: the ``overlap_exact`` flags, ``areas(pairs)``: ``overlap_areas``,
    ``dist(pairs)``: ``pair_distances`` on the unit sphere, ``rad``: the radians rows for the libm re-decision.
    Returns ``(links, near)``: the linked pairs and the pairs decided within NEAR_REL of a threshold."""
    near = np.zeros((0, 2), dtype=np.int32)
    if method == "by_distance":
        d = dist(pairs) * 6371
        check = d < distance
        close = np.abs(d - distance) <= NEAR_REL * abs(distance)
        for k in np.nonzero(close)[0]:  # CUDA libm vs glibc: re-decide in the reference's arithmetic
            check[k] = _haversine_libm(rad[pairs[k, 0]], rad[pairs[k, 1]]) * 6371 < distance
        return pairs[check], pairs[close]
    flag = exact(pairs)
    pos = (flag & 1) == 1
    if overlap == 0:
        return pairs[pos], near
    ratio = np.zeros(len(pairs))
    if pos.any():
        ar = areas(pairs[pos])
        inter = np.maximum(ar[:, 2], np.finfo(np.float64).tiny)  # exact test says positive
        ratio[pos] = inter / (ar[:, 1] + ar[:, 0] - inter)
    if overlap < 0:
        ar = areas(pairs[~pos])
        with np.errstate(divide="ignore", invalid="ignore"):
            ratio[~pos] = 0.0 / (ar[:, 1] + ar[:, 0])
    with np.errstate(invalid="ignore"):
        check = ratio > overlap
    return pairs[check], pairs[pos & (np.abs(ratio - overlap) <= NEAR_REL)]


def link_events(keys_sorted, win, method="by_overlap", soup=None, com=None, overlap=0, distance=1000, first=0,
                last=None, stats=None):
    """Linked pairs among events sorted by ``keys_sorted`` (events.py:160-217).

    Returns ``(links, npairs_in_range, near)``: links (m, 2) positions i < j in the sorted order with i in
    [first, last); near lists the pairs decided within NEAR_REL of a threshold (float64 decisions only; the exact
    overlap test has no such pairs)."""
    import time as _time

    tick = [_time.perf_counter()]

    def lap(name):
        if stats is not None:
            now = _time.perf_counter()
            stats["t_" + name] = stats.get("t_" + name, 0.0) + now - tick[0]
            tick[0] = now

    lo, hi = windows(keys_sorted, win)
    lap("windows")
    n = len(lo)
    last = n if last is None else last
    n_in_range = int((hi[first:last] - lo[first:last]).sum())
    near = np.zeros((0, 2), dtype=np.int32)
    if method == "by_distance":
        pairs = candidate_pairs(lo, hi, None, first, last)
        # the reference feeds (lon, lat) where haversine expects (lat, lon) (events.py:189-195); kept
        rad = np.radians(np.asarray(com, dtype=np.float64).reshape(-1, 2))
        links, near = decide_pairs(pairs, method, distance=distance, dist=lambda p: pair_distances(rad, p), rad=rad)
    elif method == "by_overlap":
        if overlap < 0:
            pairs = candidate_pairs(lo, hi, None, first, last)  # 0 / union > overlap holds for disjoint pairs too
        else:
            box = soup.bounds()
            if not soup.lattice:  # float boxes: integer boxes that contain them
                box = np.c_[np.floor(box[:, :2]), np.ceil(box[:, 2:])]
                box = np.clip(box, -2**30, 2**30)
            pairs = candidate_pairs(lo, hi, box.astype(np.int32), first, last)
        lap("candidates")
        if soup.lattice:
            links, near = decide_pairs(pairs, method, overlap, exact=lambda p: overlap_exact(soup, p),
                                       areas=lambda p: overlap_areas(soup, p))
            lap("overlap_exact")
        else:
            # polygons off any common lattice: float64 areas; an intersection below 1e-12 of the summed areas is
            # rounding noise of the triangle-fan sum and counts as empty (such pairs are listed as near)
            ar = overlap_areas(soup, pairs)
            noise = 1e-12 * (ar[:, 0] + ar[:, 1])
            inter = np.where(ar[:, 2] > noise, ar[:, 2], 0.0)
            with np.errstate(divide="ignore", invalid="ignore"):
                ratio = inter / (ar[:, 1] + ar[:, 0] - inter)
                check = ratio > overlap
            near = pairs[(np.abs(ar[:, 2]) <= 10 * noise) | (np.abs(ratio - overlap) <= NEAR_REL)]
            links = pairs[check]
    else:
        raise ValueError("'{}' not supported as method! Supported methods are 'by_overlap' and 'by_distance'".format(method))
    if stats is not None:
        stats["pairs_in_range"] = stats.get("pairs_in_range", 0) + n_in_range
        stats["candidates"] = stats.get("candidates", 0) + len(pairs)
        stats["links"] = stats.get("links", 0) + len(links)
        stats["near"] = stats.get("near", 0) + len(near)
    return links, n_in_range, near


def component_min(n, links):
    """For every node 0..n-1 the smallest node index of its connected component."""
    if len(links) == 0:
        return np.arange(n, dtype=np.int64)
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components

    g = coo_matrix((np.ones(len(links), dtype=np.int8), (links[:, 0], links[:, 1])), shape=(n, n))
    _, comp = connected_components(g, directed=False)
    cmin = np.full(comp.max() + 1, n, dtype=np.int64)
    np.minimum.at(cmin, comp, np.arange(n, dtype=np.int64))
    return cmin[comp]


def labels_from_links(n, links):
    """events.py:225-238: every event starts with its own index, a group takes the smallest member index, then the
    labels are renumbered densely in ascending order."""
    label = component_min(n, links)
    _, dense = np.unique(label, return_inverse=True)
    return dense.astype(np.int64)


def default_time_range(dates):
    """events.py:155-157: the smallest positive difference of consecutive dates, in hours."""
    date_dif = pd.Series(dates).diff()
    return date_dif[date_dif > pd.Timedelta(0)].min().total_seconds() / 3600


def track_columnar(dates, method="by_overlap", soup=None, com=None, time_range=None, overlap=0, distance=1000,
                   stats=None):
    """Labels (in input order) for events given as columns.  Raises like the reference when no pair is in range."""
    dates = np.asarray(dates)
    n = len(dates)
    if time_range is None:
        time_range = default_time_range(dates)
    keys, window = time_keys(dates)
    order = np.argsort(keys, kind="stable")
    sorted_already = bool(np.all(order == np.arange(n)))
    ks = keys if sorted_already else keys[order]
    if soup is not None and not sorted_already:
        soup = soup.take(order)
    if com is not None and not sorted_already:
        com = np.asarray(com)[order]
    links, n_in_range, near = link_events(ks, window(time_range), method, soup, com, overlap, distance, stats=stats)
    if n_in_range == 0:
        raise ValueError("No events detected in the time range: {}".format(time_range))
    links = order[links] if not sorted_already else links
    return labels_from_links(n, links.reshape(-1, 2)), (order[near] if not sorted_already else near)


def track_events(events, time_range=None, method="by_overlap", buffer=0, overlap=0, distance=1000):
    """events.py:151-241; ``buffer`` other than 0 is not supported (GEOS buffering is out of scope)."""
    events = events.reset_index(drop=True)
    if method not in ("by_overlap", "by_distance"):
        # the reference builds the candidate pairs first, so an empty range is reported before a bad method
        keys, window = time_keys(events.date.values)
        tr = default_time_range(events.date.values) if time_range is None else time_range
        lo, hi = windows(np.sort(keys), window(tr))
        if int((hi - lo).sum()) == 0:
            raise ValueError("No events detected in the time range: {}".format(tr))
        raise ValueError("'{}' not supported as method! Supported methods are 'by_overlap' and 'by_distance'".format(method))
    soup = com = None
    if method == "by_overlap":
        if buffer != 0:
            raise NotImplementedError("track_events(by_overlap): only buffer=0 is supported")
        soup = soup_from_geometries(list(events.geometry))
    else:
        com = np.asarray(list(events.com), dtype=np.float64)
    labels, near = track_columnar(events.date.values, method, soup, com, time_range, overlap, distance)
    events["label"] = labels
    if len(near):
        events.attrs["near_threshold_pairs"] = np.asarray(near).tolist()
    return events.sort_values(by=["label", "date"])
