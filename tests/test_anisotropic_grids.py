"""Flag grids (to_xarray, Detector) on grids whose longitude and latitude spacings differ: the buffer of
processing/events.py:75-79, r = (dlon + dlat) / 4 degrees, is measured in degrees, an ellipse in index units."""

from fractions import Fraction
from math import gcd, isqrt

import numpy as np
import pandas as pd
import pytest
import torch

import wavebreaking_b200 as wb
from oracle import geom as G
from oracle import pipeline as P
from wavebreaking_b200 import _lib, compat, detect, pipeline, spatial, synthetic
from test_indices import _contour_set_from_rings, compare_events

# (dlon, dlat): 5:4, 4:3, 3:4 (dlon < dlat), 11:4 (aspect 2.75) and 23:8 (aspect 2.875, where a diagonal unit step
# has lattice points inside the band and the rasteriser's unit-step shortcut must be off)
SPACINGS = [(1.25, 1.0), (1.0, 0.75), (0.75, 1.0), (2.75, 1.0), (2.875, 1.0)]


# ------------------------------------------------------------------ the rule and its limits (no device)
def test_grid_ratio_accepts_exact_small_ratios_below_aspect_3():
    assert detect.grid_ratio(0.625, 0.5) == (5, 4)  # MERRA-2
    assert detect.grid_ratio(1.25, 1.0) == (5, 4)
    assert detect.grid_ratio(2.5, 2.0) == (5, 4)
    assert detect.grid_ratio(1.0, 0.75) == (4, 3)
    assert detect.grid_ratio(0.75, 1.0) == (3, 4)
    assert detect.grid_ratio(2.75, 1.0) == (11, 4)
    assert detect.grid_ratio(2.875, 1.0) == (23, 8)
    assert detect.grid_ratio(0.5, 0.5) == (1, 1)
    assert detect.grid_ratio(0.1, 0.1 * (1 + 1e-12)) == (1, 1)  # spacings equal within 1e-9 stay isotropic


@pytest.mark.parametrize("dlon,dlat,match", [(3.0, 1.0, "aspect"), (1.0, 3.0, "aspect"), (1.0, 0.7, "integers <= 64"),
                                             (65.0 / 64.0, 1.0, "integers <= 64"), (0.0, 1.0, "positive")])
def test_grid_ratio_refuses_unsupported_spacings(dlon, dlat, match):
    with pytest.raises(ValueError, match=match):
        detect.grid_ratio(dlon, dlat)


@pytest.mark.parametrize("p,q", [(5, 4), (4, 3), (3, 4), (11, 4), (23, 8)])
def test_no_exact_ties_between_band_and_lattice(p, q):
    """16 p^2 q^2 C^2 == (p + q)^2 L has no solution for primitive edge directions |a|, |b| < 200 (a longer edge is a
    multiple g (a, b): C and sqrt(L) scale by g and the equation is the same), so the strict '<' of the rule never
    meets an exact tie; also the unit-step shortcut condition 16 p^2 q^2 >= (p + q)^2 (p^2 + q^2) holds up to 11:4
    and fails at 23:8"""
    kc, kl = 16 * p * p * q * q, (p + q) ** 2
    ties = []
    for a in range(0, 200):
        for b in range(-199, 200):
            if (a == 0 and b <= 0) or gcd(a, abs(b)) != 1:
                continue
            rhs = kl * (p * p * a * a + q * q * b * b)
            if rhs % kc == 0 and isqrt(rhs // kc) ** 2 == rhs // kc:
                ties.append((a, b))
    assert ties == []
    assert (kc >= kl * (p * p + q * q)) == (max(p, q) / min(p, q) < 2.76)


def _rule_fraction(pieces, i, j, lon, lat, dlon, dlat):
    """the to_xarray rule for grid point (i, j), in exact rational degrees: inside (non-zero winding), on the boundary
    or closer than (dlon + dlat) / 4 degrees to an edge"""
    r2 = (Fraction(dlon) + Fraction(dlat)) ** 2 / 16
    X, Y = Fraction(lon[i]), Fraction(lat[j])
    wn = 0
    for ring in pieces:
        pts = [(Fraction(lon[x]), Fraction(lat[y])) for x, y in np.asarray(ring)]
        for k in range(len(pts)):
            (x0, y0), (x1, y1) = pts[k], pts[(k + 1) % len(pts)]
            dx, dy, ex, ey = x1 - x0, y1 - y0, X - x0, Y - y0
            cross = dx * ey - dy * ex
            if y0 <= Y < y1 and cross > 0:
                wn += 1
            if y1 <= Y < y0 and cross < 0:
                wn -= 1
            L, D = dx * dx + dy * dy, ex * dx + ey * dy
            if D <= 0:
                d2 = ex * ex + ey * ey
            elif D >= L:
                d2 = (X - x1) ** 2 + (Y - y1) ** 2
            else:
                d2 = cross * cross / L
            if d2 < r2:
                return True
    return wn != 0


# ------------------------------------------------------------------ random polygons on anisotropic lattices
def _random_polygons_fuzz(seed, dlon, dlat, per_job=40):
    """calculate_properties + to_xarray on random simple lattice polygons (inside, across and beyond the last meridian)
    of a grid with spacings dlon, dlat: member counts, sums and properties (index-unit radius) and the flag grids
    (degree-space radius) equal the oracle; a sample of flag cells also equals the rule evaluated in fractions"""
    detect.clear_contexts()
    rng = np.random.default_rng(1300 + seed)
    nlon, nlat, add, njobs = 40, 21, 10, 2
    lon = np.arange(nlon) * dlon
    lat = -10.0 + np.arange(nlat) * dlat
    grid = P.Grid(lon, lat, synthetic.time_axis(njobs, 6.0))
    assert (grid.dlon, grid.dlat) == (dlon, dlat)
    rings = []
    while len(rings) < njobs * per_job:
        cx, cy = rng.integers(7, nlon + add - 7), rng.integers(7, nlat - 7)
        k = rng.integers(3, 12)
        ang = np.sort(rng.uniform(0, 2 * np.pi, k))
        rad = rng.uniform(0.8, 6.4, k)
        ring = np.c_[np.rint(cx + rad * np.cos(ang)), np.rint(cy + rad * np.sin(ang))].astype(int)
        keep = [0]
        for i in range(1, len(ring)):
            if (ring[i] != ring[keep[-1]]).any():
                keep.append(i)
        ring = ring[keep]
        if len(ring) > 1 and (ring[0] == ring[-1]).all():
            ring = ring[:-1]
        if len(ring) >= 3 and G.ring_is_simple(ring) and abs(G._ring_area2(ring)) > 0:
            rings.append(ring)
    jobs = np.repeat(np.arange(njobs), per_job)
    cs, closed, nx = _contour_set_from_rings(rings, jobs, njobs, nlat, nlon, add)
    data = rng.standard_normal((njobs, nlat, nlon))
    inten = rng.standard_normal((njobs, nlat, nlon))
    coords = detect.coord_tables(lat, lon, dlon, dlat)
    tables, flags = detect.run_indices(cs, spatial.to_device(data), coords, dlon, dlat,
                                       intensity=spatial.to_device(inten), which=("cutoffs",), gmax_nx=int(nx.max()),
                                       want_flags=True, min_caps=dict(seg_cap=8192))
    frame = pd.DataFrame({"date": grid.time[jobs], "level": 2.0, "closed": True, "exp_lon": nx * dlon,
                          "mean_lat": 0.0, "geometry": closed})
    want = dict(streamers=pd.DataFrame(), overturnings=pd.DataFrame(),
                cutoffs=P.calculate_cutoffs(data, grid, frame, intensity=inten, periodic_add=add * dlon))
    assert len(want["cutoffs"]) >= 20  # rings narrower than min_exp = 5 degrees of longitude are no events
    tab = tables["cutoffs"]
    assert (tab.split == 1).any(), np.bincount(tab.split)  # events across the last meridian
    compare_events(cs, tables, flags, want, grid, [2.0], data)
    props = detect.finish_properties(tab, grid.lon, grid.lat, grid.nlon)
    assert np.array_equal(props["intensity"], want["cutoffs"].intensity.values)
    # the rule in exact fractions on a sample of cells next to the events (where the band decides)
    fl = flags[detect.KINDS.index("cutoffs")].cpu().numpy()
    near = np.zeros_like(fl[0], dtype=bool)
    for e in range(len(tab)):
        for piece in want["cutoffs"].attrs["_index_pieces"][e]:
            x, y = np.asarray(piece).T
            near[max(y.min() - 1, 0):y.max() + 2, max(x.min() - 1, 0):x.max() + 2] = True
    cand = np.argwhere(near)
    for j, i in cand[rng.choice(len(cand), min(len(cand), 60), replace=False)]:
        for t in range(njobs):
            sel = [e for e in range(len(tab)) if int(tab.job[e]) == t]
            got = any(_rule_fraction(want["cutoffs"].attrs["_index_pieces"][e], i, j, lon, lat, dlon, dlat)
                      for e in sel)
            assert bool(fl[t, j, i]) == got, (t, j, i)


@pytest.mark.parametrize("dlon,dlat", SPACINGS)
def test_properties_and_flags_of_random_polygons_anisotropic_emu(emu, dlon, dlat):
    _random_polygons_fuzz(0, dlon, dlat)


@pytest.mark.gpu
@pytest.mark.parametrize("dlon,dlat", SPACINGS)
def test_properties_and_flags_of_random_polygons_anisotropic_gpu(gpu, dlon, dlat):
    _random_polygons_fuzz(1, dlon, dlat, per_job=70)


def _rings_raster_fuzz(seed, dlon, dlat):
    """wbk_rasterize_rings_grid (to_xarray for arbitrary event tables) on random simple polygons vs the oracle's buffer +
    contains rule in degree space, for the int8 grid and the last-writer float64 grid"""
    rng = np.random.default_rng(1400 + seed)
    nlat, nlon = 40, 64
    lon, lat = np.arange(nlon) * dlon, np.arange(nlat) * dlat
    LON, LAT = np.meshgrid(lon, lat)
    rings = []
    while len(rings) < 30:
        cx, cy = rng.integers(9, nlon - 9), rng.integers(9, nlat - 9)
        k = rng.integers(3, 12)
        ang = np.sort(rng.uniform(0, 2 * np.pi, k))
        rad = rng.uniform(0.8, 8.4, k)
        ring = np.unique(np.c_[np.rint(cx + rad * np.cos(ang)), np.rint(cy + rad * np.sin(ang))].astype(int), axis=0)
        ring = ring[np.argsort(np.arctan2(ring[:, 1] - ring[:, 1].mean(), ring[:, 0] - ring[:, 0].mean()))]
        if len(ring) >= 3 and G.ring_is_simple(ring) and abs(G._ring_area2(ring)) > 0:
            rings.append(ring)
    ring_t = rng.integers(0, 3, len(rings))
    vals = rng.standard_normal(len(rings))
    got = detect.rasterize_rings(rings, ring_t, nlat, nlon, 3, spacing=(dlon, dlat)).cpu().numpy()
    dev = spatial.to_device(np.zeros(1)).device
    out = torch.zeros((3, nlat, nlon), dtype=torch.float64, device=dev)
    got_v = detect.rasterize_rings(rings, ring_t, nlat, nlon, 3, spacing=(dlon, dlat), values=(out, vals)).cpu().numpy()
    want = np.zeros((3, nlat * nlon), dtype=np.int8)
    want_v = np.zeros((3, nlat * nlon))
    r = (dlon + dlat) / 4
    for ring, t, v in zip(rings, ring_t, vals):
        sel = G.buffered_contains([np.c_[lon[ring[:, 0]], lat[ring[:, 1]]]], r, LON.ravel(), LAT.ravel())
        want[t, sel] = 1
        want_v[t, sel] = v
    assert np.array_equal(got.reshape(3, -1), want)
    assert np.array_equal(got_v.reshape(3, -1), want_v)


@pytest.mark.parametrize("dlon,dlat", SPACINGS)
def test_rings_raster_grid_form_emu(emu, dlon, dlat):
    _rings_raster_fuzz(0, dlon, dlat)


@pytest.mark.gpu
@pytest.mark.parametrize("dlon,dlat", SPACINGS)
def test_rings_raster_grid_form_gpu(gpu, dlon, dlat):
    _rings_raster_fuzz(1, dlon, dlat)


# ------------------------------------------------------------------ whole pipeline
def _run(nlat, nlon, ntime, levels, step_hours=6.0):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, np.arange(ntime) * step_hours)
    grid = P.Grid(lon, lat, synthetic.time_axis(ntime, step_hours))
    assert grid.dlon != grid.dlat
    det = pipeline.Detector(lat, lon, levels=levels)
    res = det.run_batch(spatial.to_device(raw))
    want = P.detect_steps(raw, grid, levels=levels)
    for k, kind in enumerate(detect.KINDS):
        assert len(res.tables[kind]) == len(want["events"][kind]), kind
        assert np.array_equal(res.flags[k].cpu().numpy(), want["flags"][kind]), kind
    compare_events(res.contours, res.tables, res.flags, want["events"], grid, levels, want["smoothed"])
    nsplit = sum(int((res.tables[kind].split == 1).sum()) for kind in detect.KINDS)
    assert nsplit > 0  # events that straddle the last meridian (clipped and rasterised on the device)
    return res


@pytest.mark.parametrize("nlat,nlon,ntime,levels", [(91, 144, 2, [2.0, -2.0]), (181, 288, 1, [2.0])])
def test_detector_anisotropic_emu(emu, nlat, nlon, ntime, levels):
    _run(nlat, nlon, ntime, levels)


@pytest.mark.gpu
@pytest.mark.parametrize("nlat,nlon,ntime,levels", [(181, 288, 4, [2.0, -2.0]), (361, 576, 3, [2.0, -2.0])])
def test_detector_anisotropic_gpu(gpu, nlat, nlon, ntime, levels):
    _run(nlat, nlon, ntime, levels)


# ------------------------------------------------------------------ drop-in API
def _field(nlat=91, nlon=144, ntime=2):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, np.arange(ntime) * 6.0, dtype=np.float64)
    time = np.datetime64("1959-06-03T12", "ns") + np.arange(ntime) * np.timedelta64(6, "h")
    return compat.Field(raw, ("time", "lat", "lon"), {"time": time, "lat": lat, "lon": lon}, name="PV"), \
        P.Grid(lon, lat, time), raw


def _oracle_frame(frame):
    out = pd.DataFrame({k: frame[k].values for k in frame.columns if k != "geometry"})
    out["geometry"] = [[np.asarray(r, dtype=float) for r in compat.geometry_rings(g)] for g in frame["geometry"]]
    return out


def _api_case():
    data, grid, raw = _field()
    assert (grid.dlon, grid.dlat) == (2.5, 2.0)
    # the reference's known-answer square (tests/test_wavebreaking.py:116-128) on a 2.5 x 2 degree grid: 5 x 6 points
    # inside or on the boundary, none closer than r = 1.125 degrees outside
    sq = compat.make_frame({"date": [grid.time[0]]}, [compat.Polygon([(0, 0), (10, 0), (10, 10), (0, 10)])])
    flag = wb.to_xarray(data=data, events=sq, name="test_flag")
    assert flag.values.dtype == np.int8 and flag.values.sum() == 30
    assert np.array_equal(flag.values, P.to_xarray(np.zeros_like(raw), _oracle_frame(sq), grid))
    # a value column: later events overwrite earlier ones
    ev = compat.make_frame({"date": [grid.time[0], grid.time[0], grid.time[1]], "val": [3.0, 7.0, 5.0]},
                           [compat.Polygon([(0, 0), (10, 0), (10, 10), (0, 10)]),
                            compat.Polygon([(5, 4), (15, 4), (20, 16), (5, 14)]),
                            compat.Polygon([(100, -30), (130, -20), (105, 10)])])
    want_ev = _oracle_frame(ev)
    assert np.array_equal(wb.to_xarray(data, ev, flag="val").values,
                          P.to_xarray(np.zeros_like(raw), want_ev, grid, "val"))
    assert np.array_equal(wb.to_xarray(data, ev).values, P.to_xarray(np.zeros_like(raw), want_ev, grid))
    # frames of the index functions
    sm = wb.calculate_smoothed_field(data, 5)
    want_sm = P.smooth_field(raw, 5)
    c_o = P.calculate_contours(want_sm, 2, grid, 120, original_coordinates=False)
    st = wb.calculate_streamers(data=sm, contour_levels=2, periodic_add=120)
    co = wb.calculate_cutoffs(data=sm, contour_levels=2, periodic_add=120)
    for got, want in ((st, P.calculate_streamers(want_sm, grid, c_o)), (co, P.calculate_cutoffs(want_sm, grid, c_o))):
        assert len(got) == len(want) > 0
        assert np.array_equal(wb.to_xarray(sm, got).values, P.to_xarray(np.zeros_like(want_sm), want, grid))


def test_to_xarray_anisotropic_emu(emu):
    _api_case()


@pytest.mark.gpu
def test_to_xarray_anisotropic_gpu(gpu):
    _api_case()


# ------------------------------------------------------------------ refusals
def _refusals():
    for dlon, dlat, match in ((3.0, 1.0, "aspect"), (1.0, 65.0 / 64.0, "integers <= 64")):
        lon, lat = np.arange(20) * dlon, np.arange(10) * dlat
        time = np.datetime64("2000-01-01T00", "ns") + np.arange(1) * np.timedelta64(6, "h")
        data = compat.Field(np.zeros((1, 10, 20)), ("time", "lat", "lon"), {"time": time, "lat": lat, "lon": lon})
        sq = compat.make_frame({"date": [time[0]]}, [compat.Polygon([(lon[2], lat[2]), (lon[5], lat[2]),
                                                                     (lon[5], lat[5])])])
        with pytest.raises(ValueError, match=match):
            wb.to_xarray(data, sq)
        with pytest.raises(ValueError, match=match):
            pipeline.Detector(lat, lon)
        pipeline.Detector(lat, lon, want_flags=False).close()  # the event tables need no flag metric
        # the C-ABI refuses the same spacings with a message that names them
        ring = [np.array([[2, 2], [5, 2], [5, 5]])]
        lib = _lib.get()
        out = torch.zeros((1, 10, 20), dtype=torch.int8, device=lib.device)
        xy = torch.tensor(ring[0], dtype=torch.int32, device=lib.device)
        off = torch.tensor([0, 3], dtype=torch.int32, device=lib.device)
        t = torch.zeros(1, dtype=torch.int32, device=lib.device)
        with pytest.raises(_lib.WbkError, match="wbk_rasterize_rings_grid.*dlon=") as err:
            lib.call("wbk_rasterize_rings_grid", _lib.ptr(xy), _lib.ptr(off), _lib.ptr(t), None, 1, 10, 20, 1, dlon,
                     dlat, _lib.ptr(out), None, None, lib.stream())
        assert err.value.code == _lib.ERR_INVALID
        cs, closed, nx = _contour_set_from_rings(ring, np.zeros(1, dtype=np.int64), 1, 10, 20, 4)
        with pytest.raises(_lib.WbkError, match="wbk_events_raster.*dlon=") as err:
            detect.run_indices(cs, spatial.to_device(np.zeros((1, 10, 20))),
                               detect.coord_tables(lat, lon, dlon, dlat), dlon, dlat, which=("cutoffs",),
                               gmax_nx=int(nx.max()), want_flags=True)
        assert err.value.code == _lib.ERR_INVALID


def test_unsupported_spacings_are_refused_emu(emu):
    _refusals()
