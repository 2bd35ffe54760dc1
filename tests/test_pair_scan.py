"""The streamer pair scan (streamer_prep_kernel + pair_scan_kernel) against the reference's pair matrices.

The reference keeps the pairs with geo < geo_dis, cont > cont_dis and |x1 - x2| <= 120 (streamer_index.py:130-157).
The device skips 32 x 32 tiles whose bounding boxes are provably further apart than geo_dis and decides every pair
in fp32 (__sinf) first; only pairs inside an error margin are re-decided in fp64 and, within 1e-9 of a threshold,
listed in the near list (wbk_near_list).  These tests place thresholds on lattice distances, on coarse grids whose
column gaps fold past 180 degrees of longitude, near the pole and across the seam, and check the near list pair by
pair and the streamers event by event.  Every emulator test has a GPU twin with the same parameters: only there do
__sinf and CUDA's libm run.  The *_sinf_worst tests run the emulator with __sinf at its documented error bound."""

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import geom as G
from oracle import pipeline as P
from wavebreaking_b200 import _lib, detect, spatial, synthetic
from test_indices import _contour_set_from_rings, _random_walk_contour, compare_events

R = 6371.0
GRIDS = {"0.25": (721, 1440), "1": (181, 360), "2.5x2": (91, 144), "2.8125": (65, 128), "3": (61, 120),
         "4": (46, 90), "5": (37, 72)}


@pytest.fixture()
def emu_sinf_worst(emu_lib):
    """The emulator build in which __sinf errs by its documented maximum (2^-21.41), sign alternating per call."""
    import build_emu

    prev = _lib._LIB
    lib = _lib.use_library(build_emu.build(variant="sinf_worst"), "cpu")
    detect.clear_contexts()
    yield lib
    detect.clear_contexts()
    _lib._LIB = prev


def _grid(name, njobs=1):
    nlat, nlon = GRIDS[name]
    lat, lon = synthetic.grid_coords(nlat, nlon)
    return P.Grid(lon, lat, synthetic.time_axis(njobs, 6.0))


def _run(grid, walks, geo_dis, cont_dis, data=None, want_flags=False):
    """hand-made open contours, one job each, through wbk_index_run; returns the streamer table, the flag grids and
    the near list as [job, contour, i, j, bits] (bit 0 kept, bit 1 geo band, bit 2 cont band) with its total count"""
    detect.clear_contexts()
    njobs = len(walks)
    add = int(120 / grid.dlon)
    jobs = np.arange(njobs)
    cs, contours, nx = _contour_set_from_rings(walks, jobs, njobs, grid.nlat, grid.nlon, add)
    meta = cs.meta.cpu().numpy().copy()
    meta[:, 0] = 0  # open contours
    cs.meta = torch.from_numpy(meta).to(cs.meta.device)
    cs._host = None
    if data is None:
        data = np.zeros((njobs, grid.nlat, grid.nlon))
    coords = detect.coord_tables(grid.lat, grid.lon, grid.dlon, grid.dlat)
    tables, flags = detect.run_indices(cs, spatial.to_device(data), coords, grid.dlon, grid.dlat,
                                       which=("streamers",), gmax_nx=int(nx.max()), geo_dis=geo_dis,
                                       cont_dis=cont_dis, want_flags=want_flags)
    lib = _lib.get()
    ctx = detect.get_context(grid.nlat, grid.nlon, add, njobs)
    recs = torch.zeros((_lib.NEAR_CAP, 4), dtype=torch.int32, device=lib.device)
    cnt = torch.zeros(1, dtype=torch.int32, device=lib.device)
    lib.call("wbk_near_list", ctx.handle, _lib.ptr(recs), _lib.NEAR_CAP, _lib.ptr(cnt), lib.stream())
    total = int(cnt.cpu()[0])
    r = recs.cpu().numpy()[:min(total, _lib.NEAR_CAP)]
    near = np.c_[r[:, 0], r[:, 1], r[:, 2], r[:, 3] & 0x0FFFFFFF, (r[:, 3] >> 28) & 7]
    return cs, tables, flags, near, total


def _matrices(pts, grid):
    """the reference's geo and cont matrices of one contour (streamer_index.py:130-135)"""
    coords = np.c_[grid.lat[pts[:, 1]], grid.lon[pts[:, 0] % grid.nlon]]
    geo = P.dist.pairwise(np.radians(coords)) * R
    on = np.insert(np.diagonal(geo, 1), 0, 0)
    cont = np.cumsum(np.triu(np.tile(on, (len(on), 1)), k=1), axis=1)
    return geo, cont


# ------------------------------------------------------------------------------------ near-band completeness
def _row(grid, lat):
    return int(np.argmin(np.abs(grid.lat - lat)))


def _other_row(grid, y0, k):
    """the row k rows south of y0, or north of it if that is the south pole or beyond (the pole rows are one point,
    where every longitude is the same distance away)"""
    for y1 in (y0 - k, y0 + k):
        if 0 < y1 < grid.nlat - 1:
            return y1
    return None


def _legs(grid, kind, y0, k):
    """An open contour of two zonal legs: east along row ya, then west along row yb, across the seam and into the
    extended part.  Every point of the outbound leg pairs with points of the return leg k rows / columns away along
    the whole legs (a family of zonal translates with one lattice distance, each decided with different fp32
    longitudes), the along-contour distance between them growing towards the west end."""
    W = grid.nlon + int(120 / grid.dlon)
    x0 = max(0, W - 600)  # 0.25 degrees: the last 120 real columns and the 480 columns of the extension
    xs = np.arange(x0, W)
    if kind == "zonal":
        ya = yb = y0
        out = xs[((xs - x0) // k) % 2 == 0]
        back = xs[((xs - x0) // k) % 2 == 1][::-1]
    else:
        ya, yb = y0, _other_row(grid, y0, k)
        out, back = xs, xs[::-1]
    return np.r_[np.c_[out, np.full(len(out), ya)], np.c_[back, np.full(len(back), yb)]].astype(np.int64)


def _lattice_pair(grid, kind, lat, target):
    """row, offset k and the reference's distance of the lattice pair of the given orientation nearest to target km"""
    y0 = _row(grid, lat)
    best = None
    for k in range(1, 121):
        y1 = y0 if kind == "zonal" else _other_row(grid, y0, k)
        if y1 is None:
            break
        dx, dy = (0 if kind == "meridional" else k), y1 - y0
        a = np.radians([[grid.lat[y0], grid.lon[0]], [grid.lat[y0 + dy], grid.lon[dx % grid.nlon]]])
        d = float(P.dist.pairwise(a)[0, 1] * R)
        if d > 0 and (best is None or abs(np.log(d / target)) < abs(np.log(best[2] / target))):
            best = (y0, k, d)
    return best


# (grid, target g in km, orientation, latitude, sign of the 1e-12 offset): every target on every grid, orientations
# and latitudes cycled so that each grid sees all of them
NEAR_CASES = []
for _gi, _gname in enumerate(("0.25", "1", "2.5x2", "2.8125", "3", "4")):
    for _ti, _target in enumerate((25, 50, 100, 200, 400, 800, 1600, 3200)):
        NEAR_CASES.append((_gname, _target, ("meridional", "zonal", "diagonal")[(_ti + _gi) % 3],
                           (0.0, 45.0, 70.0, 85.5)[(_ti + 2 * _gi) % 4], (1, -1)[(_ti + _gi) % 2]))


def _near_band(gname, target, kind, lat, sign, cont_dis=1500.0):
    grid = _grid(gname)
    y0, k, d = _lattice_pair(grid, kind, lat, target)
    walk = _legs(grid, kind, y0, k)
    g = d * (1 + sign * 1e-12)
    _, _, _, near, total = _run(grid, [walk], g, cont_dis)
    assert total == len(near) <= _lib.NEAR_CAP
    geo, cont = _matrices(walk, grid)
    x = walk[:, 0]
    i, j = np.triu_indices(len(walk), k=1)
    ok_x = np.abs(x[i] - x[j]) <= 120
    must = ok_x & (cont[i, j] > cont_dis * (1 + 2e-9)) & (np.abs(geo[i, j] - g) <= 0.5e-9 * g)
    assert must.sum() >= 8, (gname, target, kind, lat, int(must.sum()))
    listed = {(int(a), int(b)): int(f) for a, b, f in zip(near[:, 2], near[:, 3], near[:, 4])}
    for a, b in zip(i[must], j[must]):
        f = listed.get((int(a), int(b)))
        assert f is not None and f & 2, (gname, target, kind, lat, a, b, walk[a], walk[b])
        assert bool(f & 1) == (geo[a, b] < g), (a, b)
    for (a, b), f in listed.items():
        if f & 2:
            assert abs(geo[a, b] - g) <= 2e-9 * g, (a, b, geo[a, b], g)
    return int(must.sum())


@pytest.mark.parametrize("gname,target,kind,lat,sign", NEAR_CASES)
def test_near_band_is_complete_emu(emu, gname, target, kind, lat, sign):
    _near_band(gname, target, kind, lat, sign)


@pytest.mark.gpu
@pytest.mark.parametrize("gname,target,kind,lat,sign", NEAR_CASES)
def test_near_band_is_complete_gpu(gpu, gname, target, kind, lat, sign):
    _near_band(gname, target, kind, lat, sign)


# the fp32 margin matters where the threshold is small: every target up to 400 km on four grids
SINF_CASES = [c for c in NEAR_CASES if c[1] <= 400 and c[0] in ("0.25", "1", "2.5x2", "4")]


@pytest.mark.parametrize("gname,target,kind,lat,sign", SINF_CASES)
def test_near_band_is_complete_sinf_worst(emu_sinf_worst, gname, target, kind, lat, sign):
    _near_band(gname, target, kind, lat, sign)


CONT_CASES = [("1", 100, "meridional", 45.0, 1, 500.0), ("1", 400, "diagonal", 0.0, -1, 5000.0),
              ("2.5x2", 800, "zonal", 45.0, 1, 500.0), ("0.25", 50, "diagonal", 45.0, -1, 5000.0),
              ("4", 1600, "meridional", 70.0, 1, 5000.0)]


@pytest.mark.parametrize("gname,target,kind,lat,sign,cont_dis", CONT_CASES)
def test_near_band_across_cont_dis_emu(emu, gname, target, kind, lat, sign, cont_dis):
    _near_band(gname, target, kind, lat, sign, cont_dis)


@pytest.mark.gpu
@pytest.mark.parametrize("gname,target,kind,lat,sign,cont_dis", CONT_CASES)
def test_near_band_across_cont_dis_gpu(gpu, gname, target, kind, lat, sign, cont_dis):
    _near_band(gname, target, kind, lat, sign, cont_dis)


def _cont_threshold(gname, lat, sign):
    """cont_dis placed 1e-12 above / below the along-contour distance of one pair well inside geo_dis: the pair is
    listed with the cont bit, kept iff the reference's row cumsum exceeds the threshold"""
    grid = _grid(gname)
    walk = _legs(grid, "meridional", _row(grid, lat), 3)
    geo, cont = _matrices(walk, grid)
    x = walk[:, 0]
    ii, jj = np.nonzero(np.triu((np.abs(x[:, None] - x[None, :]) <= 120) & (cont > 1000) & (geo < 600), k=1))
    assert len(ii)
    i, j = int(ii[len(ii) // 2]), int(jj[len(ii) // 2])
    c = float(cont[i, j]) * (1 + sign * 1e-12)
    _, _, _, near, total = _run(grid, [walk], 1000.0, c)
    assert total == len(near)
    rec = near[(near[:, 2] == i) & (near[:, 3] == j)]
    assert len(rec) == 1 and rec[0, 4] & 4
    assert bool(rec[0, 4] & 1) == (cont[i, j] > c)
    band = np.abs(cont - c) <= 0.5e-9 * c
    for a, b, f in zip(near[:, 2], near[:, 3], near[:, 4]):
        if f & 4:
            assert abs(cont[a, b] - c) <= 2e-9 * c
    must = np.triu(band & (geo < 1000 * (1 - 2e-9)) & (np.abs(x[:, None] - x[None, :]) <= 120), k=1)
    listed = set(zip(near[:, 2].tolist(), near[:, 3].tolist()))
    assert all((int(a), int(b)) in listed for a, b in zip(*np.nonzero(must)))


CONT_THRESHOLD_CASES = [("1", 45.0, 1), ("1", 45.0, -1), ("3", 70.0, 1), ("0.25", 0.0, -1)]


@pytest.mark.parametrize("gname,lat,sign", CONT_THRESHOLD_CASES)
def test_cont_threshold_pair_is_listed_emu(emu, gname, lat, sign):
    _cont_threshold(gname, lat, sign)


@pytest.mark.gpu
@pytest.mark.parametrize("gname,lat,sign", CONT_THRESHOLD_CASES)
def test_cont_threshold_pair_is_listed_gpu(gpu, gname, lat, sign):
    _cont_threshold(gname, lat, sign)


# ------------------------------------------------------------------------------------ event parity
def _spike(grid, ybase, amp, spike_x, tip=None):
    """a three-wave sine across the extended grid with one strict extreme (row ybase + tip, default amp + 2) at
    spike_x and its periodic copy: on a coarse grid the two tips are one point 360 degrees apart (distance 0) and a
    pair of the reference"""
    W = grid.nlon + int(120 / grid.dlon)
    xs = np.arange(W)
    ys = ybase + np.rint(amp * np.sin(2 * np.pi * xs / grid.nlon * 3)).astype(int)
    ys[xs % grid.nlon == spike_x] = ybase + (amp + 2 if tip is None else tip)
    return np.c_[xs, ys].astype(np.int64)


def _band_walk(rng, W, ylo, yhi, y0):
    """random walk across the extended width that stays between rows ylo and yhi (revisited points dropped)"""
    x, y = 0, y0
    pts = [(x, y)]
    while x < W - 1:
        dx = int(rng.choice([1, 1, 0]))
        dy = int(rng.choice([-1, 0, 1])) if dx else int(rng.choice([-1, 1]))
        x = min(x + dx, W - 1)
        y = int(min(max(y + dy, ylo), yhi))
        pts.append((x, y))
    seen, out = set(), []
    for p in pts:
        if p not in seen:
            seen.add(p)
            out.append(p)
    return np.asarray(out, dtype=np.int64)


def _event_parity(grid, walks, geo_dis, cont_dis, seed=0, min_events=1):
    """streamers of hand-made open contours (one job each) vs calculate_streamers, event by event; events may differ
    only where a listed near pair lies inside them or where the near-tie bit marks them.  Every common event has the
    oracle's member count, com, mean_var and area; the rings, pieces and flag grids are compared as well unless an
    event across the last meridian is not a simple ring (GEOS-invalid, SURVEY A.5: its pieces are unpinned)."""
    rng = np.random.default_rng(900 + seed)
    njobs = len(walks)
    data = rng.standard_normal((njobs, grid.nlat, grid.nlon))
    cs, tables, flags, near, total = _run(grid, walks, geo_dis, cont_dis, data=data, want_flags=True)
    assert total == len(near)
    nx = np.array([len(np.unique(w[:, 0])) for w in walks])
    frame = pd.DataFrame({"date": grid.time[:njobs], "level": 2.0, "closed": False, "exp_lon": nx * grid.dlon,
                          "mean_lat": 0.0, "geometry": walks})
    w = P.calculate_streamers(data, grid, frame, geo_dis=geo_dis, cont_dis=cont_dis)
    tab = tables["streamers"]
    got = list(zip(tab.job.tolist(), tab.ind1.tolist(), tab.ind2.tolist()))
    want = []
    if len(w):
        bp = w.attrs["_basepoints"]
        want = list(zip(bp["_contour"].tolist(), bp["_ind1"].tolist(), bp["_ind2"].tolist()))
    assert len(want) >= min_events, len(want)
    rings = detect.event_rings(cs, tab)
    unpinned = any((r[:, 0] >= grid.nlon).any() and not G.ring_is_simple(r) for r in rings)
    if got == want and not unpinned:
        empty = pd.DataFrame()
        compare_events(cs, tables, flags, dict(streamers=w, overturnings=empty, cutoffs=empty), grid, [2.0], data)
        return len(want)

    def excused(key, marked):
        jb, a, b = key
        inside = (near[:, 0] == jb) & (near[:, 2] <= b) & (near[:, 3] >= a)
        return marked or bool(inside.any())

    for e, key in enumerate(got):
        if key not in set(want):
            assert excused(key, tab.near[e] != 0), ("device only", key)
    for key in want:
        if key not in set(got):
            assert excused(key, False), ("oracle only", key)
    props = detect.finish_properties(tab, grid.lon, grid.lat, grid.nlon)
    for k, key in enumerate(want):
        if key in set(got):
            e, row = got.index(key), w.iloc[k]
            assert tab.sums[e, 5] == len(w.attrs["_members"][k]), key
            assert props["com"][e] == row.com or props["com_near_integer"][e], key
            assert props["mean_var"][e] == row.mean_var and props["event_area"][e] == row.event_area, key
    return len(want)


SPIKE_CASES = [("3", 30, 3, 7), ("4", 25, 3, 5), ("5", 18, 2, 11)]


@pytest.mark.parametrize("gname,ybase,amp,spike_x", SPIKE_CASES)
def test_spike_and_its_periodic_copy_emu(emu, gname, ybase, amp, spike_x):
    grid = _grid(gname)
    _event_parity(grid, [_spike(grid, ybase, amp, spike_x)], 800.0, 1500.0)


@pytest.mark.gpu
@pytest.mark.parametrize("gname,ybase,amp,spike_x", SPIKE_CASES)
def test_spike_and_its_periodic_copy_gpu(gpu, gname, ybase, amp, spike_x):
    grid = _grid(gname)
    _event_parity(grid, [_spike(grid, ybase, amp, spike_x)], 800.0, 1500.0)


def _pair_through_fold(gname, ybase, amp, spike_x):
    """the base points of the spike contour equal the reference's, among them the tip and its periodic copy, whose
    column gap is exactly nlon (the tile bound once skipped their tile: 3 degrees [(6, 8)] for [(6, 8), (7, 127)],
    4 degrees [] for [(5, 95)])"""
    grid = _grid(gname)
    walk = _spike(grid, ybase, amp, spike_x)
    _, tables, _, _, _ = _run(grid, [walk], 800.0, 1500.0)
    tab = tables["streamers"]
    got = sorted(zip(tab.ind1.tolist(), tab.ind2.tolist()))
    bp = P.streamer_basepoints(walk, grid)
    want = sorted(zip(bp.ind1.tolist(), bp.ind2.tolist()))
    assert got == want
    assert any(b - a == grid.nlon for a, b in want)


@pytest.mark.parametrize("gname,ybase,amp,spike_x", SPIKE_CASES[:2])
def test_tile_bound_keeps_a_pair_one_turn_apart_emu(emu, gname, ybase, amp, spike_x):
    _pair_through_fold(gname, ybase, amp, spike_x)


@pytest.mark.gpu
@pytest.mark.parametrize("gname,ybase,amp,spike_x", SPIKE_CASES[:2])
def test_tile_bound_keeps_a_pair_one_turn_apart_gpu(gpu, gname, ybase, amp, spike_x):
    _pair_through_fold(gname, ybase, amp, spike_x)


# polar contours: rows 84-88 degrees on grids of 2.5 x 2 and 2.8125 degrees, where 180 degrees of longitude are
# a few hundred km and pairs whose column gap folds past 180 degrees lie within geo_dis
POLAR_CASES = [("2.5x2", 0, 800.0), ("2.5x2", 1, 2000.0), ("2.8125", 2, 800.0), ("2.8125", 3, 2000.0)]


def _polar(gname, seed, geo_dis):
    grid = _grid(gname, njobs=2)
    rng = np.random.default_rng(40 + seed)
    W = grid.nlon + int(120 / grid.dlon)
    ylo, yhi = _row(grid, 84.0), _row(grid, 88.0)
    walks = [_band_walk(rng, W, ylo, yhi, _row(grid, 86.0)),
             _spike(grid, _row(grid, 86.0), 1, int(rng.integers(0, grid.nlon)), tip=-3)]
    _event_parity(grid, walks, geo_dis, 1500.0, seed)


@pytest.mark.parametrize("gname,seed,geo_dis", POLAR_CASES)
def test_polar_pairs_folded_past_180_degrees_emu(emu, gname, seed, geo_dis):
    _polar(gname, seed, geo_dis)


@pytest.mark.gpu
@pytest.mark.parametrize("gname,seed,geo_dis", POLAR_CASES)
def test_polar_pairs_folded_past_180_degrees_gpu(gpu, gname, seed, geo_dis):
    _polar(gname, seed, geo_dis)


WALK_CASES = [("2.5x2", 0, 100.0, 500.0), ("2.5x2", 1, 400.0, 1500.0), ("2.5x2", 2, 800.0, 5000.0),
              ("2.5x2", 3, 2000.0, 1500.0), ("2.8125", 4, 100.0, 1500.0), ("2.8125", 5, 400.0, 5000.0),
              ("2.8125", 6, 800.0, 500.0), ("2.8125", 7, 2000.0, 5000.0)]


def _walks(gname, seed, geo_dis, cont_dis):
    grid = _grid(gname, njobs=2)
    rng = np.random.default_rng(60 + seed)
    W = grid.nlon + int(120 / grid.dlon)
    _event_parity(grid, [_random_walk_contour(rng, W, grid.nlat) for _ in range(2)], geo_dis, cont_dis, seed,
                  min_events=0)


@pytest.mark.parametrize("gname,seed,geo_dis,cont_dis", WALK_CASES)
def test_random_walks_across_thresholds_emu(emu, gname, seed, geo_dis, cont_dis):
    _walks(gname, seed, geo_dis, cont_dis)


@pytest.mark.gpu
@pytest.mark.parametrize("gname,seed,geo_dis,cont_dis", WALK_CASES)
def test_random_walks_across_thresholds_gpu(gpu, gname, seed, geo_dis, cont_dis):
    _walks(gname, seed, geo_dis, cont_dis)


# ------------------------------------------------------------------------------------ near threshold on the GPU
@pytest.mark.gpu
@pytest.mark.parametrize("nlat,nlon", [(181, 360), (721, 1440)])
def test_near_threshold_pairs_are_listed_kept_and_rejected_gpu(gpu, nlat, nlon):
    """test_indices.test_near_threshold_pairs_are_listed_kept_and_rejected_emu on the device's arithmetic: a
    threshold 1e-12 above / below the distance of one pair of the synthetic field's full-width contour; the pair is
    listed whether it is kept or rejected"""
    from wavebreaking_b200 import pipeline

    detect.clear_contexts()
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, np.array([6.0]))
    grid = P.Grid(lon, lat, synthetic.time_axis(1, 6))
    base = pipeline.Detector(lat, lon, levels=[2.0]).run_batch(spatial.to_device(raw))
    assert base.near_total == 0 and len(base.near) == 0
    cs = base.contours
    c = int(np.argmax(cs.host()["nx"]))  # the full-width contour
    pts = cs.contour_points(c)
    x = pts[:, 0]
    X = np.radians(np.c_[lat[pts[:, 1]], lon[x % nlon]])
    on = np.r_[0.0, [P.dist.pairwise(X[k - 1:k], X[k:k + 1])[0, 0] * R for k in range(1, len(X))]]
    # rows of the reference's matrices for a sample of first points (cont: the row cumsum, streamer_index.py:135)
    found = None
    for i in np.linspace(0, len(pts) - 2, 40).astype(int):
        geo = P.dist.pairwise(X[i:i + 1], X)[0] * R
        cont = np.r_[np.zeros(i + 1), np.cumsum(on[i + 1:])]
        jj = np.nonzero((np.arange(len(pts)) > i) & (np.abs(x - x[i]) <= 120) & (cont > 2500) & (geo > 300)
                        & (geo < 1200))[0]
        if len(jj):
            j = int(jj[len(jj) // 2])
            found = (int(i), j, float(geo[j]), float(cont[j]))
            break
    assert found is not None
    i, j, gij, cij = found
    for which, value in (("geo_dis", gij), ("cont_dis", cij)):
        for factor in (1 + 1e-12, 1 - 1e-12):
            kw = {which: value * factor}
            if which == "cont_dis":
                kw["geo_dis"] = gij * 1.5
            res = pipeline.Detector(lat, lon, levels=[2.0], **kw).run_batch(spatial.to_device(raw))
            rec = res.near[(res.near[:, 3] == i) & (res.near[:, 4] == j)]
            assert len(rec) == 1, (which, factor, res.near)
            flags = int(rec[0, 5])
            assert flags & (2 if which == "geo_dis" else 4)
            if which == "geo_dis":
                assert bool(flags & 1) == (gij < kw[which])
            else:
                assert bool(flags & 1) == (cij > kw[which])
            assert res.near_total == len(res.near) >= 1
