"""wbk_track_overlap (tracking.overlap_areas): the float64 areas area(A), area(B), area(A n B) behind the by_overlap
ratio, against exact rational areas (oracle.geom._sweep_exact, non-zero winding per ring, any orientation), on
lattice and off-lattice (multi)polygons, under translation, through the linking decision and the public API, and on
the polygons the pipeline builds."""

from fractions import Fraction

import numpy as np
import pytest

from oracle import geom
from test_tracking import _oracle_labels, _rect, _star, soup_of
from wavebreaking_b200 import compat, pipeline, spatial, synthetic, tracking

TOL = 1e-12  # |inter - exact| <= TOL * (A + B): three orders of magnitude inside tracking.NEAR_REL
SHIFTS = [(360, 180), (1430, 700), (4000, 4000)]  # (1430, 700): the east edge of the 0.25 degree grid
OFF_SCALE, OFF_SHIFT = 2 ** 10, 1  # off-lattice: x / 8 (+ 2^-13 on odd polygons) = (1024 x + 0 | 1) / 8192


# ------------------------------------------------------------------ generators
def _is_ring(p):
    return len(p) >= 3 and geom._ring_area2([(int(x), int(y)) for x, y in p]) != 0 and geom.ring_is_simple(p)


def _oriented(rng, ring):
    """the same region, from a random start vertex (a different fan origin), wound either way"""
    ring = np.roll(ring, rng.integers(len(ring)), axis=0)
    return ring[::-1].copy() if rng.random() < 0.5 else ring


def _shape(rng, span=10):
    """a simple non-convex star or a rectangle, oriented at random"""
    while True:
        p = _rect(rng, span - 4) if rng.random() < 0.5 else _star(rng, span)
        if _is_ring(p):
            return _oriented(rng, p)


def _multi(rng, span=10):
    """2-4 parts that do not overlap each other; a new part is often placed against an existing one so that the
    two touch along an edge or at a corner"""
    parts = [_shape(rng, span)]
    k = rng.integers(2, 5)
    while len(parts) < k:
        p, q = _shape(rng, span), parts[rng.integers(len(parts))]
        mode = rng.integers(3)
        if mode == 0:  # on the right-hand side of q: a shared vertical line
            p = p + [q[:, 0].max() - p[:, 0].min(), q[:, 1].min() - p[:, 1].min() + rng.integers(-2, 3)]
        elif mode == 1:  # at the top right corner of q's box
            p = p + [q[:, 0].max() - p[:, 0].min(), q[:, 1].max() - p[:, 1].min()]
        else:
            p = p + rng.integers(0, span, 2)
        if not any(geom.overlap_positive_exact([r], [p]) for r in parts):
            parts.append(p)
    return parts


def _noisy(rng, ring):
    """the same region with collinear vertices (edge midpoints on the lattice) and repeated consecutive vertices"""
    out = []
    for a, b in zip(ring, np.roll(ring, -1, axis=0)):
        out.append(a)
        if rng.random() < 0.3:
            out.append(a)
        if ((b - a) % 2 == 0).all() and (a != b).any() and rng.random() < 0.7:
            out.append((a + b) // 2)
    return np.array(out)


def _comb(rng, teeth, x0=0, y0=0):
    """a comb: base of height hb, teeth of random widths, gaps and heights (4 teeth x 4 vertices + 2)"""
    w = rng.integers(1, 4, teeth)
    g = rng.integers(1, 4, teeth - 1)
    h = rng.integers(1, 120, teeth)
    hb = int(rng.integers(1, 6))
    left = np.r_[0, np.cumsum(w[:-1] + g)]  # left edge of every tooth
    right = left + w
    pts = [(0, 0), (int(right[-1]), 0)]
    for i in range(teeth - 1, -1, -1):
        if i < teeth - 1:
            pts.append((int(right[i]), hb))
        pts += [(int(right[i]), hb + int(h[i])), (int(left[i]), hb + int(h[i]))]
        if i > 0:
            pts.append((int(left[i]), hb))
    return np.array(pts) + [x0, y0]


def _big_star(rng, n, cx=160, cy=160):
    while True:
        ang = np.sort(rng.choice(4096, n, replace=False)) * (2 * np.pi / 4096)
        rad = rng.uniform(60, 150, n)
        p = np.c_[np.rint(cx + rad * np.cos(ang)), np.rint(cy + rad * np.sin(ang))].astype(np.int64)
        if _is_ring(p):
            return p


def _checkerboard(rng, k, s=2, x0=0, y0=0):
    """(k x k + 1) // 2 squares of side s that touch each other at corners, each wound at random"""
    return [_oriented(rng, np.array([[0, 0], [s, 0], [s, s], [0, s]]) + [x0 + s * i, y0 + s * j])
            for i in range(k) for j in range(k) if (i + j) % 2 == 0]


def small_cases(seed, n=48):
    """(polys, pairs): all pairs of n random shapes and multipolygons, plus identical, nested, edge-sharing and
    degenerate pairs; every coordinate in [0, 96)"""
    rng = np.random.default_rng(seed)
    polys, pairs = [], []
    for _ in range(n):
        u = rng.random()
        if u < 0.4:
            polys.append([_shape(rng)])
        elif u < 0.8:
            polys.append(_multi(rng))
        elif u < 0.9:
            polys.append([_noisy(rng, r) for r in _multi(rng)])
        else:  # a two-vertex ring of zero area beside a real part
            p = _shape(rng)
            polys.append([p, np.array([p[0], p[0] + rng.integers(-3, 4, 2)])] if rng.random() < 0.5 else
                         [np.array([[0, 9], [5, 9]]), p])
    pairs += [(i, j) for i in range(n) for j in range(i + 1, n)]
    for _ in range(12):
        i = int(rng.integers(n))
        a = polys[i]
        lo = np.min([r.min(axis=0) for r in a], axis=0) - rng.integers(0, 2, 2)
        hi = np.max([r.max(axis=0) for r in a], axis=0) + rng.integers(0, 2, 2)
        box = np.array([lo, [hi[0], lo[1]], hi, [lo[0], hi[1]]])
        k = len(polys)
        polys += [[_oriented(rng, r) for r in a[::-1]],  # the same region: other start vertices, windings, part order
                  [_oriented(rng, box)],  # a box that contains it
                  [_oriented(rng, box + [hi[0] - lo[0], 0])]]  # the box's right-hand neighbour: one shared edge
        pairs += [(i, k), (k, i), (i, k + 1), (k + 1, i), (k + 1, k + 2)]
    polys = [[r + 16 for r in p] for p in polys]  # room for the placements of _multi
    assert 0 <= min(int(r.min()) for p in polys for r in p) and max(int(r.max()) for p in polys for r in p) < 96
    return polys, np.array(pairs, dtype=np.int32)


def large_cases(seed, count=1):
    """(polys, pairs) with > 256 edges per polygon spanning hundreds of cells, and a checkerboard of > 64 rings"""
    rng = np.random.default_rng(seed)
    polys, pairs = [], []
    for _ in range(count):
        k = len(polys)
        polys += [[_oriented(rng, _comb(rng, 70))], [_oriented(rng, _comb(rng, 70, *rng.integers(0, 40, 2)))],
                  [_oriented(rng, _big_star(rng, 300))],
                  _checkerboard(rng, 14, 2, *rng.integers(60, 140, 2)),
                  _checkerboard(rng, 14, 2, *rng.integers(60, 140, 2))]
        pairs += [(k, k + 1), (k + 1, k), (k, k + 2), (k + 2, k + 1), (k + 3, k + 2), (k + 2, k + 3), (k + 3, k + 4)]
        cb = polys[k + 3]
        polys.append([_oriented(rng, r + [2, 0]) for r in cb])  # the complement's squares: edges touch, no overlap
        pairs.append((k + 3, len(polys) - 1))
    return polys, np.array(pairs, dtype=np.int32)


# ------------------------------------------------------------------ exact reference and checks
def _exact(polys, pairs, scale=1):
    """Fraction (A, B, A n B) per pair; the coordinates are integers times 1 / scale"""
    s2 = scale * scale
    return [tuple(v / s2 for v in geom._sweep_exact(polys[i], polys[j])) for i, j in pairs]


def _check_areas(got, want):
    """area(A), area(B) bit for bit, |inter - exact| <= TOL * (A + B); returns the largest relative error"""
    worst = 0.0
    for k, (a, b, ab) in enumerate(want):
        assert Fraction(got[k, 0]) == a and Fraction(got[k, 1]) == b, (k, got[k], a, b)
        err = float(abs(Fraction(got[k, 2]) - ab) / (a + b))
        assert err <= TOL, (k, got[k], ab)
        worst = max(worst, err)
    return worst


def _shifted(polys, d):
    return [[r + d for r in p] for p in polys]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _off_lattice(polys):
    """integer rings of polygon k -> (1024 x + (k odd)) as integers (exact reference) and / 8192 as floats"""
    ints = [[r * OFF_SCALE + OFF_SHIFT * (k % 2) for r in p] for k, p in enumerate(polys)]
    return ints, [[r / (OFF_SCALE * 8) for r in p] for p in ints]


def _float_soup(polys):
    rings = [r for p in polys for r in p]
    return tracking.PolygonSoup(np.concatenate(rings).astype(np.float64), np.r_[0, np.cumsum([len(r) for r in rings])],
                                np.r_[0, np.cumsum([len(p) for p in polys])], False)


def _check_translated(polys, pairs, shifts):
    base = tracking.overlap_areas(soup_of(polys), pairs)
    for d in shifts:
        assert np.array_equal(_bits(tracking.overlap_areas(soup_of(_shifted(polys, d)), pairs)), _bits(base)), d


# ------------------------------------------------------------------ 1 + 2: areas and translation
def _check_small(seed, n=48):
    polys, pairs = small_cases(seed, n)
    return _check_areas(tracking.overlap_areas(soup_of(polys), pairs), _exact(polys, pairs))


def _check_large(seed, count, shifts):
    polys, pairs = large_cases(seed, count)
    _check_translated(polys, pairs, shifts)
    return _check_areas(tracking.overlap_areas(soup_of(polys), pairs), _exact(polys, pairs))


def test_mixed_orientation_repro_emu(emu):
    """two squares, the second wound clockwise, inside a 6 x 6 square: the parts must not cancel"""
    sq = lambda x, y, s: np.array([[x, y], [x + s, y], [x + s, y + s], [x, y + s]])
    A, B = [sq(0, 0, 2), sq(4, 0, 2)[::-1].copy()], [sq(0, 0, 6)]
    got = tracking.overlap_areas(soup_of([A, B]), [[0, 1], [1, 0]])
    assert got.tolist() == [[8.0, 36.0, 8.0], [36.0, 8.0, 8.0]]


def test_zero_area_ring_encloses_nothing_emu(emu):
    """a two-point ring (a sliver piece of the meridian split) that crosses, touches or lies inside the other polygon
    adds no overlap, in the exact test as in the areas"""
    sq = lambda x, y, s: np.array([[x, y], [x + s, y], [x + s, y + s], [x, y + s]])
    polys = [[sq(20, 20, 4)], [np.array([[18, 22], [26, 22]]), sq(30, 20, 2)], [sq(30, 20, 2), np.array([[21, 21],
             [23, 23]])], [np.array([[24, 21], [24, 23]]), sq(10, 10, 2)[::-1].copy()], [sq(22, 20, 4)]]
    pairs = np.array([(0, 1), (1, 0), (0, 2), (2, 0), (0, 3), (3, 0), (1, 4), (4, 1)], dtype=np.int32)
    want = _exact(polys, pairs)
    assert (tracking.overlap_exact(soup_of(polys), pairs) & 1).tolist() == [int(ab > 0) for _, _, ab in want]
    _check_areas(tracking.overlap_areas(soup_of(polys), pairs), want)


@pytest.mark.parametrize("seed", [0, 1])
def test_areas_match_exact_emu(emu, seed):
    """~1.2 k pairs of random (multi)polygons per seed, every ring wound at random; largest error seen in the
    emulator: 6.8e-16 of A + B"""
    _check_small(seed)


def test_areas_translation_invariant_emu(emu):
    """the same pairs moved by (360, 180), (1430, 700) and (4000, 4000): the same areas bit for bit"""
    polys, pairs = small_cases(2, n=32)
    _check_translated(polys, pairs, SHIFTS)


def test_large_polygons_emu(emu):
    """combs and stars of 280-300 edges spanning 100-300 cells, checkerboards of 98 rings (two chunks of ring areas),
    also moved by (360, 180); largest error seen in the emulator: 1.8e-15 of A + B"""
    _check_large(0, 1, SHIFTS[:1])


# ------------------------------------------------------------------ 3: off-lattice
def _check_off_lattice(seed, large=0):
    polys, pairs = small_cases(seed, n=32)
    if large:
        lp, lpairs = large_cases(seed, large)
        pairs = np.r_[pairs, lpairs + len(polys)]
        polys = polys + lp
    ints, floats = _off_lattice(polys)
    assert not tracking.soup_from_geometries([compat.MultiPolygon(p) for p in floats]).lattice
    got = tracking.overlap_areas(_float_soup(floats), pairs)
    return _check_areas(got, _exact(ints, pairs, OFF_SCALE * 8))


def test_off_lattice_areas_emu(emu):
    """the shapes at x / 8, every other polygon moved by 2^-13 (exact in float64, off any common lattice); largest
    error seen in the emulator: 6.7e-16 of A + B"""
    _check_off_lattice(3)



# ------------------------------------------------------------------ 4: the linking decision
def _lookup(pairs, values):
    """f(p) = the rows of values for the pairs p (decide_pairs asks for subsets of the pairs)"""
    row = {tuple(p): k for k, p in enumerate(pairs.tolist())}
    return lambda p: values[[row[tuple(q)] for q in np.asarray(p).tolist()]]


def _thresholds(rng, ratios):
    inner = [r for r in ratios if 0 < r < 1]
    return [-0.5, 0.0, 0.2, 1.0] + [float(inner[k]) for k in rng.choice(len(inner), 4, replace=False)]


def _check_decisions(pairs, ratios, thresholds, decide, tiny=()):
    """every pair decided unlike its exact ratio is listed as near and lies within 2 NEAR_REL of the threshold; so
    does every listed pair (pairs of `tiny`, whose float path counts a tiny intersection as empty, excepted)"""
    band = 2 * Fraction(tracking.NEAR_REL)
    wrong = 0
    for thr in thresholds:
        links, near = decide(thr)
        got, near = set(map(tuple, links.tolist())), set(map(tuple, near.tolist()))
        for p, r in zip(map(tuple, pairs.tolist()), ratios):
            close = abs(r - Fraction(thr)) <= band or p in tiny
            if (p in got) != (r > Fraction(thr)):
                wrong += 1
                assert p in near and close, (p, thr, r)
            if p in near:
                assert close, (p, thr, r)
    return wrong


def _check_lattice_decisions(seed, n, shifts):
    polys, pairs = small_cases(seed, n)
    want = _exact(polys, pairs)
    ratios = [ab / (a + b - ab) for a, b, ab in want]
    thresholds = _thresholds(np.random.default_rng(seed), ratios)
    for d in [(0, 0)] + shifts:
        soup = soup_of(_shifted(polys, d))
        flags, areas = tracking.overlap_exact(soup, pairs), tracking.overlap_areas(soup, pairs)
        _check_areas(areas, want)
        _check_decisions(pairs, ratios, thresholds, lambda thr: tracking.decide_pairs(
            pairs, "by_overlap", thr, exact=_lookup(pairs, flags), areas=_lookup(pairs, areas)))


def _check_float_decisions(seed, n):
    """soup.lattice == False: link_events on all pairs i < j (float keys 0, 1, ..., window n)"""
    polys, _ = small_cases(seed, n)
    ints, floats = _off_lattice(polys)
    m = len(polys)
    pairs = np.array([(i, j) for i in range(m) for j in range(i + 1, m)], dtype=np.int32)
    want = _exact(ints, pairs, OFF_SCALE * 8)
    ratios = [ab / (a + b - ab) for a, b, ab in want]
    # the float path counts an intersection below 1e-12 (A + B) as empty and lists those up to 1e-11 (A + B) as near
    tiny = {p for p, (a, b, ab) in zip(map(tuple, pairs.tolist()), want) if ab <= Fraction(1, 10 ** 11) * (a + b)}
    soup = _float_soup(floats)
    keys = np.arange(m, dtype=np.float64)
    decide = lambda thr: tracking.link_events(keys, float(m), "by_overlap", soup, overlap=thr)[::2]
    _check_decisions(pairs, ratios, [-0.5, 0.0, 0.2, 1.0], decide, tiny)


def test_decisions_emu(emu):
    """decide_pairs at -0.5, 0, 0.2, 1.0 and four exact ratios of the pairs (rounded to float64), also moved by
    (1430, 700) and (4000, 4000); identical regions (ratio exactly 1) at 1.0"""
    _check_lattice_decisions(4, 32, SHIFTS[1:])


def test_float_decisions_emu(emu):
    _check_float_decisions(5, 12)


# ------------------------------------------------------------------ 5: labels through the public API
def _frame_case(seed, nsteps=6, per_step=5):
    rng = np.random.default_rng(seed)
    polys = [[r + 16 for r in (_multi(rng) if rng.random() < 0.6 else [_shape(rng)])] for _ in range(nsteps * per_step)]
    t0 = np.datetime64("2000-01-01T00", "ns")
    dates = np.array([t0 + (k // per_step) * np.timedelta64(1, "h") for k in range(len(polys))])
    return dates, polys


def _check_labels(dates, polys, overlaps=(0, 0.2, 0.5)):
    import wavebreaking_b200 as wb

    com = np.zeros((len(polys), 2))
    ints, floats = _off_lattice(polys)
    lattice = [compat.MultiPolygon([r * 0.25 - 30.0 for r in p]) for p in polys]  # lon / lat on a 0.25 degree grid
    for geoms, lat in ((lattice, True), ([compat.MultiPolygon(p) for p in floats], False)):
        assert tracking.soup_from_geometries(geoms).lattice == lat
        ev = compat.make_frame({"date": list(dates), "com": list(map(tuple, com))}, geoms)
        for o in overlaps:
            got = wb.track_events(ev, overlap=o)
            want = _oracle_labels(dates, polys if lat else ints, com, method="by_overlap", overlap=o)
            assert np.array_equal(got.label.sort_index().values, want), (lat, o)


def test_track_events_mixed_orientation_emu(emu):
    """MultiPolygon(two squares, one wound clockwise) and the 6 x 6 square an hour later: ratio 8 / 36"""
    sq = lambda x, y, s: np.array([[x, y], [x + s, y], [x + s, y + s], [x, y + s]])
    dates = np.array([np.datetime64("2000-01-01T00", "ns"), np.datetime64("2000-01-01T01", "ns")])
    polys = [[sq(16, 16, 2), sq(20, 16, 2)[::-1].copy()], [sq(16, 16, 6)]]
    _check_labels(dates, polys, (0, 0.2, 0.25))
    assert _oracle_labels(dates, polys, np.zeros((2, 2)), overlap=0.2).tolist() == [0, 0]
    _check_labels(*_frame_case(6))


# ------------------------------------------------------------------ 6: the pipeline's polygons
def _check_pipeline(nlat, nlon, hours, levels, max_pairs, rng):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    det = pipeline.Detector(lat, lon, levels=list(levels), want_pieces=True)
    raw = synthetic.pv_field(nlat, nlon, np.asarray(hours, dtype=np.float64))
    res = det.run_batch(spatial.to_device(raw))
    soup, _ = pipeline.events_soup(res, "streamers", det)
    # every event's rings (the meridian pieces of a split event) share one orientation
    _, vsign = tracking._edge_table(soup)
    live = np.diff(soup.ring_off) > 0
    ring_sign = np.zeros(len(live), dtype=np.int32)
    ring_sign[live] = vsign[soup.ring_off[:-1][live]]
    nsplit = 0
    for e in range(len(soup)):
        s = ring_sign[soup.poly_off[e]:soup.poly_off[e + 1]]
        assert len(set(s[s != 0].tolist())) <= 1, e
        nsplit += int(len(s) > 1)
    # the pairs whose boxes intersect (the candidates of tracking), against the exact areas
    box = soup.bounds()
    i, j = np.nonzero(np.triu((box[:, None, 0] <= box[None, :, 2]) & (box[None, :, 0] <= box[:, None, 2]) &
                              (box[:, None, 1] <= box[None, :, 3]) & (box[None, :, 1] <= box[:, None, 3]), 1))
    pairs = np.c_[i, j].astype(np.int32)
    if len(pairs) > max_pairs:
        nv = np.diff(soup.ring_off[soup.poly_off])
        size = nv[pairs[:, 0]] + nv[pairs[:, 1]]
        big = np.argsort(-size, kind="stable")[:max_pairs // 4]  # the largest pairs, and a random sample of the rest
        rest = rng.choice(np.setdiff1d(np.arange(len(pairs)), big), max_pairs - len(big), replace=False)
        pairs = pairs[np.r_[big, rest]]
    polys = [[soup.xy[soup.ring_off[r]:soup.ring_off[r + 1]].astype(np.int64) for r in
              range(soup.poly_off[e], soup.poly_off[e + 1])] for e in range(len(soup))]
    worst = _check_areas(tracking.overlap_areas(soup, pairs), _exact(polys, pairs))
    return nsplit, len(pairs), worst


def test_pipeline_polygons_emu(emu):
    """streamers of a 61 x 120 grid across the last meridian (split into pieces); largest error seen in the
    emulator: 1.4e-15 of A + B"""
    nsplit, npairs, _ = _check_pipeline(61, 120, 288.0 + np.arange(4), (2.0, -2.0), 400, np.random.default_rng(0))
    assert nsplit > 0 and npairs > 50


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_areas_match_exact_gpu(gpu):
    """seeds 0-5 (9.6 k pairs), then the translations; largest error seen on a B200: 9.8e-16 of A + B"""
    worst = max(_check_small(seed, 56) for seed in range(6))
    polys, pairs = small_cases(6, 32)
    _check_translated(polys, pairs, SHIFTS)
    print("small pairs: largest error", worst)


@pytest.mark.gpu
def test_large_polygons_gpu(gpu):
    """three sets of combs, stars and checkerboards, moved by every shift; largest error seen on a B200: 5.7e-15 of
    A + B"""
    print("large pairs: largest error", _check_large(1, 3, SHIFTS))


@pytest.mark.gpu
def test_off_lattice_areas_gpu(gpu):
    """small and large shapes off the lattice; largest error seen on a B200: 5.5e-15 of A + B"""
    print("off-lattice: largest error", max(_check_off_lattice(seed, 2) for seed in (7, 8)))


@pytest.mark.gpu
def test_decisions_gpu(gpu):
    for seed in (9, 10):
        _check_lattice_decisions(seed, 48, SHIFTS)
    _check_float_decisions(11, 32)


@pytest.mark.gpu
def test_track_events_mixed_orientation_gpu(gpu):
    for seed in (12, 13):
        _check_labels(*_frame_case(seed, nsteps=10, per_step=8))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(181, 360), (721, 1440)])
def test_pipeline_polygons_gpu(gpu, shape):
    """the largest candidate pairs of streamers and a sample of the rest; largest error seen on a B200: 8.3e-15 of
    A + B (721 x 1440)"""
    nlat, nlon = shape
    nsplit, npairs, worst = _check_pipeline(nlat, nlon, 500.0 + np.arange(3), (2.0,), 120, np.random.default_rng(1))
    print(shape, "pipeline pairs", npairs, "largest error", worst)
    assert npairs > 50
