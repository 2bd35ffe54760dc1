"""Arena regrowth in Detector.stream: every slot-owned arena and the context arenas forced to overflow, one at a time
and all at once, give the results of an unforced run, and a climatology and a tracker still count each batch once."""

import numpy as np
import pytest

from wavebreaking_b200 import detect, pipeline, spatial, synthetic

NLAT, NLON, NT, T = 61, 120, 5, 2  # batches of 2, 2 and 1 steps
HOUR0 = 288.0  # at 61 x 120 the synthetic record has events across the last meridian: the clipper's pieces
LEVELS = [2.0, -2.0]
TINY = dict(seg_cap=64, contour_cap=4, sel_cap=1, pair_cap=16, event_cap=1)  # context arenas (detect.default_caps)


def _record():
    lat, lon = synthetic.grid_coords(NLAT, NLON)
    raw = synthetic.pv_field(NLAT, NLON, HOUR0 + np.arange(NT))
    return lat, lon, raw, synthetic.time_axis(NT, 1)


def _shrink_context(monkeypatch, keys):
    orig = detect.default_caps
    monkeypatch.setattr(detect, "default_caps", lambda *a: {**orig(*a), **{k: TINY[k] for k in keys}})


def _run(det, raw, depth, small=(), **kw):
    """Stream raw after setting the slot capacities ``small`` to 1 on the slots of the full batches; returns per batch
    the summary, the event tables, the flag grids and the pieces."""
    for idx in range(depth):
        for k in small:
            setattr(det._slot(T, idx), k, 1)  # the buffers stay larger: only the kernels' bounds see the capacity
    out = []
    batches = [spatial.to_device(raw[t:t + T]) for t in range(0, len(raw), T)]
    for res in det.stream(batches, depth=depth, **kw):
        out.append((pipeline.summarize(res), res.tables, res.flags[:, :res.ntime].cpu().numpy().copy(), res.pieces))
    return out


def _same(got, want):
    assert len(got) == len(want)
    for (s, tabs, flags, pieces), (s0, tabs0, flags0, pieces0) in zip(got, want):
        assert s == s0
        assert np.array_equal(flags, flags0)
        for kind in detect.KINDS:
            a, b = tabs[kind], tabs0[kind]
            for col in ("job", "contour", "ind1", "ind2", "box", "orientation", "split", "near", "sums"):
                assert np.array_equal(getattr(a, col), getattr(b, col)), (kind, col)
            if b.rings is not None:
                assert np.array_equal(a.rings.off, b.rings.off) and np.array_equal(a.rings.packed, b.rings.packed)
        assert (pieces is None) == (pieces0 is None)
        if pieces0 is not None:
            assert all(np.array_equal(pieces[k], pieces0[k]) for k in ("ev", "off", "xy", "overflow"))


_REF = {}


def _reference(depth):
    if depth not in _REF:
        lat, lon, raw, _ = _record()
        _REF[depth] = _run(pipeline.Detector(lat, lon, levels=LEVELS, want_pieces=True), raw, depth)
    return _REF[depth]


# ------------------------------------------------------------------------------------------- one arena at a time
@pytest.mark.parametrize("small,grown", [("cap_c", "cap_c"), ("cap_p", "cap_c"), ("cap_e", "cap_e"),
                                         ("cap_r", "cap_r"), ("cap_sr", "cap_sr"), ("cap_sv", "cap_sv")])
def test_slot_arena_regrowth_emu(emu, small, grown):
    """``grown``: the key the overflow writes to ``_grow``; a pack overflow grows cap_c and cap_p together"""
    lat, lon, raw, _ = _record()
    det = pipeline.Detector(lat, lon, levels=LEVELS, want_pieces=True)
    got = _run(det, raw, 2, small=(small,))
    assert grown in det._grow and small in det._grow
    _same(got, _reference(2))


@pytest.mark.parametrize("arena", ["contour_cap", "event_cap", "pair_cap", "seg_cap"])  # (one selection slot suffices)
def test_context_arena_regrowth_emu(emu, monkeypatch, arena):
    _shrink_context(monkeypatch, [arena])
    lat, lon, raw, _ = _record()
    det = pipeline.Detector(lat, lon, levels=LEVELS, want_pieces=True)
    got = _run(det, raw, 2)
    assert arena in det._grow
    _same(got, _reference(2))


# ------------------------------------------------------------------------------------------- everything at once
def _counted(det, raw, depth, **kw):
    dates = _record()[3]
    clim = pipeline.FlagClimatology(det, pipeline.groups_from_dates(dates, "month"), ngroups=12)
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=2)
    out = _run(det, raw, depth, climatology=clim, trackers=[tr], **kw)
    return out, clim, tr


@pytest.mark.parametrize("depth", [1, 3])
def test_everything_overflows_counted_once_emu(emu, monkeypatch, depth):
    lat, lon, raw, _ = _record()
    want, clim0, tr0 = _counted(pipeline.Detector(lat, lon, levels=LEVELS, want_pieces=True), raw, depth)
    _shrink_context(monkeypatch, ["event_cap", "pair_cap"])
    det = pipeline.Detector(lat, lon, levels=LEVELS, want_pieces=True)
    got, clim, tr = _counted(det, raw, depth, small=("cap_e",))
    assert {"event_cap", "pair_cap", "cap_e", "cap_r"} <= set(det._grow)  # (one status: index and fetch overflow)
    _same(got, want)
    assert clim.steps.sum() == NT and np.array_equal(clim.steps, clim0.steps)
    assert np.array_equal(clim.counts(), clim0.counts()) and clim.counts().any()
    assert tr.cursor == NT and tr.n_events == tr0.n_events > 0 and len(tr.host_ms) == len(got)
    assert np.array_equal(tr.labels(), tr0.labels())
    assert np.array_equal(tr.near, tr0.near)
