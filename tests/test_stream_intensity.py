"""Event intensity in streamed, file and sharded detection: intensity items (a field, or u and v whose momentum flux is
computed on the device) in Detector.stream, io.detect_file and sharding.run_sharded, against detect.run_indices, the
drop-in path's momentum flux and the oracle."""

import os
import socket
import sys

import numpy as np
import pytest
import torch

from oracle import pipeline as P
from wavebreaking_b200 import detect, pipeline, sharding, spatial, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVELS = [1.5, 2.0, 3.0]  # the multi-level configuration with intensity (BASELINE.md C25-L)


def _record(nlat, nlon, ntime, hour0=0.0):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, hour0 + np.arange(ntime) * 6.0)
    return lat, lon, raw


def _noise(shape, dtype, seed, nan=False):
    a = np.random.default_rng(seed).standard_normal(shape).astype(dtype)
    if nan:  # the zonal means of the momentum flux skip NaNs (numpy.nanmean)
        a[:, 3, 5] = np.nan
        a[-1, 7, :] = np.nan
    return a


def _wind(nlat, nlon, ntime, dtype=np.float32):
    """u and v as the measurement plan makes them: synthetic PV fields of two other seeds"""
    hours = np.arange(ntime) * 6.0
    u = synthetic.pv_field(nlat, nlon, hours, seed=synthetic.SEED + 1, dtype=dtype)
    v = synthetic.pv_field(nlat, nlon, hours, seed=synthetic.SEED + 2, dtype=dtype)
    return u, v


def _slices(a, T):
    return [spatial.to_device(np.ascontiguousarray(a[t:t + T])) for t in range(0, len(a), T)]


def _stream(det, raw, T, items=None, depth=2, **kw):
    """Stream raw in batches of T steps (the last one partial); returns the results and per kind the concatenated
    sums."""
    res = list(det.stream(_slices(raw, T), depth=depth, intensity=items, **kw))
    sums = {k: np.concatenate([r.tables[k].sums for r in res]) for k in detect.KINDS}
    return res, sums


def _items(inten, T):
    return _slices(inten, T)


def _uv_items(u, v, T):
    return list(zip(_slices(u, T), _slices(v, T)))


def _props(det, res, kind):
    tab = [r.tables[kind] for r in res]
    return np.concatenate([detect.finish_properties(t, det.lon, det.lat, det.nlon)["intensity"] for t in tab])


def _same_tables(a, b, with_intensity=True):
    for ra, rb in zip(a, b):
        for kind in detect.KINDS:
            ta, tb = ra.tables[kind], rb.tables[kind]
            assert np.array_equal(ta.job, tb.job) and np.array_equal(ta.box, tb.box), kind
            assert np.array_equal(ta.ind1, tb.ind1) and np.array_equal(ta.ind2, tb.ind2), kind
            cols = slice(None) if with_intensity else [0, 1, 3, 4, 5]
            assert np.array_equal(ta.sums[:, cols], tb.sums[:, cols]), kind


# ------------------------------------------------------------------------------------------- stream vs drop-in
@pytest.mark.parametrize("depth", [1, 3])
@pytest.mark.parametrize("idtype", [np.float32, np.float64])
def test_stream_intensity_matches_run_indices_and_oracle_emu(emu, depth, idtype):
    """three levels, batches of 2 steps with a partial last one, float32 input"""
    nlat, nlon, ntime, T = 91, 180, 3, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    inten = _noise(raw.shape, idtype, seed=3)
    det = pipeline.Detector(lat, lon, levels=LEVELS)
    # the reference's exp_lon.max() over the whole record
    gmax = detect.contours(spatial.smooth(raw, 5), LEVELS, det.add).max_nx
    res, sums = _stream(det, raw, T, _items(inten, T), depth=depth, gmax_nx=gmax)
    assert sum(len(s) for s in sums.values()) > 0
    # the drop-in path on the same steps: detect.run_indices with the intensity converted to the smoothed field's dtype
    for b, r in enumerate(res):
        t0 = b * T
        sm = spatial.smooth(raw[t0:t0 + r.ntime], 5)
        cs = detect.contours(sm, LEVELS, det.add)
        tables, _ = detect.run_indices(cs, sm, det.coords, det.dlon, det.dlat, want_flags=True, gmax_nx=gmax,
                                       intensity=spatial.to_device(np.ascontiguousarray(inten[t0:t0 + r.ntime])))
        for kind in detect.KINDS:
            assert np.array_equal(r.tables[kind].sums, tables[kind].sums), (b, kind)
    # the oracle, event by event
    want = P.detect_steps(raw, P.Grid(lon, lat, synthetic.time_axis(ntime, 6)), levels=LEVELS, intensity=inten)
    for kind in detect.KINDS:
        assert len(sums[kind]) == len(want["events"][kind]), kind
        if len(sums[kind]):
            assert np.array_equal(_props(det, res, kind), want["events"][kind].intensity.values), kind
            assert (sums[kind][:, 2] != 0).all()
    # without intensity: the same tables and flags, and 0 intensity sums (the reference's "0 if None")
    det0 = pipeline.Detector(lat, lon, levels=LEVELS)
    flags0 = []
    for r0, r in zip(det0.stream(_slices(raw, T), depth=depth, gmax_nx=gmax), res):
        _same_tables([r0], [r], with_intensity=False)
        assert all((r0.tables[k].sums[:, 2] == 0).all() for k in detect.KINDS)
        flags0.append(r0.flags[:, :r0.ntime].numpy().copy())
    want_flags = np.stack([want["flags"][k] for k in detect.KINDS])
    assert np.array_equal(np.concatenate(flags0, axis=1), want_flags)


def test_uv_items_equal_momentum_flux_items_emu(emu):
    nlat, nlon, ntime, T = 46, 90, 5, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    for dtype in (np.float32, np.float64):
        u, v = _noise(raw.shape, dtype, 4, nan=True), _noise(raw.shape, dtype, 5, nan=True)
        mf = spatial.momentum_flux(u, v).numpy()
        assert mf.dtype == dtype
        det = pipeline.Detector(lat, lon, levels=LEVELS)
        got, gs = _stream(det, raw, T, _uv_items(u, v, T))
        want, _ = _stream(det, raw, T, _items(mf, T))
        _same_tables(got, want)
        assert sum(len(s) for s in gs.values()) > 0


@pytest.mark.parametrize("flip_lat,flip_lon", [(True, False), (False, True), (True, True)])
def test_descending_storage_emu(emu, flip_lat, flip_lon):
    """input and intensity stored with descending latitudes and / or longitudes give the ascending run's tables"""
    nlat, nlon, ntime, T = 46, 90, 5, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    inten = _noise(raw.shape, np.float32, 6)
    u, v = _wind(nlat, nlon, ntime)

    def stored(a):
        return np.ascontiguousarray(a[:, ::-1 if flip_lat else 1, ::-1 if flip_lon else 1])

    lat_s, lon_s = (lat[::-1] if flip_lat else lat), (lon[::-1] if flip_lon else lon)
    asc, _ = _stream(pipeline.Detector(lat, lon, levels=LEVELS), raw, T, _items(inten, T))
    det_s = pipeline.Detector(lat_s, lon_s, levels=LEVELS)
    desc, sums = _stream(det_s, stored(raw), T, _items(stored(inten), T))
    _same_tables(desc, asc)
    assert sum(len(s) for s in sums.values()) > 0
    # (u, v) as stored: the zonal means are summed in the stored order, as numpy does on the stored arrays
    mf = spatial.momentum_flux(stored(u), stored(v)).numpy()
    got, _ = _stream(det_s, stored(raw), T, _uv_items(stored(u), stored(v), T))
    want, _ = _stream(det_s, stored(raw), T, _items(mf, T))
    _same_tables(got, want)
    if not flip_lon:  # the zonal sums see the same order as in the ascending run
        want_asc, _ = _stream(pipeline.Detector(lat, lon, levels=LEVELS), raw, T, _uv_items(u, v, T))
        _same_tables(got, want_asc)


# ------------------------------------------------------------------------------------------- re-runs
def _tracked(det, raw, T, items, depth=2):
    dates = synthetic.time_axis(len(raw), 6)
    clim = pipeline.FlagClimatology(det, np.zeros(len(raw), dtype=np.int32))
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=6)
    res, sums = _stream(det, raw, T, items, depth=depth, climatology=clim, trackers=[tr])
    return res, sums, clim, tr


def test_regrowth_with_intensity_emu(emu, monkeypatch):
    nlat, nlon, ntime, T = 46, 90, 5, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, v = _wind(nlat, nlon, ntime)
    res, sums, clim, tr = _tracked(pipeline.Detector(lat, lon, levels=LEVELS, want_pieces=True), raw, T,
                                   _uv_items(u, v, T))
    tiny = dict(max_jobs=4, seg_cap=64, contour_cap=4, sel_cap=1, pair_cap=16, event_cap=1)
    monkeypatch.setattr(detect, "default_caps", lambda nlat, nlon, add, njobs: dict(tiny, max_jobs=int(njobs)))
    det = pipeline.Detector(lat, lon, levels=LEVELS, want_pieces=True)
    res2, sums2, clim2, tr2 = _tracked(det, raw, T, _uv_items(u, v, T))
    assert det._grow
    _same_tables(res2, res)
    assert clim2.steps.tolist() == [ntime] and np.array_equal(clim2.counts(), clim.counts())
    assert tr2.cursor == ntime and tr2.n_events == tr.n_events == len(sums["streamers"])
    assert np.array_equal(tr2.labels(), tr.labels())


def test_pieces_rerun_with_intensity_emu(emu):
    nlat, nlon, ntime, T = 61, 120, 4, 2
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, 288.0 + np.arange(ntime))  # events across the last meridian: pieces
    inten = _noise(raw.shape, np.float64, 7)
    levels = [2.0, -2.0]
    res, sums, clim, tr = _tracked(pipeline.Detector(lat, lon, levels=levels, want_pieces=True), raw, T,
                                   _items(inten, T))
    det = pipeline.Detector(lat, lon, levels=levels, want_pieces=True)
    for idx in range(2):
        det._slot(T, idx).cap_sr = 1  # the buffers are larger: only the check sees the small capacity
    res2, sums2, clim2, tr2 = _tracked(det, raw, T, _items(inten, T))
    assert "cap_sr" in det._grow
    _same_tables(res2, res)
    assert clim2.steps.tolist() == [ntime] and np.array_equal(clim2.counts(), clim.counts())
    assert tr2.cursor == ntime and tr2.n_events == tr.n_events
    assert np.array_equal(tr2.labels(), tr.labels())


# ------------------------------------------------------------------------------------------- detect_file
def test_detect_file_intensity_emu(emu, tmp_path):
    from wavebreaking_b200 import io

    nlat, nlon, ntime, T = 46, 90, 5, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    inten = _noise(raw.shape, np.float32, 8)
    u, v = _wind(nlat, nlon, ntime)
    for name, a in (("pv", raw), ("inten", inten), ("u", u), ("v", v)):
        np.save(str(tmp_path / (name + ".npy")), a)
    path = str(tmp_path / "pv.npy")
    det = pipeline.Detector(lat, lon, levels=LEVELS)
    for spec, items in ((str(tmp_path / "inten.npy"), _items(inten, T)),
                        ((str(tmp_path / "u.npy"), str(tmp_path / "v.npy")), _uv_items(u, v, T))):
        want, _ = _stream(det, raw, T, items)
        got = [r for _, r in io.detect_file(path, lat, lon, batch=T, depth=2, levels=LEVELS, intensity=spec)]
        assert len(got) == len(want)
        _same_tables(got, want)
    np.save(str(tmp_path / "short.npy"), inten[:3])
    with pytest.raises(ValueError, match="shape"):
        next(io.detect_file(path, lat, lon, batch=T, levels=LEVELS, intensity=str(tmp_path / "short.npy")))


# ------------------------------------------------------------------------------------------- refusals
def test_refusals_emu(emu):
    nlat, nlon, ntime, T = 46, 90, 4, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    det = pipeline.Detector(lat, lon, levels=[2.0])
    f = _items(_noise(raw.shape, np.float32, 9), T)
    d = _items(_noise(raw.shape, np.float64, 9), T)
    bad = [
        ([f[0][:1]] + f[1:], "shape"),                                   # an item shaped unlike its batch
        ([(f[0], f[0][:, :, :-1])] + f[1:], "u and v differ"),           # u and v of different shapes
        ([(f[0], d[0])] + f[1:], "u and v differ"),                      # u and v of different dtypes
        ([f[0].to(torch.int16)] + f[1:], "int16"),                       # packed u / v are out of scope
        ([(f[0].to(torch.int16), f[0].to(torch.int16))] + f[1:], "int16"),
        ([f[0].to(torch.float16)] + f[1:], "float32 or float64"),
        ([(f[0], f[0], f[0])] + f[1:], "pair"),
    ]
    for items, match in bad:
        with pytest.raises(ValueError, match=match):
            list(det.stream(_slices(raw, T), intensity=items))
    assert not det._slots  # refused before any device work on the batch
    # the intensity ends before the batches: the batches before it are run (and counted) once, the last one is not
    clim = pipeline.FlagClimatology(det, np.zeros(ntime, dtype=np.int32))
    with pytest.raises(ValueError, match="ended before the batches"):
        list(det.stream(_slices(raw, T), depth=1, intensity=f[:1], climatology=clim))
    assert clim.steps.tolist() == [T]
    # submit / run_batch take the same item form and refuse the same way
    with pytest.raises(ValueError, match="shape"):
        det.run_batch(spatial.to_device(raw), intensity=(f[0],))


# ------------------------------------------------------------------------------------------- sharded runs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


NT_SHARD = 7


def _shard_inputs():
    lat, lon, raw = _record(46, 90, NT_SHARD)
    u, v = _wind(46, 90, NT_SHARD)
    return lat, lon, raw, u, v


def _shard_worker(rank, world, port, emu_path, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    from wavebreaking_b200 import _lib, pipeline, sharding, spatial

    _lib.use_library(emu_path, "cpu")
    lat, lon, raw, u, v = _shard_inputs()
    t0, t1 = sharding.shard_range(NT_SHARD, rank, world)
    det = pipeline.Detector(lat, lon, levels=LEVELS)
    res = list(det.stream(_slices(raw[t0:t1], 2), depth=2, intensity=_uv_items(u[t0:t1], v[t0:t1], 2)))
    _, _, one = sharding.run_sharded(det, spatial.to_device(raw), intensity=(spatial.to_device(u),
                                                                             spatial.to_device(v)))
    np.savez(os.path.join(out_dir, "rank_{}.npz".format(rank)),
             **{"stream_" + k: _props(det, res, k) for k in detect.KINDS},
             **{"sharded_" + k: _props(det, [one], k) for k in detect.KINDS})
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_intensity_gloo(emu, emu_lib, tmp_path):
    """the intensity column of the two ranks' events, concatenated, equals the single-process run's"""
    import torch.multiprocessing as mp

    mp.spawn(_shard_worker, args=(2, _free_port(), emu_lib, str(tmp_path)), nprocs=2, join=True)
    lat, lon, raw, u, v = _shard_inputs()
    det = pipeline.Detector(lat, lon, levels=LEVELS)
    ranks = [np.load(tmp_path / "rank_{}.npz".format(r)) for r in range(2)]
    # the stream over the whole record takes the same batches of 2 steps as the two shards (4 + 3 steps)
    streamed = list(det.stream(_slices(raw, 2), depth=2, intensity=_uv_items(u, v, 2)))
    whole = det.run_batch(spatial.to_device(raw), intensity=(spatial.to_device(u), spatial.to_device(v)))
    n = 0
    for kind in detect.KINDS:
        got = np.concatenate([z["stream_" + kind] for z in ranks])
        assert np.array_equal(got, _props(det, streamed, kind)), kind
        got = np.concatenate([z["sharded_" + kind] for z in ranks])
        assert np.array_equal(got, _props(det, [whole], kind)), kind
        n += len(got)
    assert n > 0
    # one process: run_sharded slices the intensity like the field
    _, _, one = sharding.run_sharded(det, spatial.to_device(raw), intensity=spatial.to_device(u))
    _same_tables([one], [det.run_batch(spatial.to_device(raw), intensity=(spatial.to_device(u),))])


# ------------------------------------------------------------------------------------------- GPU
def _graph_case(nlat, nlon, T, shared, uv):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    slabs = [spatial.synth_pv(T, nlat, nlon, hour0=500.0 + T * b, hour_step=1.0) for b in range(2)]
    tail = spatial.synth_pv(T - 3, nlat, nlon, hour0=500.0 + 2 * T, hour_step=1.0)

    def wind(n, b):
        return tuple(spatial.synth_pv(n, nlat, nlon, hour0=500.0 + T * b, hour_step=1.0, seed=synthetic.SEED + k)
                     for k in (1, 2))

    if uv:
        islabs, itail = [wind(T, b) for b in range(2)], wind(T - 3, 2)
    else:
        islabs = [spatial.synth_pv(T, nlat, nlon, hour0=900.0 + T * b, dtype=torch.float64) for b in range(2)]
        itail = spatial.synth_pv(T - 3, nlat, nlon, hour0=900.0 + 2 * T, dtype=torch.float64)
    batches = [slabs[i % 2] for i in range(6)] + [tail]  # every slot sees its buffers 3 times: eager, capture, replay
    items = [islabs[i % 2] for i in range(6)] + [itail]
    det = pipeline.Detector(lat, lon, levels=LEVELS, graphs=True)
    got = list(det.stream(batches, depth=2, shared_stream=shared, intensity=items))
    assert det.graph_replays >= 4
    eager = pipeline.Detector(lat, lon, levels=LEVELS)
    want = list(eager.stream(batches, depth=2, intensity=items))
    assert eager.graph_replays == 0
    _same_tables(got, want)
    assert any(len(r.tables[k]) for r in got for k in detect.KINDS)
    # detect.run_indices on one replayed batch (the drop-in path reads the same field)
    b = 4
    field = items[b] if not uv else spatial.momentum_flux(*items[b])
    sm = spatial.smooth(batches[b], 5)
    tables, _ = detect.run_indices(detect.contours(sm, LEVELS, det.add), sm, det.coords, det.dlon, det.dlat,
                                   intensity=field, gmax_nx=det.nlon + det.add, want_flags=True)
    for kind in detect.KINDS:
        assert np.array_equal(got[b].tables[kind].sums, tables[kind].sums), kind


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(181, 360), (721, 1440)])
@pytest.mark.parametrize("shared", [False, True])
def test_stream_intensity_graphs_gpu(gpu, shape, shared):
    _graph_case(shape[0], shape[1], 8, shared, uv=shared)


@pytest.mark.gpu
def test_pinned_host_uv_gpu(gpu):
    """pinned-host float32 (u, v) at 721 x 1440 with CUDA graphs equals device-resident items"""
    nlat, nlon, T = 721, 1440, 6
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = [spatial.synth_pv(T, nlat, nlon, hour0=300.0 + T * b) for b in range(2)]
    uv = [tuple(spatial.synth_pv(T, nlat, nlon, hour0=300.0 + T * b, seed=synthetic.SEED + k) for k in (1, 2))
          for b in range(2)]
    pin = [r.cpu().pin_memory() for r in raw]
    pin_uv = [tuple(x.cpu().pin_memory() for x in p) for p in uv]
    det = pipeline.Detector(lat, lon, levels=LEVELS, graphs=True)
    got = list(det.stream([pin[i % 2] for i in range(6)], depth=2, intensity=[pin_uv[i % 2] for i in range(6)]))
    assert det.graph_replays >= 2
    want = list(pipeline.Detector(lat, lon, levels=LEVELS).stream([raw[i % 2] for i in range(6)], depth=2,
                                                                 intensity=[uv[i % 2] for i in range(6)]))
    _same_tables(got, want)
    assert any((r.tables[k].sums[:, 2] != 0).any() for r in got for k in detect.KINDS)


@pytest.mark.gpu
def test_three_levels_oracle_gpu(gpu):
    nlat, nlon, ntime, T = 91, 180, 4, 3
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, v = _wind(nlat, nlon, ntime)
    det = pipeline.Detector(lat, lon, levels=LEVELS)
    res, sums = _stream(det, raw, T, _uv_items(u, v, T))
    mf = spatial.momentum_flux(u, v).cpu().numpy()
    want = P.detect_steps(raw, P.Grid(lon, lat, synthetic.time_axis(ntime, 6)), levels=LEVELS, intensity=mf)
    for kind in detect.KINDS:
        assert len(sums[kind]) == len(want["events"][kind]), kind
        if len(sums[kind]):
            assert np.array_equal(_props(det, res, kind), want["events"][kind].intensity.values), kind
