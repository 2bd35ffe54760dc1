"""CF-packed int16 intensity and (u, v) in streamed, file and sharded detection, decoded on the device: wbk_mflux on
packed u and v, the rasteriser's int16 intensity, Detector(intensity_packing=...), io.detect_file and
sharding.run_sharded, against host-decoded float64 inputs and the oracle."""

import ctypes
import os
import socket
import sys

import numpy as np
import pytest
import torch

from oracle import pipeline as P
from wavebreaking_b200 import _lib, detect, pipeline, sharding, spatial, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVELS = [1.5, 2.0, 3.0]
# ERA5 packs every variable with its own scale_factor / add_offset; -32767 is its _FillValue
PK_U = (3.1e-4, 0.25, -32767)
PK_V = (4.7e-4, -0.5, 32767)
PK_F = (2.3e-4, 0.125, -32767)
PK_PV = (2.0e-4, 0.1, None)


def _pack(x, pk, fill_every=0):
    """np.round((x - offset) / scale) as int16; every fill_every-th cell (flat order) set to the fill value"""
    scale, offset, fill = pk
    s = np.round((np.asarray(x, dtype=np.float64) - offset) / scale)
    s = np.clip(s, -32766, 32766).astype(np.int16)
    if fill_every:
        s.reshape(-1)[7::fill_every] = fill
    return s


def _decode(s, pk):
    """what xarray makes of a packed variable: float64(s) * scale_factor + add_offset, the fill value -> NaN"""
    scale, offset, fill = pk
    x = s.astype(np.float64) * scale + offset
    if fill is not None:
        x[s == fill] = np.nan
    return x


def _record(nlat, nlon, ntime):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    return lat, lon, synthetic.pv_field(nlat, nlon, np.arange(ntime) * 6.0)


def _wind(nlat, nlon, ntime):
    hours = np.arange(ntime) * 6.0
    return tuple(synthetic.pv_field(nlat, nlon, hours, seed=synthetic.SEED + k) for k in (1, 2))


def _dev(a):
    """a device tensor of a's dtype (int16 stays int16)"""
    return torch.from_numpy(np.ascontiguousarray(a)).to(_lib.get().device)


def _slices(a, T):
    return [_dev(a[t:t + T]) for t in range(0, len(a), T)]


def _uv_items(u, v, T):
    return list(zip(_slices(u, T), _slices(v, T)))


def _stream(det, raw, T, items=None, depth=2, **kw):
    res = list(det.stream(_slices(raw, T), depth=depth, intensity=items, **kw))
    sums = {k: np.concatenate([r.tables[k].sums for r in res]) for k in detect.KINDS}
    return res, sums


def _same_tables(a, b):
    assert len(a) == len(b)
    for ra, rb in zip(a, b):
        for kind in detect.KINDS:
            ta, tb = ra.tables[kind], rb.tables[kind]
            assert np.array_equal(ta.job, tb.job) and np.array_equal(ta.box, tb.box), kind
            assert np.array_equal(ta.ind1, tb.ind1) and np.array_equal(ta.ind2, tb.ind2), kind
            assert np.array_equal(ta.sums, tb.sums, equal_nan=True), kind


def _props(det, res, kind):
    return np.concatenate([detect.finish_properties(r.tables[kind], det.lon, det.lat, det.nlon)["intensity"]
                           for r in res])


def _some_intensity(res):
    s = np.concatenate([r.tables[k].sums[:, 2] for r in res for k in detect.KINDS])
    return bool(((s != 0) & np.isfinite(s)).any())


# ------------------------------------------------------------------------------------------- the kernel
@pytest.mark.parametrize("nlon", [90, 1447])  # one pairwise leaf, several leaves
def test_packed_mflux_abi_emu(emu, nlon):
    ntime, nlat = 2, 5
    rng = np.random.default_rng(nlon)
    u = _pack(rng.standard_normal((ntime, nlat, nlon)) * 3.0, PK_U, fill_every=37)
    v = _pack(rng.standard_normal((ntime, nlat, nlon)) * 3.0, PK_V, fill_every=53)
    du, dv = _decode(u, PK_U), _decode(v, PK_V)
    assert np.isnan(du).any() and np.isnan(dv).any()
    packing = (_lib.SmoothOpts * 2)(_lib.smooth_opts(False, False, *PK_U), _lib.smooth_opts(False, False, *PK_V))
    for sequential in (0, 1):
        out = torch.empty((ntime, nlat, nlon), dtype=torch.float64)
        emu.call("wbk_mflux", _lib.ptr(_dev(u)), _lib.ptr(_dev(v)), _lib.ptr(out), _lib.I16, ntime, nlat, nlon,
                 sequential, packing, None)
        if sequential:  # longitude is not the contiguous axis of the user's array: numpy sums it sequentially
            ut, vt = (np.ascontiguousarray(np.swapaxes(a, 1, 2)) for a in (du, dv))
            want = P.momentum_flux(np.swapaxes(ut, 1, 2), np.swapaxes(vt, 1, 2))
        else:
            want = P.momentum_flux(du, dv)
        assert np.array_equal(out.numpy(), want, equal_nan=True), sequential
        assert np.isnan(want).any() and np.isfinite(want).any()
    # refusals: packed u / v need both packings, float ones take none, the flux is written in stored order
    out = torch.empty((ntime, nlat, nlon), dtype=torch.float64)
    flipped = (_lib.SmoothOpts * 2)(_lib.smooth_opts(True, False, *PK_U), _lib.smooth_opts(False, False, *PK_V))
    for args, match in (((_dev(u), _dev(v), _lib.I16, None), "packing"),
                        ((_dev(du), _dev(dv), _lib.F64, packing), "packing"),
                        ((_dev(u), _dev(v), _lib.I16, flipped), "flip")):
        with pytest.raises(_lib.WbkError, match=match):
            emu.call("wbk_mflux", _lib.ptr(args[0]), _lib.ptr(args[1]), _lib.ptr(out), args[2], ntime, nlat, nlon, 0,
                     args[3], None)


# ------------------------------------------------------------------------------------------- stream
@pytest.mark.parametrize("depth", [1, 3])
def test_packed_uv_items_emu(emu, depth):
    """three levels, batches of 2 steps with a partial last one: packed (u, v) items give the tables of float64 items
    holding the flux of the host-decoded u and v"""
    nlat, nlon, ntime, T = 46, 90, 5, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, v = _wind(nlat, nlon, ntime)
    pu, pv = _pack(u, PK_U, fill_every=401), _pack(v, PK_V, fill_every=577)
    mf = P.momentum_flux(_decode(pu, PK_U), _decode(pv, PK_V))
    det = pipeline.Detector(lat, lon, levels=LEVELS, intensity_packing=(PK_U, PK_V))
    got, sums = _stream(det, raw, T, _uv_items(pu, pv, T), depth=depth)
    want, _ = _stream(pipeline.Detector(lat, lon, levels=LEVELS), raw, T, _slices(mf, T), depth=depth)
    _same_tables(got, want)
    assert sum(len(s) for s in sums.values()) > 0 and _some_intensity(got)


@pytest.mark.parametrize("flip_lat,flip_lon", [(True, False), (False, True), (True, True)])
def test_packed_field_descending_emu(emu, flip_lat, flip_lon):
    """a packed single field stored with descending coordinates, with fill values inside events, gives the tables of
    the host-decoded float64 field stored the same way"""
    nlat, nlon, ntime, T = 46, 90, 5, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, _ = _wind(nlat, nlon, ntime)

    def stored(a):
        return np.ascontiguousarray(a[:, ::-1 if flip_lat else 1, ::-1 if flip_lon else 1])

    lat_s, lon_s = (lat[::-1] if flip_lat else lat), (lon[::-1] if flip_lon else lon)
    pf = _pack(stored(u), PK_F, fill_every=97)
    det = pipeline.Detector(lat_s, lon_s, levels=LEVELS, intensity_packing=PK_F)
    got, sums = _stream(det, stored(raw), T, _slices(pf, T))
    want, _ = _stream(pipeline.Detector(lat_s, lon_s, levels=LEVELS), stored(raw), T,
                      _slices(_decode(pf, PK_F), T))
    _same_tables(got, want)
    allsums = np.concatenate([s[:, 2] for s in sums.values()])
    assert np.isnan(allsums).any()  # a fill value inside an event
    assert _some_intensity(got)


def test_packed_against_oracle_emu(emu):
    """packed PV (packing=) and packed u, v against the reference on the decoded fields"""
    nlat, nlon, ntime, T = 91, 180, 3, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, v = _wind(nlat, nlon, ntime)
    praw, pu, pv = _pack(raw, PK_PV), _pack(u, PK_U), _pack(v, PK_V)  # no fill values: out of member cells
    draw, du, dv = _decode(praw, PK_PV), _decode(pu, PK_U), _decode(pv, PK_V)
    det = pipeline.Detector(lat, lon, levels=LEVELS, packing=PK_PV, intensity_packing=(PK_U, PK_V))
    gmax = detect.contours(spatial.smooth(draw, 5), LEVELS, det.add).max_nx  # exp_lon.max() of the whole record
    res, sums = _stream(det, praw, T, _uv_items(pu, pv, T), gmax_nx=gmax)
    want = P.detect_steps(draw, P.Grid(lon, lat, synthetic.time_axis(ntime, 6)), levels=LEVELS,
                          intensity=P.momentum_flux(du, dv))
    for kind in detect.KINDS:
        assert len(sums[kind]) == len(want["events"][kind]), kind
        if len(sums[kind]):
            assert np.array_equal(_props(det, res, kind), want["events"][kind].intensity.values), kind
    assert _some_intensity(res)
    flags = np.concatenate([r.flags[:, :r.ntime].numpy() for r in res], axis=1)
    assert np.array_equal(flags, np.stack([want["flags"][k] for k in detect.KINDS]))


# ------------------------------------------------------------------------------------------- re-runs
def _tracked(det, raw, T, items):
    dates = synthetic.time_axis(len(raw), 6)
    clim = pipeline.FlagClimatology(det, np.zeros(len(raw), dtype=np.int32))
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=6)
    res, sums = _stream(det, raw, T, items, climatology=clim, trackers=[tr])
    return res, sums, clim, tr


def test_packed_regrowth_emu(emu, monkeypatch):
    """re-runs with larger arenas carry the packed items unchanged"""
    nlat, nlon, ntime, T = 46, 90, 5, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, v = _wind(nlat, nlon, ntime)
    praw = _pack(raw, PK_PV)
    items = _uv_items(_pack(u, PK_U, fill_every=401), _pack(v, PK_V), T)
    kw = dict(levels=LEVELS, want_pieces=True, packing=PK_PV, intensity_packing=(PK_U, PK_V))
    res, sums, clim, tr = _tracked(pipeline.Detector(lat, lon, **kw), praw, T, items)
    tiny = dict(max_jobs=4, seg_cap=64, contour_cap=4, sel_cap=1, pair_cap=16, event_cap=1)
    monkeypatch.setattr(detect, "default_caps", lambda nlat, nlon, add, njobs: dict(tiny, max_jobs=int(njobs)))
    det = pipeline.Detector(lat, lon, **kw)
    res2, sums2, clim2, tr2 = _tracked(det, praw, T, items)
    assert det._grow
    _same_tables(res2, res)
    assert _some_intensity(res2)
    assert clim2.steps.tolist() == [ntime] and np.array_equal(clim2.counts(), clim.counts())
    assert tr2.cursor == ntime and tr2.n_events == tr.n_events == len(sums["streamers"])
    assert np.array_equal(tr2.labels(), tr.labels())


# ------------------------------------------------------------------------------------------- detect_file
def test_detect_file_packed_emu(emu, tmp_path):
    from wavebreaking_b200 import io

    nlat, nlon, ntime, T = 46, 90, 5, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, v = _wind(nlat, nlon, ntime)
    praw, pu, pv = _pack(raw, PK_PV), _pack(u, PK_U, fill_every=401), _pack(v, PK_V, fill_every=577)
    files = {}
    for name, a in (("pv", praw), ("u", pu), ("v", pv), ("u32", u), ("v32", v)):
        np.save(str(tmp_path / (name + ".npy")), a)
        a.tofile(str(tmp_path / (name + ".bin")))
        files[name] = str(tmp_path / name)
    assert io.open_field(files["pv"] + ".npy").dtype == np.int16
    assert io.open_field(files["u"] + ".bin", shape=u.shape, dtype=np.int16).dtype == np.int16
    kw = dict(levels=LEVELS, packing=PK_PV, intensity_packing=(PK_U, PK_V))
    want, _ = _stream(pipeline.Detector(lat, lon, **kw), praw, T, _uv_items(pu, pv, T))
    assert _some_intensity(want)
    for ext, fkw in ((".npy", {}), (".bin", dict(shape=raw.shape, dtype=np.int16))):
        got = [r for _, r in io.detect_file(files["pv"] + ext, lat, lon, batch=T, depth=2,
                                            intensity=(files["u"] + ext, files["v"] + ext), **fkw, **kw)]
        _same_tables(got, want)
    # .npy files carry their own dtype: an int16 PV file with float32 u / v files
    want, _ = _stream(pipeline.Detector(lat, lon, levels=LEVELS, packing=PK_PV), praw, T, _uv_items(u, v, T))
    got = [r for _, r in io.detect_file(files["pv"] + ".npy", lat, lon, batch=T, depth=2, levels=LEVELS,
                                        packing=PK_PV, intensity=(files["u32"] + ".npy", files["v32"] + ".npy"))]
    _same_tables(got, want)


# ------------------------------------------------------------------------------------------- refusals
def test_packed_refusals_emu(emu):
    nlat, nlon, ntime, T = 46, 90, 4, 2
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, v = _wind(nlat, nlon, ntime)
    p = _slices(_pack(u, PK_U), T)
    f = _slices(u, T)
    plain = pipeline.Detector(lat, lon, levels=[2.0])
    single = pipeline.Detector(lat, lon, levels=[2.0], intensity_packing=PK_F)
    pair = pipeline.Detector(lat, lon, levels=[2.0], intensity_packing=(PK_U, PK_V))
    bad = [
        (plain, [p[0]] + p[1:], "intensity_packing"),                        # int16 without a packing
        (plain, [(p[0], p[0])] + p[1:], "int16"),
        (single, [f[0].to(torch.float16)] + f[1:], "float32 or float64"),
        (single, [(p[0], p[0])] + p[1:], "pair of packings"),                # one packing, (u, v) items
        (pair, [p[0]] + p[1:], "pair of packings"),                          # two packings, a single field
        (single, f, "intensity_packing"),                                    # a packing with float items
        (pair, list(zip(f, f)), "intensity_packing"),
        (pair, [(p[0], f[0])] + list(zip(p[1:], p[1:])), "u and v differ"),  # u int16, v float
    ]
    for det, items, match in bad:
        with pytest.raises(ValueError, match=match):
            list(det.stream(_slices(raw, T), intensity=items))
        assert not det._slots  # refused before any device work on the batch
    for pk in ((float("nan"), 0.0, None), (1.0, float("inf"), None), ((1.0, 0.0, None), (float("inf"), 0.0, None))):
        with pytest.raises(ValueError, match="finite"):
            pipeline.Detector(lat, lon, levels=[2.0], intensity_packing=pk)
    with pytest.raises(ValueError, match="intensity_packing"):
        pipeline.Detector(lat, lon, levels=[2.0], intensity_packing=(1.0, 0.0))


def test_raster_refuses_int16_without_packing_emu(emu):
    nlat, nlon = 46, 90
    lat, lon, raw = _record(nlat, nlon, 1)
    det = pipeline.Detector(lat, lon, levels=[2.0])
    sm = spatial.smooth(raw, 5)
    cs = detect.contours(sm, [2.0], det.add)
    ctx = detect.get_context(nlat, nlon, det.add, 1, {})
    prm = det._prm(cs.max_nx)
    work = torch.empty(2 * max(cs.npoints, 1), dtype=torch.float64)
    emu.call("wbk_index_run", ctx.handle, cs.njobs, 1, _lib.ptr(cs.job_off), _lib.ptr(cs.pt_off), _lib.ptr(cs.meta),
             _lib.ptr(cs.pts), cs.ncontours, cs.npoints, _lib.ptr(det.coords), _lib.ptr(work), ctypes.byref(prm), None)
    inten = _dev(_pack(raw, PK_F))
    with pytest.raises(_lib.WbkError, match="packing"):
        emu.call("wbk_events_raster", ctx.handle, _lib.ptr(cs.job_off), _lib.ptr(cs.pt_off), _lib.ptr(cs.pts),
                 _lib.ptr(det.coords), _lib.ptr(sm), _lib.F64, _lib.ptr(inten), _lib.I16, None, 1, None,
                 ctypes.byref(prm), None)


# ------------------------------------------------------------------------------------------- sharded runs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


NT_SHARD = 7


def _shard_inputs():
    lat, lon, raw = _record(46, 90, NT_SHARD)
    u, v = _wind(46, 90, NT_SHARD)
    return lat, lon, _pack(raw, PK_PV), _pack(u, PK_U, fill_every=401), _pack(v, PK_V)


def _shard_detector(lat, lon):
    return pipeline.Detector(lat, lon, levels=LEVELS, packing=PK_PV, intensity_packing=(PK_U, PK_V))


def _shard_worker(rank, world, port, emu_path, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    _lib.use_library(emu_path, "cpu")
    lat, lon, raw, u, v = _shard_inputs()
    det = _shard_detector(lat, lon)
    _, _, one = sharding.run_sharded(det, _dev(raw), intensity=(_dev(u), _dev(v)))
    np.savez(os.path.join(out_dir, "rank_{}.npz".format(rank)),
             **{"sharded_" + k: _props(det, [one], k) for k in detect.KINDS})
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_packed_intensity_gloo(emu, emu_lib, tmp_path):
    """the intensity column of the two ranks' events, concatenated, equals the single-process run's"""
    import torch.multiprocessing as mp

    lat, lon, raw, u, v = _shard_inputs()
    det = _shard_detector(lat, lon)
    whole = det.run_batch(_dev(raw), intensity=(_dev(u), _dev(v)))
    # one process: run_sharded slices the packed items like the field
    _, _, one = sharding.run_sharded(det, _dev(raw), intensity=(_dev(u), _dev(v)))
    _same_tables([one], [whole])
    assert _some_intensity([whole])
    mp.spawn(_shard_worker, args=(2, _free_port(), emu_lib, str(tmp_path)), nprocs=2, join=True)
    ranks = [np.load(tmp_path / "rank_{}.npz".format(r)) for r in range(2)]
    n = 0
    for kind in detect.KINDS:
        got = np.concatenate([z["sharded_" + kind] for z in ranks])
        assert np.array_equal(got, _props(det, [whole], kind), equal_nan=True), kind
        n += len(got)
    assert n > 0


# ------------------------------------------------------------------------------------------- GPU
def _tpack(x, pk):
    """_pack on the device"""
    scale, offset, _ = pk
    return torch.round((x.double() - offset) / scale).clamp(-32766, 32766).to(torch.int16)


def _tdecode(s, pk):
    scale, offset, fill = pk
    x = s.double() * scale + offset
    return x if fill is None else torch.where(s == fill, torch.full_like(x, float("nan")), x)


def _graph_case(nlat, nlon, T, shared, uv):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    slabs = [spatial.synth_pv(T, nlat, nlon, hour0=500.0 + T * b, hour_step=1.0) for b in range(2)]
    tail = spatial.synth_pv(T - 3, nlat, nlon, hour0=500.0 + 2 * T, hour_step=1.0)

    def field(n, b, seed, pk):
        x = _tpack(spatial.synth_pv(n, nlat, nlon, hour0=500.0 + T * b, hour_step=1.0, seed=seed), pk)
        x.view(-1)[7::997] = pk[2]
        return x

    def item(n, b):
        if uv:
            return field(n, b, synthetic.SEED + 1, PK_U), field(n, b, synthetic.SEED + 2, PK_V)
        return field(n, b, synthetic.SEED + 3, PK_F)

    islabs, itail = [item(T, b) for b in range(2)], item(T - 3, 2)
    batches = [slabs[i % 2] for i in range(6)] + [tail]  # every slot sees its buffers 3 times: eager, capture, replay
    items = [islabs[i % 2] for i in range(6)] + [itail]
    packing = (PK_U, PK_V) if uv else PK_F
    det = pipeline.Detector(lat, lon, levels=LEVELS, graphs=True, intensity_packing=packing)
    got = list(det.stream(batches, depth=2, shared_stream=shared, intensity=items))
    assert det.graph_replays >= 4
    eager = pipeline.Detector(lat, lon, levels=LEVELS, intensity_packing=packing)
    want = list(eager.stream(batches, depth=2, intensity=items))
    assert eager.graph_replays == 0
    _same_tables(got, want)
    assert _some_intensity(got)
    # detect.run_indices on one replayed batch with the host-decoded float64 field / flux
    b = 4
    if uv:
        dec = spatial.momentum_flux(_tdecode(items[b][0], PK_U), _tdecode(items[b][1], PK_V))
    else:
        dec = _tdecode(items[b], PK_F)
    assert dec.dtype == torch.float64
    sm = spatial.smooth(batches[b], 5)
    tables, _ = detect.run_indices(detect.contours(sm, LEVELS, det.add), sm, det.coords, det.dlon, det.dlat,
                                   intensity=dec, gmax_nx=det.nlon + det.add, want_flags=True)
    for kind in detect.KINDS:
        assert np.array_equal(got[b].tables[kind].sums, tables[kind].sums, equal_nan=True), kind


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(181, 360), (721, 1440)])
@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("uv", [False, True])
def test_packed_intensity_graphs_gpu(gpu, shape, shared, uv):
    _graph_case(shape[0], shape[1], 8, shared, uv)


@pytest.mark.gpu
def test_pinned_host_packed_gpu(gpu):
    """pinned-host packed PV + u + v at 721 x 1440 with CUDA graphs equal device-resident host-decoded float64 items"""
    nlat, nlon, T = 721, 1440, 6
    lat, lon = synthetic.grid_coords(nlat, nlon)

    def slab(b, seed=None):
        return spatial.synth_pv(T, nlat, nlon, hour0=300.0 + T * b, seed=seed)

    praw = [_tpack(slab(b), PK_PV) for b in range(2)]
    puv = [(_tpack(slab(b, synthetic.SEED + 1), PK_U), _tpack(slab(b, synthetic.SEED + 2), PK_V)) for b in range(2)]
    for pu, _ in puv:
        pu.view(-1)[7::4001] = PK_U[2]
    pin = [r.cpu().pin_memory() for r in praw]
    pin_uv = [tuple(x.cpu().pin_memory() for x in p) for p in puv]
    det = pipeline.Detector(lat, lon, levels=LEVELS, graphs=True, packing=PK_PV, intensity_packing=(PK_U, PK_V))
    got = list(det.stream([pin[i % 2] for i in range(6)], depth=2, intensity=[pin_uv[i % 2] for i in range(6)]))
    assert det.graph_replays >= 2
    draw = [_tdecode(r, PK_PV) for r in praw]
    duv = [(_tdecode(pu, PK_U), _tdecode(pv, PK_V)) for pu, pv in puv]
    want = list(pipeline.Detector(lat, lon, levels=LEVELS).stream([draw[i % 2] for i in range(6)], depth=2,
                                                                 intensity=[duv[i % 2] for i in range(6)]))
    _same_tables(got, want)
    assert _some_intensity(got)


@pytest.mark.gpu
def test_packed_three_levels_oracle_gpu(gpu):
    nlat, nlon, ntime, T = 91, 180, 4, 3
    lat, lon, raw = _record(nlat, nlon, ntime)
    u, v = _wind(nlat, nlon, ntime)
    praw, pu, pv = _pack(raw, PK_PV), _pack(u, PK_U), _pack(v, PK_V)
    draw = _decode(praw, PK_PV)
    det = pipeline.Detector(lat, lon, levels=LEVELS, packing=PK_PV, intensity_packing=(PK_U, PK_V))
    gmax = detect.contours(spatial.smooth(draw, 5), LEVELS, det.add).max_nx
    res, sums = _stream(det, praw, T, _uv_items(pu, pv, T), gmax_nx=gmax)
    want = P.detect_steps(draw, P.Grid(lon, lat, synthetic.time_axis(ntime, 6)), levels=LEVELS,
                          intensity=P.momentum_flux(_decode(pu, PK_U), _decode(pv, PK_V)))
    for kind in detect.KINDS:
        assert len(sums[kind]) == len(want["events"][kind]), kind
        if len(sums[kind]):
            assert np.array_equal(_props(det, res, kind), want["events"][kind].intensity.values), kind
    assert _some_intensity(res)
    flags = np.concatenate([r.flags[:, :r.ntime].cpu().numpy() for r in res], axis=1)
    assert np.array_equal(flags, np.stack([want["flags"][k] for k in detect.KINDS]))
