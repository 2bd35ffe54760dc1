"""Flag-frequency climatologies: wbk_flag_counts, FlagClimatology in Detector.stream, reduce_climatology and
flag_frequency, against numpy sums of the flag grids."""

import os
import socket
import sys

import numpy as np
import pytest
import torch

from oracle import pipeline as P
from wavebreaking_b200 import _lib, api, compat, detect, pipeline, spatial, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------- wbk_flag_counts
def _want_counts(flags, group, ngroups):
    nk, nt, nc = flags.shape
    want = np.zeros((ngroups, nk, nc), dtype=np.int64)
    for t in range(nt):
        if 0 <= group[t] < ngroups:
            want[group[t]] += flags[:, t] != 0
    return want


def _flag_counts_case(lib, nkinds, ntime, ncells, misalign, seed):
    rng = np.random.default_rng(seed)
    values = np.array([0, 0, 0, 1, 1, -1, 7, -128], dtype=np.int8)
    dev = lib.device
    buf = torch.tensor(rng.choice(values, size=nkinds * ntime * ncells + 16), device=dev)  # (a 64-byte aligned copy)
    flags = buf[misalign:misalign + nkinds * ntime * ncells]
    assert (flags.data_ptr() % 16 == 0) == (misalign == 0)
    ngroups = 3
    # runs of equal groups, steps not counted (-1) and values outside [0, ngroups) that must be ignored like -1
    group = np.repeat(np.array([0, 0, 2, -1, 1, 5, 1, -7, 2], dtype=np.int32), max(1, ntime // 9) + 1)[:ntime]
    counts = torch.zeros((ngroups, nkinds, ncells), dtype=torch.int32, device=dev)
    g_dev = torch.from_numpy(group).to(dev)
    for _ in range(3):  # several calls add up
        lib.call("wbk_flag_counts", _lib.ptr(flags), nkinds, ntime, ncells, _lib.ptr(g_dev), ngroups, _lib.ptr(counts),
                 lib.stream())
    # a batch whose groups are all out of range changes no counter
    bad = torch.from_numpy(np.array([-1, 3, 99, -2] * ntime, dtype=np.int32)[:ntime]).to(dev)
    lib.call("wbk_flag_counts", _lib.ptr(flags), nkinds, ntime, ncells, _lib.ptr(bad), ngroups, _lib.ptr(counts),
             lib.stream())
    got = counts.cpu().numpy().view(np.uint32).astype(np.int64)
    host = flags.cpu().numpy().reshape(nkinds, ntime, ncells)
    assert np.array_equal(got, 3 * _want_counts(host, group, ngroups))


@pytest.mark.parametrize("nkinds", [1, 3])
@pytest.mark.parametrize("ncells,misalign", [(160, 0), (45, 0), (160, 1)])  # vector path, scalar path, misaligned view
def test_flag_counts_matches_numpy_emu(emu, nkinds, ncells, misalign):
    _flag_counts_case(emu, nkinds, 19, ncells, misalign, seed=ncells + nkinds + misalign)


def test_flag_counts_refusals_emu(emu):
    f = torch.zeros(64, dtype=torch.int8)
    g = torch.zeros(4, dtype=torch.int32)
    c = torch.zeros(64, dtype=torch.int32)
    bad = [(f, 0, 4, 16, g, 1, c), (f, 1, -1, 16, g, 1, c), (f, 1, 4, -16, g, 1, c), (f, 1, 4, 16, g, 0, c),
           (None, 1, 4, 16, g, 1, c), (f, 1, 4, 16, None, 1, c), (f, 1, 4, 16, g, 1, None)]
    for fl, nk, nt, nc, gr, ng, cn in bad:
        with pytest.raises(_lib.WbkError, match="wbk_flag_counts"):
            emu.call("wbk_flag_counts", _lib.ptr(fl), nk, nt, nc, _lib.ptr(gr), ng, _lib.ptr(cn), None)
    # nothing to do: no pointer is needed
    emu.call("wbk_flag_counts", None, 3, 0, 16, None, 1, None, None)
    emu.call("wbk_flag_counts", None, 3, 4, 0, None, 1, None, None)


# ------------------------------------------------------------------------------------------- groups_from_dates
def test_groups_from_dates():
    dates = np.array(["1999-12-31T23", "2000-01-01T00", "2000-02-29T23", "2000-03-01T00", "2000-05-31T23",
                      "2000-06-01T00", "2000-08-31T23", "2000-09-01T00", "2000-11-30T23", "2000-12-01T00", "NaT"],
                     dtype="datetime64[h]")
    assert list(pipeline.groups_from_dates(dates, "month")) == [11, 0, 1, 2, 4, 5, 7, 8, 10, 11, -1]
    assert list(pipeline.groups_from_dates(dates, "season")) == [0, 0, 0, 1, 1, 2, 2, 3, 3, 0, -1]
    assert list(pipeline.groups_from_dates(dates, "all")) == [0] * 10 + [-1]
    assert pipeline.groups_from_dates(dates, "month").dtype == np.int32
    with pytest.raises(ValueError):
        pipeline.groups_from_dates(dates, "year")
    with pytest.raises(ValueError):
        pipeline.groups_from_dates(np.arange(3), "month")


# ------------------------------------------------------------------------------------------- Detector.stream
START = np.datetime64("2000-01-31T06", "h")  # 6-hourly: the record enters February at step 3


def _record(nlat, nlon, ntime, step_hours=6, hour0=0.0):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, hour0 + np.arange(ntime) * float(step_hours))
    dates = START + np.arange(ntime) * np.timedelta64(step_hours, "h")
    return lat, lon, raw, dates


def _stream_climatology(det, raw, groups, T, ngroups=12, **kw):
    """Stream `raw` in batches of T steps (the last one partial) with a climatology; returns it and the flag grids
    [3, ntime, nlat, nlon] the run returned."""
    clim = pipeline.FlagClimatology(det, groups, ngroups=ngroups)
    batches = [spatial.to_device(raw[t:t + T]) for t in range(0, len(raw), T)]
    got = []
    for res in det.stream(batches, climatology=clim, **kw):
        if res.flags_packed is not None:
            got.append(pipeline.unpack_flags(res.flags_packed, res.ntime, det.nlat, det.nlon).copy())
        else:
            got.append(res.flags[:, :res.ntime].cpu().numpy().copy())
    return clim, np.concatenate(got, axis=1)


def _want_from_flags(flags, groups, ngroups):
    nlat, nlon = flags.shape[2:]
    want = _want_counts(flags.reshape(3, flags.shape[1], -1), groups, ngroups)
    return want.reshape(ngroups, 3, nlat, nlon), np.bincount(groups[groups >= 0], minlength=ngroups)


def _check(clim, flags, groups):
    want, steps = _want_from_flags(flags, groups, clim.ngroups)
    assert np.array_equal(clim.counts().astype(np.int64), want)
    assert np.array_equal(clim.steps, steps)
    assert clim.cursor == len(groups)
    freq = clim.frequency()
    with np.errstate(invalid="ignore", divide="ignore"):
        assert np.allclose(freq, 100.0 * want / steps[:, None, None, None], equal_nan=True)
    assert np.isnan(freq[steps == 0]).all()


@pytest.mark.parametrize("depth", [1, 3])
@pytest.mark.parametrize("shape", [(46, 90), (41, 80)])  # 4140 cells: byte loads; 3280 = 16 * 205: 16-byte loads
def test_stream_monthly_climatology_emu(emu, depth, shape):
    nlat, nlon = shape
    lat, lon, raw, dates = _record(nlat, nlon, 7)
    groups = pipeline.groups_from_dates(dates, "month")
    assert list(groups) == [0, 0, 0, 1, 1, 1, 1]
    det = pipeline.Detector(lat, lon, levels=[2.0])
    clim, flags = _stream_climatology(det, raw, groups, T=3, depth=depth)  # batches of 3, 3 and 1 steps
    assert flags.any()
    _check(clim, flags, groups)
    assert clim.counts().shape == (12, 3, nlat, nlon) and clim.counts().dtype == np.uint32


def test_stream_climatology_matches_oracle_flags_emu(emu):
    nlat, nlon, ntime = 46, 90, 5
    lat, lon, raw, dates = _record(nlat, nlon, ntime)
    groups = pipeline.groups_from_dates(dates, "month")
    det = pipeline.Detector(lat, lon, levels=[2.0])
    clim, _ = _stream_climatology(det, raw, groups, T=2, depth=2)
    want = P.detect_steps(raw, P.Grid(lon, lat, synthetic.time_axis(ntime, 6)), levels=[2.0])
    oracle_flags = np.stack([want["flags"][kind] for kind in detect.KINDS])
    counts, steps = _want_from_flags(oracle_flags, groups, 12)
    assert oracle_flags.any()
    assert np.array_equal(clim.counts().astype(np.int64), counts)
    assert np.array_equal(clim.steps, steps)


def test_stream_climatology_counts_regrown_batches_once_emu(emu, monkeypatch):
    """arenas too small for every batch: each batch overflows, is re-run with larger arenas and counted once"""
    lat, lon, raw, dates = _record(46, 90, 5)
    groups = pipeline.groups_from_dates(dates, "month")
    tiny = dict(max_jobs=4, seg_cap=64, contour_cap=4, sel_cap=1, pair_cap=16, event_cap=1)
    monkeypatch.setattr(detect, "default_caps", lambda nlat, nlon, add, njobs: dict(tiny, max_jobs=int(njobs)))
    det = pipeline.Detector(lat, lon, levels=[2.0, -2.0])
    clim, flags = _stream_climatology(det, raw, groups, T=2, depth=2)
    assert det._grow  # the arenas were regrown
    _check(clim, flags, groups)
    assert clim.steps.sum() == 5


def test_stream_climatology_with_pieces_emu(emu):
    """want_pieces: a batch whose piece buffers are too small is re-run (want_pieces capacity path) and counted once"""
    lat, lon, raw, dates = _record(46, 90, 4, hour0=384.0)  # events that straddle the last meridian: 6 pieces
    groups = pipeline.groups_from_dates(dates, "month")
    det = pipeline.Detector(lat, lon, levels=[2.0], want_pieces=True)
    for idx in range(2):
        det._slot(2, idx).cap_sr = 1  # the buffers are larger: only the check sees the small capacity
    clim, flags = _stream_climatology(det, raw, groups, T=2, depth=2)
    assert "cap_sr" in det._grow  # at least one batch took the want_pieces capacity path
    _check(clim, flags, groups)


def test_climatology_refusals_emu(emu):
    lat, lon, raw, dates = _record(46, 90, 4)
    with pytest.raises(ValueError, match="want_flags"):
        pipeline.FlagClimatology(pipeline.Detector(lat, lon, want_flags=False), np.zeros(4, dtype=np.int32))
    det = pipeline.Detector(lat, lon, levels=[2.0])
    with pytest.raises(ValueError, match="outside"):
        pipeline.FlagClimatology(det, np.array([0, 1, 12, 0]), ngroups=12)
    with pytest.raises(ValueError, match="outside"):
        pipeline.FlagClimatology(det, np.array([0, -2, 1, 0]))
    with pytest.raises(ValueError):
        pipeline.FlagClimatology(det, np.zeros(4, dtype=np.float64))
    # the stream runs past the end of the group array
    clim = pipeline.FlagClimatology(det, np.zeros(3, dtype=np.int32))
    with pytest.raises(ValueError, match="group array"):
        list(det.stream([spatial.to_device(raw[:2]), spatial.to_device(raw[2:])], depth=1, climatology=clim))
    assert clim.steps.tolist() == [2]  # the first batch was counted, the second refused
    # a Detector without flag grids cannot feed a climatology
    with pytest.raises(ValueError, match="want_flags"):
        list(pipeline.Detector(lat, lon, want_flags=False).stream([spatial.to_device(raw)], climatology=clim))


def test_detect_file_climatology_emu(emu, tmp_path):
    lat, lon, raw, dates = _record(46, 90, 5)
    path = str(tmp_path / "pv.npy")
    np.save(path, raw)
    groups = pipeline.groups_from_dates(dates, "season")
    det = pipeline.Detector(lat, lon, levels=[2.0])
    clim = pipeline.FlagClimatology(det, groups, ngroups=4)
    from wavebreaking_b200 import io

    flags = np.concatenate([r.flags[:, :r.ntime].cpu().numpy().copy() for _, r in
                            io.detect_file(path, lat, lon, batch=2, depth=2, levels=[2.0], climatology=clim)], axis=1)
    _check(clim, flags, groups)


# ------------------------------------------------------------------------------------------- flag_frequency
def _field(values, time, lat, lon, dims=("time", "lat", "lon")):
    coords = {"time": time, "lat": compat._Coord(lat, {"units": "degrees_north"}),
              "lon": compat._Coord(lon, {"units": "degrees_east"})}
    return compat.Field(values, dims, coords, name="flag")


def _freq_numpy(values, months_of_steps, months):
    sel = np.ones(len(months_of_steps), bool) if months is None else np.isin(months_of_steps, months)
    with np.errstate(invalid="ignore"):
        return 100.0 * (values[sel] != 0).sum(axis=0) / sel.sum()


def test_flag_frequency_hand_written_field_emu(emu):
    rng = np.random.default_rng(3)
    nt, nlat, nlon = 9, 7, 12
    time = np.datetime64("2001-01-30", "D") + np.arange(nt) * np.timedelta64(2, "D")  # January into February
    month = time.astype("datetime64[M]").astype(int) % 12 + 1
    lat = np.linspace(-60, 60, nlat)
    lon = np.arange(nlon) * 30.0
    values = rng.choice(np.array([0, 0, 1], dtype=np.int8), size=(nt, nlat, nlon))
    data = _field(values, time, lat, lon)
    for months in (None, [2], [1, 2], [7]):
        out = api.flag_frequency(data, months=months)
        assert out.dims == ("lat", "lon") and out.values.dtype == np.float64
        assert out.attrs["units"] == "%" and "long_name" in out.attrs
        assert np.allclose(out.values, _freq_numpy(values, month, months), equal_nan=True), months
    assert np.isnan(api.flag_frequency(data, months=[7]).values).all()
    # another dimension order and descending latitudes: the result keeps both
    swapped = _field(np.ascontiguousarray(values[:, ::-1].transpose(1, 0, 2)), time, lat[::-1], lon,
                     dims=("lat", "time", "lon"))
    out = api.flag_frequency(swapped, months=[1])
    assert out.dims == ("lat", "lon")
    assert np.allclose(out.values, _freq_numpy(values, month, [1])[::-1])
    with pytest.raises(TypeError):
        api.flag_frequency(_field(values.astype(np.float64), time, lat, lon))
    with pytest.raises(ValueError, match="datetime64"):
        api.flag_frequency(_field(values, np.arange(nt, dtype=np.float64), lat, lon), months=[1])
    assert np.allclose(api.flag_frequency(_field(values, np.arange(nt, dtype=np.float64), lat, lon)).values,
                       _freq_numpy(values, month, None))


def _lazy_flags(nlat, nlon, ntime):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, np.arange(ntime) * 6.0).astype(np.float64)
    time = np.datetime64("2002-02-28T00", "h") + np.arange(ntime) * np.timedelta64(12, "h")  # into March
    data = _field(raw[:, ::-1], time, lat[::-1], lon)  # stored with descending latitudes, like ERA5
    events = api.calculate_cutoffs(data, 2.0)
    flags = api.to_xarray(data, events)
    return flags, time


def test_flag_frequency_of_lazy_to_xarray_output_emu(emu):
    flags, time = _lazy_flags(46, 90, 4)
    assert flags._values is None
    out_all = api.flag_frequency(flags)
    out_mar = api.flag_frequency(flags, months=[3])
    assert flags._values is None  # counted on the device: nothing was downloaded
    month = time.astype("datetime64[M]").astype(int) % 12 + 1
    values = flags.values
    assert values.any()
    assert np.allclose(out_all.values, _freq_numpy(values, month, None))
    assert np.allclose(out_mar.values, _freq_numpy(values, month, [3]))


# ------------------------------------------------------------------------------------------- sharded runs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


NT_SHARD = 6
SHARD_START = np.datetime64("2000-01-31T12", "h")  # February starts at step 2, the shard boundary is at step 3


def _shard_worker(rank, world, port, backend, emu_path, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist

    if backend == "nccl":
        torch.cuda.set_device(rank)
    dist.init_process_group(backend, rank=rank, world_size=world)
    from wavebreaking_b200 import _lib, pipeline, sharding, spatial, synthetic

    if emu_path is not None:
        _lib.use_library(emu_path, "cpu")
    nlat, nlon = 46, 90
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, np.arange(NT_SHARD) * 6.0)
    dates = SHARD_START + np.arange(NT_SHARD) * np.timedelta64(6, "h")
    groups = pipeline.groups_from_dates(dates, "month")
    t0, t1 = sharding.shard_range(NT_SHARD, rank, world)
    det = pipeline.Detector(lat, lon, levels=[2.0])
    clim = pipeline.FlagClimatology(det, groups, ngroups=12, t0=t0)
    list(det.stream([spatial.to_device(raw[t0:t1])], depth=1, climatology=clim))
    counts, steps = sharding.reduce_climatology(clim)
    np.save(os.path.join(out_dir, "counts_{}.npy".format(rank)), counts)
    np.save(os.path.join(out_dir, "steps_{}.npy".format(rank)), steps)
    dist.barrier()
    dist.destroy_process_group()


def _single_process_counts():
    nlat, nlon = 46, 90
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, np.arange(NT_SHARD) * 6.0)
    groups = pipeline.groups_from_dates(SHARD_START + np.arange(NT_SHARD) * np.timedelta64(6, "h"), "month")
    assert list(groups) == [0, 0, 1, 1, 1, 1]
    det = pipeline.Detector(lat, lon, levels=[2.0])
    clim, _ = _stream_climatology(det, raw, groups, T=NT_SHARD, depth=1)
    return clim.counts().astype(np.int64), clim.steps


def _run_two_ranks(backend, emu_path, tmp_path):
    import torch.multiprocessing as mp

    mp.spawn(_shard_worker, args=(2, _free_port(), backend, emu_path, str(tmp_path)), nprocs=2, join=True)
    counts, steps = _single_process_counts()
    for rank in range(2):
        got = np.load(tmp_path / "counts_{}.npy".format(rank))
        assert got.dtype == np.int64 and np.array_equal(got, counts), rank
        assert np.array_equal(np.load(tmp_path / "steps_{}.npy".format(rank)), steps), rank
    assert counts.any()


def test_two_rank_gloo_reduce_climatology(emu_lib, tmp_path):
    prev = _lib._LIB
    _lib.use_library(emu_lib, "cpu")
    try:
        _run_two_ranks("gloo", emu_lib, tmp_path)
    finally:
        _lib._LIB = prev


# ------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_flag_counts_matches_numpy_gpu(gpu):
    for nkinds in (1, 3):
        for ncells, misalign in ((361 * 720, 0), (181 * 360, 0), (361 * 720, 3)):
            _flag_counts_case(gpu, nkinds, 37, ncells, misalign, seed=nkinds + misalign)
    # 3 * ntime * ncells passes 2**31 at 721 x 1440 with 700 steps: 64-bit offsets
    ntime, ncells = 700, 721 * 1440
    flags = torch.zeros((3, ntime, ncells), dtype=torch.int8, device=gpu.device)
    flags[2, ntime - 1, ncells - 16:] = 1
    flags[2, ntime - 2, ncells - 1] = 5
    group = torch.zeros(ntime, dtype=torch.int32, device=gpu.device)
    counts = torch.zeros((1, 3, ncells), dtype=torch.int32, device=gpu.device)
    gpu.call("wbk_flag_counts", _lib.ptr(flags), 3, ntime, ncells, _lib.ptr(group), 1, _lib.ptr(counts), gpu.stream())
    got = counts.cpu().numpy()
    assert got.sum() == 17 and got[0, 2, -1] == 2 and got[0, 2, ncells - 16] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(181, 360), (361, 720)])  # byte loads; 16-byte loads
@pytest.mark.parametrize("packed", [False, True])
def test_stream_climatology_gpu(gpu, shape, packed):
    """graphs=True, a shared stream and separate streams, the bit-packed download on and off, a partial last batch"""
    nlat, nlon = shape
    T = 4
    lat, lon = synthetic.grid_coords(nlat, nlon)
    slabs = [spatial.synth_pv(T, nlat, nlon, hour0=float(24 * s), hour_step=1.0) for s in range(2)]
    tail = spatial.synth_pv(T - 1, nlat, nlon, hour0=100.0, hour_step=1.0)
    batches = [slabs[i % 2] for i in range(6)] + [tail]  # every slot sees its buffers 3 times: eager, capture, replay
    ntime = 6 * T + T - 1
    dates = np.datetime64("2003-04-30T14", "h") + np.arange(ntime) * np.timedelta64(1, "h")  # into May at step 10
    groups = pipeline.groups_from_dates(dates, "month")
    for shared in (False, True):
        det = pipeline.Detector(lat, lon, levels=[2.0], graphs=True)
        clim = pipeline.FlagClimatology(det, groups, ngroups=12)
        ph = ([torch.zeros(pipeline.packed_nbytes(3 * T * nlat * nlon), dtype=torch.uint8).pin_memory()
               for _ in range(2)] if packed else None)
        got = []
        for res in det.stream(iter(batches), depth=2, shared_stream=shared, packed_host=ph, climatology=clim):
            if packed:
                got.append(pipeline.unpack_flags(res.flags_packed, res.ntime, nlat, nlon).copy())
            else:
                got.append(res.flags[:, :res.ntime].cpu().numpy())
        assert det.graph_replays >= 2
        flags = np.concatenate(got, axis=1)
        assert flags.any()
        _check(clim, flags, groups)


@pytest.mark.gpu
def test_stream_climatology_counts_regrown_batches_once_gpu(gpu, monkeypatch):
    nlat, nlon = 181, 360
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, np.arange(5) * 6.0)
    groups = pipeline.groups_from_dates(START + np.arange(5) * np.timedelta64(6, "h"), "month")
    tiny = dict(max_jobs=4, seg_cap=64, contour_cap=4, sel_cap=1, pair_cap=16, event_cap=1)
    monkeypatch.setattr(detect, "default_caps", lambda nlat, nlon, add, njobs: dict(tiny, max_jobs=int(njobs)))
    det = pipeline.Detector(lat, lon, levels=[2.0, -2.0])
    clim, flags = _stream_climatology(det, raw, groups, T=2, depth=2)
    assert det._grow
    _check(clim, flags, groups)


@pytest.mark.gpu
def test_flag_frequency_gpu(gpu):
    rng = np.random.default_rng(5)
    nt, nlat, nlon = 30, 181, 360
    time = np.datetime64("2004-06-20", "D") + np.arange(nt) * np.timedelta64(1, "D")
    month = time.astype("datetime64[M]").astype(int) % 12 + 1
    lat, lon = synthetic.grid_coords(nlat, nlon)
    values = rng.choice(np.array([0, 0, 0, 1], dtype=np.int8), size=(nt, nlat, nlon))
    data = _field(values, time, lat, lon)
    for months in (None, [7]):
        assert np.allclose(api.flag_frequency(data, months=months).values, _freq_numpy(values, month, months))
    flags, time = _lazy_flags(181, 360, 4)
    out = api.flag_frequency(flags, months=[3])
    assert flags._values is None
    month = time.astype("datetime64[M]").astype(int) % 12 + 1
    assert np.allclose(out.values, _freq_numpy(flags.values, month, [3]))


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_nccl_reduce_climatology(gpu, tmp_path):
    _run_two_ranks("nccl", None, tmp_path)
