"""Tracking while streaming: wbk_track_append, pipeline.EventTracker in Detector.stream / detect_file and
sharding.finish_tracks, against events_soup + tracking.track_columnar on the concatenated batches and the oracle."""

import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import pipeline as P
from wavebreaking_b200 import detect, pipeline, spatial, synthetic, tracking

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CROSS_HOUR0 = 288.0  # at 61 x 120 the synthetic record has streamers and overturnings across the last meridian


def _record(nlat, nlon, ntime, hour0=CROSS_HOUR0, step=1.0):
    lat, lon = synthetic.grid_coords(nlat, nlon)
    raw = synthetic.pv_field(nlat, nlon, hour0 + np.arange(ntime) * step)
    dates = synthetic.time_axis(ntime, 1)
    return lat, lon, raw, dates


def _soup_polys(soup):
    return [[soup.xy[soup.ring_off[r]:soup.ring_off[r + 1]].astype(np.int64) for r in
             range(soup.poly_off[e], soup.poly_off[e + 1])] for e in range(len(soup))]


def _run(det, batches, trackers, depth=2, **kw):
    """Stream with trackers; per kind the events_soup / com / step of every event of the same results."""
    got = {k: ([], [], []) for k in detect.KINDS}
    t = 0
    L = len(det.levels)
    for res in det.stream(batches, depth=depth, trackers=trackers, **kw):
        for kind in detect.KINDS:
            soup, com = pipeline.events_soup(res, kind, det)
            got[kind][0].append(soup)
            got[kind][1].append(com)
            got[kind][2].append(t + res.tables[kind].job.astype(np.int64) // L)
        t += res.ntime
    return {k: (tracking.PolygonSoup.concat(v[0]), np.concatenate(v[1]), np.concatenate(v[2])) for k, v in got.items()}


def _want(ref, kind, dates, method, time_range, overlap=0, distance=1000):
    soup, com, step = ref[kind]
    return tracking.track_columnar(dates[step], method, soup=soup if method == "by_overlap" else None, com=com,
                                   time_range=time_range, overlap=overlap, distance=distance)


def _sorted(pairs):
    pairs = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    return pairs[np.lexsort((pairs[:, 1], pairs[:, 0]))] if len(pairs) else pairs


def _check(tr, ref, dates):
    labels, near = _want(ref, tr.kind, dates, tr.method, tr.time_range, tr.overlap, tr.distance)
    assert np.array_equal(tr.labels(), labels), (tr.kind, tr.method, tr.overlap)
    assert np.array_equal(tr.near, _sorted(near))
    return labels


def _batches(raw, T):
    return [spatial.to_device(raw[t:t + T]) for t in range(0, len(raw), T)]


# ------------------------------------------------------------------------------------------- device polygons
def _check_window(nlat, nlon, ntime, T, levels=(2.0,)):
    lat, lon, raw, dates = _record(nlat, nlon, ntime)
    det = pipeline.Detector(lat, lon, levels=list(levels), want_pieces=True)
    dates = synthetic.time_axis(ntime + 1, 1)  # one more date: nothing is evicted after the last batch
    trs = [pipeline.EventTracker(det, dates, kind, time_range=10 ** 6) for kind in detect.KINDS]
    ref = _run(det, _batches(raw, T), trs)
    nsplit = 0
    for tr in trs:
        soup = ref[tr.kind][0]
        assert tr.n_events == len(soup) == len(tr._wkeys) > 0
        e, vs, ro, po, bb = (b.cpu().numpy() for b in tr._buf)
        n, R, V = len(soup), len(soup.ring_off) - 1, len(soup.xy)
        edges, vsign = tracking._edge_table(soup)
        assert (tr._nv, tr._nr) == (V, R)
        assert np.array_equal(po[:n + 1], soup.poly_off)
        assert np.array_equal(ro[:R + 1], soup.ring_off)
        assert np.array_equal(e[:V, :2], soup.xy)
        assert np.array_equal(e[:V], edges)
        assert np.array_equal(vs[:V], vsign)
        assert np.array_equal(bb[:n], soup.bounds())
        nsplit += int((np.diff(soup.poly_off) != 1).sum())
    return nsplit


def test_track_append_matches_events_soup_emu(emu):
    """all three kinds, events across the last meridian: device-clipper pieces and straddling overturning boxes"""
    assert _check_window(61, 120, 4, T=2, levels=(2.0, -2.0)) > 0  # some events were replaced by several pieces


def test_track_append_refusals_emu(emu):
    i = torch.zeros(64, dtype=torch.int32)
    args = [None] * 6 + [0, 0, 1, 0, 90, 1, 4]
    win = [i.data_ptr()] * 5
    from wavebreaking_b200 import _lib

    ok = args[:6] + [0, 0, 1, 1, 90, 1, 4] + win + [0, 0, 0, 64, 64, 64, None]
    ok[0] = i.data_ptr()
    emu.call("wbk_track_append", *ok)
    big = list(ok)
    big[18] = 2 ** 31 - 2  # v0: the window would pass 2**31 - 1 vertices
    with pytest.raises(_lib.WbkError, match="2\\^31 - 1"):
        emu.call("wbk_track_append", *big)
    small = list(ok)
    small[21] = 2  # cap_v
    with pytest.raises(_lib.WbkError, match="too small"):
        emu.call("wbk_track_append", *small)
    neg = list(ok)
    neg[8] = -1
    with pytest.raises(_lib.WbkError, match="wbk_track_append"):
        emu.call("wbk_track_append", *neg)


# ------------------------------------------------------------------------------------------- stream labels
@pytest.mark.parametrize("depth,T,time_range", [(1, 3, 1), (3, 2, 3), (2, 4, 2)])
def test_stream_labels_match_track_columnar_emu(emu, depth, T, time_range):
    """partial last batches (7 steps), windows that span batches, three trackers (one per kind) in one stream"""
    lat, lon, raw, dates = _record(61, 120, 7)
    det = pipeline.Detector(lat, lon, levels=[2.0], want_pieces=True)
    trs = [pipeline.EventTracker(det, dates, kind, time_range=time_range) for kind in detect.KINDS]
    ref = _run(det, _batches(raw, T), trs, depth=depth)
    linked = 0
    for tr in trs:
        if tr.kind == "cutoffs" and tr.n_events < 2:
            continue
        labels = _check(tr, ref, dates)
        linked += len(labels) - len(np.unique(labels))
        assert tr.stats["pairs_in_range"] > 0 and len(tr.host_ms) == (7 + T - 1) // T
    assert linked > 0


@pytest.mark.parametrize("method,overlap", [("by_overlap", 0.0), ("by_overlap", 0.2), ("by_distance", 0.0),
                                            ("by_overlap", -0.5)])
def test_stream_methods_two_levels_emu(emu, method, overlap):
    lat, lon, raw, dates = _record(61, 120, 6)
    det = pipeline.Detector(lat, lon, levels=[2.0, -2.0], want_pieces=True)
    trs = [pipeline.EventTracker(det, dates, kind, time_range=2, method=method, overlap=overlap, distance=900)
           for kind in ("streamers", "overturnings")]
    ref = _run(det, _batches(raw, 2), trs)
    for tr in trs:
        _check(tr, ref, dates)


def test_stream_labels_match_oracle_emu(emu):
    """hand-made case: the oracle's track_events on the polygons and dates of the stream"""
    lat, lon, raw, dates = _record(61, 120, 5)
    det = pipeline.Detector(lat, lon, levels=[2.0], want_pieces=True)
    trs = [pipeline.EventTracker(det, dates, "streamers", time_range=1),
           pipeline.EventTracker(det, dates, "streamers", time_range=2, method="by_distance", distance=800)]
    ref = _run(det, _batches(raw, 2), trs)
    soup, com, step = ref["streamers"]
    ev = pd.DataFrame({"date": pd.to_datetime(dates[step]), "geometry": _soup_polys(soup), "com": list(map(tuple, com))})
    want = P.track_events(ev, time_range=1).label.sort_index().values
    assert np.array_equal(trs[0].labels(), want)
    want = P.track_events(ev, time_range=2, method="by_distance", distance=800).label.sort_index().values
    assert np.array_equal(trs[1].labels(), want)
    assert len(np.unique(want)) < len(want)


def test_stream_tracking_regrowth_counts_batches_once_emu(emu, monkeypatch):
    lat, lon, raw, dates = _record(61, 120, 5)
    tiny = dict(max_jobs=4, seg_cap=64, contour_cap=4, sel_cap=1, pair_cap=16, event_cap=1)
    monkeypatch.setattr(detect, "default_caps", lambda nlat, nlon, add, njobs: dict(tiny, max_jobs=int(njobs)))
    det = pipeline.Detector(lat, lon, levels=[2.0], want_pieces=True)
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=2)
    ref = _run(det, _batches(raw, 2), [tr])
    assert det._grow
    assert tr.cursor == 5 and tr.n_events == len(ref["streamers"][0])
    _check(tr, ref, dates)


def test_stream_tracking_pieces_rerun_counts_batches_once_emu(emu):
    lat, lon, raw, dates = _record(61, 120, 4)
    det = pipeline.Detector(lat, lon, levels=[2.0, -2.0], want_pieces=True)
    for idx in range(2):
        det._slot(2, idx).cap_sr = 1  # the buffers are larger: only the check sees the small capacity
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=1)
    ref = _run(det, _batches(raw, 2), [tr])
    assert "cap_sr" in det._grow
    assert tr.cursor == 4 and tr.n_events == len(ref["streamers"][0])
    _check(tr, ref, dates)


def test_detect_file_trackers_emu(emu, tmp_path):
    from wavebreaking_b200 import io

    lat, lon, raw, dates = _record(61, 120, 5)
    path = str(tmp_path / "pv.npy")
    np.save(path, raw)
    det = pipeline.Detector(lat, lon, levels=[2.0], want_pieces=True)
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=1)
    soups, coms, steps = [], [], []
    for t0, res in io.detect_file(path, lat, lon, batch=2, depth=2, levels=[2.0], want_pieces=True, trackers=[tr]):
        s, c = pipeline.events_soup(res, "streamers", det)
        soups.append(s)
        coms.append(c)
        steps.append(t0 + res.tables["streamers"].job.astype(np.int64))
    ref = {"streamers": (tracking.PolygonSoup.concat(soups), np.concatenate(coms), np.concatenate(steps))}
    _check(tr, ref, dates)


def test_tracker_refusals_emu(emu):
    lat, lon, raw, dates = _record(61, 120, 4)
    det = pipeline.Detector(lat, lon, levels=[2.0], want_pieces=True)
    with pytest.raises(ValueError, match="want_pieces"):
        pipeline.EventTracker(pipeline.Detector(lat, lon, levels=[2.0]), dates, "streamers", time_range=1)
    with pytest.raises(ValueError, match="want_pieces"):
        pipeline.EventTracker(pipeline.Detector(lat, lon, levels=[2.0], want_flags=False, want_pieces=True), dates,
                              "streamers", time_range=1)
    pipeline.EventTracker(pipeline.Detector(lat, lon, levels=[2.0]), dates, "streamers", time_range=1,
                          method="by_distance")  # no polygons needed
    with pytest.raises(ValueError, match="kind"):
        pipeline.EventTracker(det, dates, "ridges", time_range=1)
    with pytest.raises(ValueError, match="not supported as method"):
        pipeline.EventTracker(det, dates, "streamers", time_range=1, method="by_area")
    with pytest.raises(ValueError, match="increase"):
        pipeline.EventTracker(det, dates[::-1], "streamers", time_range=1)
    with pytest.raises(ValueError, match="increase"):
        pipeline.EventTracker(det, np.r_[dates[:2], dates[1:]], "streamers", time_range=1)
    with pytest.raises(ValueError, match="time_range"):
        pipeline.EventTracker(det, dates, "streamers", time_range=None)
    # a Detector on another grid
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=1)
    lat2, lon2 = synthetic.grid_coords(41, 80)
    with pytest.raises(ValueError, match="grid"):
        list(pipeline.Detector(lat2, lon2, levels=[2.0], want_pieces=True).stream([spatial.to_device(raw[:, :41, :80])],
                                                                                  trackers=[tr]))
    assert tr.cursor == 0
    # a by_overlap tracker on a Detector without pieces (the tracker was built for another one)
    with pytest.raises(ValueError, match="want_pieces"):
        list(pipeline.Detector(lat, lon, levels=[2.0]).stream([spatial.to_device(raw)], trackers=[tr]))
    # past the end of the dates array: refused before the batch is submitted, so a climatology of the same stream does
    # not count it either
    clim = pipeline.FlagClimatology(det, np.zeros(8, dtype=np.int32))
    with pytest.raises(ValueError, match="dates array"):
        list(det.stream(_batches(raw[:3], 2) + _batches(raw[:2], 2), depth=1, trackers=[tr], climatology=clim))
    assert tr.cursor == 3 and clim.steps.tolist() == [3]
    tr2 = pipeline.EventTracker(det, dates, "streamers", time_range=1)
    with pytest.raises(ValueError, match="dates array"):
        list(det.stream(_batches(raw[:3], 3) + _batches(raw[:2], 2), depth=2, trackers=[tr2]))
    assert tr2.cursor == 0  # the second batch was refused before the first one was collected
    # no pair in range
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=0.5)
    list(det.stream(_batches(raw, 2), trackers=[tr]))
    assert tr.n_events > 0
    with pytest.raises(ValueError, match="No events detected in the time range"):
        tr.labels()


# ------------------------------------------------------------------------------------------- sharded runs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


NT_SHARD = 7


def _shard_worker(rank, world, port, backend, emu_path, out_dir, time_range, method):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist

    if backend == "nccl":
        torch.cuda.set_device(rank)
    dist.init_process_group(backend, rank=rank, world_size=world)
    from wavebreaking_b200 import _lib, pipeline, sharding, spatial

    if emu_path is not None:
        _lib.use_library(emu_path, "cpu")
    lat, lon, raw, dates = _record(61, 120, NT_SHARD)
    t0, t1 = sharding.shard_range(NT_SHARD, rank, world)
    det = pipeline.Detector(lat, lon, levels=[2.0], want_pieces=True)
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=time_range, method=method, distance=800, t0=t0)
    list(det.stream([spatial.to_device(raw[t:min(t + 2, t1)]) for t in range(t0, t1, 2)], depth=2, trackers=[tr]))
    labels = sharding.finish_tracks(tr)
    np.save(os.path.join(out_dir, "labels_{}.npy".format(rank)), labels)
    dist.barrier()
    dist.destroy_process_group()


def _single_process_labels(time_range, method):
    lat, lon, raw, dates = _record(61, 120, NT_SHARD)
    det = pipeline.Detector(lat, lon, levels=[2.0], want_pieces=True)
    tr = pipeline.EventTracker(det, dates, "streamers", time_range=time_range, method=method, distance=800)
    ref = _run(det, _batches(raw, 2), [tr])
    return _check(tr, ref, dates)


def _run_ranks(backend, emu_path, tmp_path, world, time_range, method):
    import torch.multiprocessing as mp

    mp.spawn(_shard_worker, args=(world, _free_port(), backend, emu_path, str(tmp_path), time_range, method),
             nprocs=world, join=True)
    want = _single_process_labels(time_range, method)
    got = np.concatenate([np.load(tmp_path / "labels_{}.npy".format(r)) for r in range(world)])
    assert np.array_equal(got, want)
    assert len(np.unique(want)) < len(want)


@pytest.mark.parametrize("world,time_range,method", [(2, 3, "by_overlap"), (3, 4, "by_overlap"),
                                                      (3, 3, "by_distance")])
def test_sharded_stream_tracking_gloo(emu, emu_lib, tmp_path, world, time_range, method):
    """time_range longer than a shard (2-4 steps): a tail links into the heads of several later ranks"""
    _run_ranks("gloo", emu_lib, tmp_path, world, time_range, method)


# ------------------------------------------------------------------------------------------- GPU
def _oracle_labels(ref, kind, dates, **kw):
    soup, com, step = ref[kind]
    ev = pd.DataFrame({"date": pd.to_datetime(dates[step]), "geometry": _soup_polys(soup), "com": list(map(tuple, com))})
    return P.track_events(ev, **kw).label.sort_index().values


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(181, 360), (721, 1440)])
def test_stream_tracking_gpu(gpu, shape):
    """48+ hourly steps with CUDA graphs, on separate streams and on a shared stream: labels equal track_columnar on
    the concatenated events_soup output and the oracle"""
    nlat, nlon = shape
    T = 8
    lat, lon = synthetic.grid_coords(nlat, nlon)
    slabs = [spatial.synth_pv(T, nlat, nlon, hour0=500.0 + T * b, hour_step=1.0) for b in range(2)]
    tail = spatial.synth_pv(T - 3, nlat, nlon, hour0=500.0 + 2 * T, hour_step=1.0)
    batches = [slabs[i % 2] for i in range(6)] + [tail]  # every slot sees its buffers 3 times: eager, capture, replay
    ntime = 6 * T + T - 3
    dates = synthetic.time_axis(ntime, 1)
    for shared in (False, True):
        det = pipeline.Detector(lat, lon, levels=[2.0], graphs=True, want_pieces=True)
        trs = [pipeline.EventTracker(det, dates, "streamers", time_range=1),
               pipeline.EventTracker(det, dates, "streamers", time_range=2, overlap=0.2),
               pipeline.EventTracker(det, dates, "streamers", time_range=1, method="by_distance", distance=400),
               pipeline.EventTracker(det, dates, "overturnings", time_range=1)]
        ref = _run(det, batches, trs, depth=2, shared_stream=shared)
        assert det.graph_replays >= 2
        for tr in trs:
            labels = _check(tr, ref, dates)
            assert len(np.unique(labels)) < len(labels)
        if nlat == 181 or not shared:
            memo = {}
            assert np.array_equal(trs[0].labels(), _oracle_labels(ref, "streamers", dates, time_range=1, _memo=memo))
            assert np.array_equal(trs[2].labels(), _oracle_labels(ref, "streamers", dates, time_range=1,
                                                                  method="by_distance", distance=400))


@pytest.mark.gpu
def test_track_append_matches_events_soup_gpu(gpu):
    assert _check_window(721, 1440, 12, T=6) > 0


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_stream_tracking_nccl(gpu, tmp_path):
    _run_ranks("nccl", None, tmp_path, 2, 3, "by_overlap")
