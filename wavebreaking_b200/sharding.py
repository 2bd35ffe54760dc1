"""Time-sharded execution across ranks (one process per GPU, torch.distributed for the plumbing).

Time steps are independent through contours -> indices -> properties -> to_xarray
(utils/index_utils.py:217-258), so every rank owns a contiguous block of the time axis and no data-path
collective is needed.  Three small host-side merges remain (SURVEY.md 8e):

1. ``exp_lon.max()`` is global over all dates (streamer_index.py:106) -> scalar MAX all-reduce;
2. event ids / row indices are global (streamer_index.py:281-283) -> exclusive prefix sum of the per-rank counts;
3. the event tables are gathered to rank 0 in rank (= time) order;
4. ``track_events`` across shard boundaries: a halo of the event table (:func:`track_sharded`), or, for events
   tracked while streaming, the heads of the later shards (:func:`finish_tracks`);
5. flag-frequency climatologies: a SUM all-reduce of the per-rank counters (:func:`reduce_climatology`).
"""

import numpy as np
import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(ntime, rank, world_size):
    """Contiguous block [t0, t1) of the time axis owned by ``rank`` (earlier ranks get the remainder)."""
    base, rem = divmod(int(ntime), int(world_size))
    t0 = rank * base + min(rank, rem)
    return t0, t0 + base + (1 if rank < rem else 0)


def _device_for_collectives():
    if dist.get_backend() == "nccl":
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def global_max(value):
    """MAX of an int over all ranks (the global exp_lon.max() / dlon)."""
    rank, ws = world()
    if ws == 1:
        return int(value)
    t = torch.tensor([int(value)], dtype=torch.int64, device=_device_for_collectives())
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return int(t.item())


def exclusive_offset(count):
    """(offset of this rank, total) for per-rank counts: global event ids = offset + local index."""
    rank, ws = world()
    if ws == 1:
        return 0, int(count)
    t = torch.zeros(ws, dtype=torch.int64, device=_device_for_collectives())
    t[rank] = int(count)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    counts = t.cpu().numpy()
    return int(counts[:rank].sum()), int(counts.sum())


def reduce_climatology(clim):
    """Totals of a ``pipeline.FlagClimatology`` over all ranks, on every rank: ``(counts, steps)``, int64
    ``[ngroups, 3, nlat, nlon]`` and int64 ``[ngroups]``.  Every rank builds its climatology from the same group array
    with ``t0`` = the start of its shard (``shard_range``), so each time step is counted on exactly one rank."""
    rank, ws = world()
    if ws == 1:
        return clim.counts().astype(np.int64), clim.steps
    dev = _device_for_collectives()
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)
        counts = clim._counts.to(device=dev, dtype=torch.int64) & 0xFFFFFFFF  # the int32 storage holds uint32 bits
    else:
        counts = torch.from_numpy(clim.counts().astype(np.int64))
    steps = torch.from_numpy(clim.steps).to(dev)
    dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    dist.all_reduce(steps, op=dist.ReduceOp.SUM)
    return counts.cpu().numpy(), steps.cpu().numpy()


def finish_tracks(tracker):
    """Collective: the labels of the events a ``pipeline.EventTracker`` tracked on this rank, equal to the labels of
    the single-process run over the whole record.  Every rank streams its shard with ``t0 = shard_range(...)[0]``.

    Every rank publishes its head (its events dated within ``time_range`` of the previous shard's last step), links
    the events still in its window (the tail of its shard) to the heads of all later ranks (several of them when
    shards are shorter than ``time_range``), and the cross-shard links are merged by :func:`boundary_labels`.  Raises
    ValueError on every rank when no pair of events was in range.  The near-threshold pairs of the cross-shard links
    are not collected: after a sharded run ``tracker.near`` holds the pairs among the rank's own events only."""
    rank, ws = world()
    tr = tracker
    n = tr.n_events
    off, _ = exclusive_offset(n)
    if tr._head is None:  # the shard ended before its head was complete: all of it is still in the window
        with tr._on_stream():
            tr._head = tr._snapshot(tr._head_size())
    head = dict(tr._head, gid=tr._head["gid"] + off) if tr._head and len(tr._head["keys"]) else None
    heads = _allgather(head)
    W = len(tr._wkeys)
    cross_local, cross_gid = np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    later = [h for h in heads[rank + 1:] if h is not None]
    if W and later:
        local_gid = tr._wgid.copy()
        with tr._on_stream():  # ordered after the last batch's tracking step
            for h in later:
                tr._append_host(h, h["gid"])
            _, links, _ = tr._link(W, W)
        links = links.astype(np.int64).reshape(-1, 2)
        cross_local, cross_gid = local_gid[links[:, 0]], tr._wgid[links[:, 1]]
        with tr._on_stream():
            tr._evict(len(tr._wkeys))
    if sum(_allgather(int(tr.stats["pairs_in_range"]))) == 0:
        raise ValueError("No events detected in the time range: {}".format(tr.time_range))
    links = np.concatenate(tr._links) if tr._links else np.zeros((0, 2), dtype=np.int64)
    return boundary_labels(n, off, links, cross_local, cross_gid)


def gather_frames(frame, dst=0):
    """Concatenate per-rank pandas tables on ``dst`` in rank (= time) order; other ranks get None."""
    import pandas as pd

    rank, ws = world()
    if ws == 1:
        return frame.reset_index(drop=True)
    parts = [None] * ws if rank == dst else None
    dist.gather_object(frame, parts, dst=dst)
    if rank != dst:
        return None
    parts = [p for p in parts if p is not None and len(p)]
    return pd.concat(parts).reset_index(drop=True) if parts else frame.iloc[:0]


def run_sharded(detector, raw_full_or_shard, ntime_total=None, is_shard=False, intensity=None):
    """Run ``detector`` on this rank's block of time steps with the global exp_lon maximum.

    Returns ``(t0, t1, BatchResult)``.  If the maximum of another rank exceeds the local one, the index
    stage is re-run with the global value (rare: every step normally has a full-width contour).
    ``intensity``: a tensor or a pair ``(u, v)`` shaped and stored like the field (an item of ``Detector.stream``'s
    ``intensity``), sliced like it.
    """
    rank, ws = world()
    if is_shard:
        shard = raw_full_or_shard
        t0, t1 = shard_range(ntime_total, rank, ws)
    else:
        t0, t1 = shard_range(raw_full_or_shard.shape[0], rank, ws)
        shard = raw_full_or_shard[t0:t1]
    item = None
    if intensity is not None:
        item = tuple(intensity) if isinstance(intensity, (tuple, list)) else (intensity,)
        if not is_shard:
            item = tuple(f[t0:t1] for f in item)
    res = detector.run_batch(shard, intensity=item)
    g = global_max(res.gmax_nx)
    if g != res.gmax_nx:
        res = detector.run_batch(shard, gmax_nx=g, intensity=item)
    return t0, t1, res


def _allgather(obj):
    rank, ws = world()
    if ws == 1:
        return [obj]
    out = [None] * ws
    dist.all_gather_object(out, obj)
    return out


def track_sharded(dates, method="by_overlap", soup=None, com=None, time_range=None, overlap=0, distance=1000,
                  stats=None):
    """``track_events`` labels for time-sharded event tables (events.py:113-241) without gathering the tables.

    Every rank passes the events of its own contiguous block of the time axis, sorted by date (columnar:
    ``dates`` plus a :class:`tracking.PolygonSoup` or the ``com`` array).  The reference links an event at t to the
    events in (t, t + time_range], so a rank only needs, besides its own events, the events of the first
    ``time_range`` hours of the following shard(s): that *halo of the event table* is the only bulk exchange.
    Linking then runs locally (same kernels as the single-process path); the cross-shard links are merged by a
    union-find over the few components that touch a shard boundary, and the dense labels (rank of the smallest
    member index, events.py:228-238) follow from an exclusive scan of the per-rank root counts.

    Returns the labels of the local events; they are identical to ``tracking.track_columnar`` on the concatenated
    table.  Raises ValueError on every rank when no pair of events is in range.
    """
    from . import tracking

    rank, ws = world()
    dates = np.asarray(dates)
    n = len(dates)
    keys, window = tracking.time_keys(dates)
    if n > 1 and np.any(np.diff(keys) < 0):
        raise ValueError("track_sharded expects the local events sorted by date")
    off, total = exclusive_offset(n)
    # ---- shard summaries: first / last key, smallest positive local difference
    dk = np.diff(keys) if n > 1 else np.zeros(0, dtype=keys.dtype)
    pos = dk[dk > 0]
    info = _allgather(dict(n=n, first=keys[0] if n else None, last=keys[-1] if n else None,
                           mind=pos.min() if len(pos) else None))
    if time_range is None:
        # events.py:155-157 on the whole table: consecutive differences inside and across the shards
        cands = [i["mind"] for i in info if i["mind"] is not None]
        prev = None
        for i in info:
            if i["n"]:
                if prev is not None and i["first"] - prev > 0:
                    cands.append(i["first"] - prev)
                prev = i["last"]
        if not cands:
            raise ValueError("No events detected in the time range: {}".format(time_range))
        dmin = min(cands)
        time_range = float(tracking._hours_of(dmin)) if keys.dtype == np.int64 else float(dmin)
    win = window(time_range)
    # ---- halo: the head of every shard (events within `win` of the end of an earlier shard), published once
    prev_last = [i["last"] for i in info[:rank] if i["n"]]
    head = None
    if n and prev_last:
        m = int(np.searchsorted(keys, max(prev_last) + win, side="right"))
        if m:
            idx = np.arange(m)
            head = dict(keys=keys[:m], gid=off + idx, soup=soup.take(idx) if soup is not None else None,
                        com=np.asarray(com)[:m] if com is not None else None)
    heads = _allgather(head)
    ext_keys, ext_gid, ext_soups, ext_com = [keys], [off + np.arange(n)], [soup], [np.asarray(com) if com is not None else None]
    if n:
        for q in range(rank + 1, ws):
            h = heads[q]
            if h is None:
                continue
            m = int(np.searchsorted(h["keys"], keys[-1] + win, side="right"))
            if m == 0:
                continue
            ext_keys.append(h["keys"][:m])
            ext_gid.append(h["gid"][:m])
            if soup is not None:
                ext_soups.append(h["soup"].take(np.arange(m)))
            if com is not None:
                ext_com.append(h["com"][:m])
    k_all = np.concatenate(ext_keys)
    g_all = np.concatenate(ext_gid).astype(np.int64)
    s_all = tracking.PolygonSoup.concat(ext_soups) if soup is not None else None
    c_all = np.concatenate(ext_com) if com is not None else None
    # ---- local linking: pairs (i, j) with i owned by this rank
    if n:
        links, n_in_range, near = tracking.link_events(k_all, win, method, s_all, c_all, overlap, distance, first=0,
                                                       last=n, stats=stats)
    else:
        links, n_in_range = np.zeros((0, 2), dtype=np.int64), 0
    tot_in_range = sum(_allgather(int(n_in_range)))
    if tot_in_range == 0:
        raise ValueError("No events detected in the time range: {}".format(time_range))
    links = np.asarray(links, dtype=np.int64).reshape(-1, 2)
    cross = links[links[:, 1] >= n]
    return boundary_labels(n, off, links[links[:, 1] < n], cross[:, 0], g_all[cross[:, 1]])


def boundary_labels(n, off, inner, cross_local, cross_gid):
    """Collective: dense labels of this rank's ``n`` events (global ids ``off`` .. ``off + n - 1``) from the links among
    them (``inner``, local index pairs) and the links from local event ``cross_local[k]`` to the event with global id
    ``cross_gid[k]`` of a later rank.  Equal to ``tracking.labels_from_links`` on the whole record."""
    from . import tracking

    rank, ws = world()
    inner = np.asarray(inner, dtype=np.int64).reshape(-1, 2)
    cross_local = np.asarray(cross_local, dtype=np.int64)
    cmin = off + tracking.component_min(n, inner)  # global id of the smallest member of the local component
    cross_edges = (np.c_[cmin[cross_local], np.asarray(cross_gid, dtype=np.int64)] if len(cross_local)
                   else np.zeros((0, 2), dtype=np.int64))
    # ---- merge: resolve the far end of every cross link to ITS local component, then union-find on the few
    #      boundary components (every rank holds the same tiny graph)
    all_cross = np.concatenate([c for c in _allgather(cross_edges) if len(c)] or [np.zeros((0, 2), dtype=np.int64)])
    mine = (all_cross[:, 1] >= off) & (all_cross[:, 1] < off + n)
    resolved = np.c_[all_cross[mine, 0], cmin[all_cross[mine, 1] - off]] if mine.any() else np.zeros((0, 2), dtype=np.int64)
    graph = np.concatenate([c for c in _allgather(resolved) if len(c)] or [np.zeros((0, 2), dtype=np.int64)])
    gmin_of = {}
    if len(graph):
        nodes, inv = np.unique(graph, return_inverse=True)
        comp_min = tracking.component_min(len(nodes), inv.reshape(-1, 2))
        gmin_of = {int(a): int(nodes[b]) for a, b in zip(nodes, comp_min)}
    gmin = np.array([gmin_of.get(int(c), int(c)) for c in cmin], dtype=np.int64) if n else np.zeros(0, dtype=np.int64)
    # ---- dense labels: rank of the component's smallest member among all components
    roots = np.unique(gmin[(gmin >= off) & (gmin < off + n)]) if n else np.zeros(0, dtype=np.int64)
    counts = _allgather(len(roots))
    base = int(sum(counts[:rank]))
    label_of_root = {int(r): base + k for k, r in enumerate(roots)}
    boundary_roots = {g for g in gmin_of.values()}
    published = _allgather({r: l for r, l in label_of_root.items() if r in boundary_roots})
    for d in published:
        label_of_root.update(d)
    return np.array([label_of_root[int(g)] for g in gmin], dtype=np.int64) if n else np.zeros(0, dtype=np.int64)
