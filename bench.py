#!/usr/bin/env python
"""Benchmark of the per-time-step detection path (BASELINE.json: "time steps/sec, 0.25 deg hourly PV
2-PVU detection").

One *step* = one batch of ``--batch`` hourly time steps of the ERA5-shaped synthetic PV field
(721 x 1440, float32) through smoothing (5 passes) -> contours at 2 PVU -> streamers + overturnings +
cutoffs (+ properties) -> the three to_xarray flag grids.  ``value`` is time steps/s with the raw field
already resident in HBM; ``e2e`` is the same through ``Detector.stream`` with the raw field in pinned host
memory (H2D inside the timed region) and the flag grids (bit-packed) + event tables copied back.

  python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1: time steps are sharded
                                                            over ranks, no data-path collective)
  python bench.py --impl reference ...                      (the CPU oracle on all host cores)
  python bench.py --workload decade-track --hours H ...     (detection of H consecutive hours sharded over the
                                                            ranks + track_events(by_overlap) across the shard
                                                            boundaries; BASELINE.json configs[4])
  python bench.py ... --dump-outputs DIR                    (also write what the last timed batch returned as
                                                            DIR/<name>.npy, see dump_outputs)

The benchmark writes nothing into the source tree (no bytecode caches either), so it runs from a read-only checkout.
"""

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the package modules imported below leave no __pycache__ in the tree

METRIC = "time steps/sec, 0.25deg hourly PV 2-PVU detection (streamers+overturnings+cutoffs+to_xarray)"
UNIT = "time steps/s"


def log(*a):
    """progress on stderr (stdout carries only the JSON line)"""
    print("[bench {:7.1f}s]".format(time.perf_counter() - _T0), *a, file=sys.stderr, flush=True)


_T0 = time.perf_counter()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default: 100 (b200) / 2 (reference)")
    ap.add_argument("--warmup", type=int, default=None, help="default: 3 (b200) / 1 (reference)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=296, help="time steps per step (2 per SM)")
    ap.add_argument("--nlat", type=int, default=721)
    ap.add_argument("--nlon", type=int, default=1440)
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--cpu-sample", type=int, default=3, help="time steps of the CPU baseline sample (~4-8 s each)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--depth", type=int, default=6, help="batches in flight in the device-resident leg (slots / streams)")
    ap.add_argument("--serial", action="store_true", help="device-resident leg on ONE stream (no kernel overlap)")
    ap.add_argument("--no-graphs", action="store_true", help="eager launches instead of one CUDA graph per batch")
    ap.add_argument("--no-extras", action="store_true", help="skip the stress line, the e2e variants and the link test")
    ap.add_argument("--workload", default="c25", choices=["c25", "decade-track"])
    ap.add_argument("--hours", type=int, default=None, help="decade-track: consecutive hours (default 8760 per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0)")
    a = ap.parse_args()
    if a.dump_outputs is not None and (a.impl != "b200" or a.workload != "c25"):
        ap.error("--dump-outputs applies to the default workload of the CUDA path (--impl b200 --workload c25)")
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.steps is None:
        a.steps = 100 if a.impl == "b200" else 2
    if a.warmup is None:
        a.warmup = 3 if a.impl == "b200" else 1
    return a


def workload_config(a):
    return {
        "workload": "synthetic ERA5-shaped 0.25deg ({}x{}) hourly PV, level 2 PVU, smoothing {} passes, "
                    "streamer+overturning+cutoff + to_xarray x3".format(a.nlat, a.nlon, a.passes),
        "l2": "inputs larger than L2: every step streams its own batch of hundreds of time steps (4.15 MB each) "
              "through the 126 MB L2",
        "parallelism": "time steps sharded over ranks, no collective",
    }


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clock / throttle sampler running while the timed region executes."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Samples before this point (warm-up) are ignored."""
        self.lines = []

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ roofline
def algorithmic_bytes(kernel, a, stats):
    """Algorithmic bytes ONE launch of `kernel` moves for a batch of a.batch time steps (DESIGN.md)."""
    cells = a.nlat * a.nlon
    T = a.batch
    per_step = {
        "smooth_fused": cells * (4 + 8),                       # float32 in, float64 out, independent of passes
        # bit planes (16 B per 54-cell strip row) + 4 corner doubles and 20 B per segment
        "ms_segments": 16 * a.nlat * ((a.nlon + 53) // 54) + 52 * stats["segments"],
        "contour_link": 20 * stats["segments"] + 4 * stats["points"],
        "events_raster": 3 * cells,                              # the three int8 flag grids
        "pair_scan": 48 * stats["points"],
        "streamer_cascade": 8 * stats["pairs"] + 4 * stats["points"],
        "streamer_prep": 20 * stats["points"],
        "overturning": 4 * stats["points"],
    }
    return per_step.get(kernel, 0) * T


def measured_traffic(kernel, batch):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return int(json.load(f)[kernel]["bytes_per_time_step"] * batch)
    except Exception:
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ CPU arms
def _oracle_step(raw, nlat, nlon, hours, passes):
    from oracle import pipeline as P
    from wavebreaking_b200 import synthetic

    lat, lon = synthetic.grid_coords(nlat, nlon)
    t0 = np.datetime64("2000-01-01T00", "ns")
    tm = t0 + (np.asarray(hours) * 3600 * 10**9).astype("timedelta64[ns]")
    grid = P.Grid(lon, lat, tm)
    out = P.detect_steps(raw, grid, levels=[2.0], passes=passes)
    return {k: len(v) for k, v in out["events"].items()}


def _ref_prepare(args):
    idx, nlat, nlon, tmpdir = args
    from wavebreaking_b200 import synthetic

    f = synthetic.pv_field(nlat, nlon, [float(idx)])
    np.save(os.path.join(tmpdir, "{}.npy".format(idx)), f)
    return idx


def _ref_process(args):
    idx, nlat, nlon, tmpdir, passes = args
    raw = np.load(os.path.join(tmpdir, "{}.npy".format(idx)))
    return _oracle_step(raw, nlat, nlon, [float(idx)], passes)


def run_reference(a):
    """--impl reference: the oracle (a restatement of the reference's CPU implementation that calls the same
    scipy / sklearn routines; the real package cannot be installed in this image) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import tempfile

    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 64))
    per_step = workers  # one time step per worker and step: a bounded sample of the workload
    total = (a.steps + a.warmup) * per_step
    tmpdir = tempfile.mkdtemp(prefix="wbk_ref_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    ctx = mp.get_context("fork")
    with ctx.Pool(workers) as pool:
        pool.map(_ref_prepare, [(i, a.nlat, a.nlon, tmpdir) for i in range(total)])
        for w in range(a.warmup):
            pool.map(_ref_process, [(w * per_step + i, a.nlat, a.nlon, tmpdir, a.passes) for i in range(per_step)])
        t0 = time.perf_counter()
        for s in range(a.steps):
            base = (a.warmup + s) * per_step
            pool.map(_ref_process, [(base + i, a.nlat, a.nlon, tmpdir, a.passes) for i in range(per_step)])
        dt = time.perf_counter() - t0
    for f in os.listdir(tmpdir):
        os.remove(os.path.join(tmpdir, f))
    os.rmdir(tmpdir)
    value = a.steps * per_step / dt
    cfg = workload_config(a)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1000.0 * dt / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg, "time_steps_per_step": per_step,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port",
                         "sample": "{} time steps per step, one per worker process; the real wavebreaking package "
                                   "is not installable here (xarray/geopandas/shapely/skimage absent), so the "
                                   "oracle port (same scipy/sklearn calls) is timed".format(per_step)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def cpu_baseline(a, raw_host, hours):
    n = raw_host.shape[0]
    # one untimed step first: imports, scipy / sklearn first-call setup, page faults of the N x N temporaries
    _oracle_step(raw_host[:1], a.nlat, a.nlon, hours[:1], a.passes)
    t0 = time.perf_counter()
    for i in range(n):
        _oracle_step(raw_host[i:i + 1], a.nlat, a.nlon, hours[i:i + 1], a.passes)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "first {} time steps of the benchmark input, single process, after one untimed warm-up step "
                      "({:.1f} s)".format(n, dt)}


# ------------------------------------------------------------------------------------------------ output dump
DUMP_SEED = 20260101
# row caps of the dumped arrays: larger outputs are replaced by a fixed, seeded sample of their rows (sorted, so that
# the order of the rows is kept).  Worst case in all: 12.6 + 2.6 + 16.8 + 3 x 4.5 + 2 x 4.5 + 0.2 MB < 64 MB
DUMP_CAPS = {"flags_sample": 3 << 20, "contours": 1 << 16, "contour_points": 1 << 21, "events": 1 << 15,
             "ring_points": 1 << 19, "ring_sizes": 1 << 15, "near": 1 << 12}
DUMP_MAX_BYTES = 64 * 10**6


def _sample_rows(n, cap):
    """Row indices kept of an array of n rows: all of them, or `cap` drawn with DUMP_SEED (same n -> same rows)."""
    if n <= cap:
        return None
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, cap, replace=False))


def dump_outputs(res, out_dir):
    """Write what the detection path returned for one batch (a pipeline.BatchResult) as out_dir/<name>.npy, float32
    where the values are exact in it and float64 otherwise, at most DUMP_MAX_BYTES in all:

      flags_sample        float32 [<= 3 Mi]   int8 flag grids [3, T, nlat, nlon] (streamers, overturnings, cutoffs) at
                                              sorted flat cell indices drawn with DUMP_SEED (all cells if there are few)
      contours            float64 [C, 5]      job (time step * levels + level), closed, nx (exp_lon in columns), sum_y,
                                              number of vertices
      contour_points      float32 [P, 2]      x, y of every contour vertex (index coordinates of the extended grid)
      <kind>_events       float64 [n, 17]     job, contour, ind1, ind2, box x0 y0 x1 y1, orientation, split, near,
                                              sums (area, area x data, area x intensity, area x x, area x y, members)
      <kind>_ring_sizes   float64 [n]         vertices of each event ring (streamers, cutoffs)
      <kind>_ring_points  float32 [m, 2]      x, y of the ring vertices
      near                float64 [k, 6]      streamer pairs decided within 1e-9 of a threshold (BatchResult.near)
      counts              float64 [8]         time steps, contours, contour vertices, streamers, overturnings, cutoffs,
                                              events that straddle the last meridian, near pairs (BatchResult.near_total)

    Arrays longer than their DUMP_CAPS entry keep a seeded sample of their rows.  An array without rows (no near pairs,
    no events of a kind) is not written: `counts` holds its length.  Returns the bytes written."""
    import torch

    from wavebreaking_b200 import detect

    os.makedirs(out_dir, exist_ok=True)
    arrays = {}

    def put(name, arr, cap_key, dtype):
        arr = np.asarray(arr)
        keep = _sample_rows(len(arr), DUMP_CAPS[cap_key])
        arrays[name] = np.ascontiguousarray((arr if keep is None else arr[keep]).astype(dtype))

    flat = res.flags.reshape(-1)
    keep = _sample_rows(flat.numel(), DUMP_CAPS["flags_sample"])
    if keep is not None:  # gathered where the grids are: those of a benchmark batch take about 1 GB
        flat = flat[torch.from_numpy(keep).to(flat.device)]
    put("flags_sample", flat.cpu().numpy(), "flags_sample", np.float32)

    h = res.contours.host()
    put("contours", np.c_[h["job"], h["closed"], h["nx"], h["sum_y"], np.diff(h["pt_off"])], "contours", np.float64)
    put("contour_points", np.c_[h["x"], h["y"]], "contour_points", np.float32)
    for kind in detect.KINDS:
        t = res.tables[kind]
        cols = np.c_[t.job, t.contour, t.ind1, t.ind2, t.box, t.orientation, t.split, t.near].astype(np.float64)
        put(kind + "_events", np.c_[cols, t.sums].reshape(len(t), 17), "events", np.float64)
        if t.rings is not None:
            put(kind + "_ring_sizes", np.diff(t.rings.off), "ring_sizes", np.float64)
            p = t.rings.packed
            put(kind + "_ring_points", np.c_[p & 0xFFFF, p >> 16], "ring_points", np.float32)
    put("near", res.near.reshape(-1, 6), "near", np.float64)
    arrays = {k: v for k, v in arrays.items() if v.size}
    arrays["counts"] = np.array([res.ntime, res.contours.ncontours, res.contours.npoints, *res.counts, res.n_split,
                                 res.near_total], dtype=np.float64)

    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("output dump of {} bytes exceeds {} (DUMP_CAPS)".format(total, DUMP_MAX_BYTES))
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    return total


# ------------------------------------------------------------------------------------------------ GPU arm
def _setup_ranks():
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def _max_over_ranks(ms, world):
    import torch
    import torch.distributed as dist

    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def link_test(nbytes_up, nbytes_down, reps=5):
    """Concurrent pinned host -> device and device -> host copies of the sizes one e2e step moves, on two streams:
    the ceiling of the host link for this rank while all other ranks do the same (GB/s each way)."""
    import torch

    up_h = torch.empty(nbytes_up, dtype=torch.uint8, pin_memory=True)
    up_d = torch.empty(nbytes_up, dtype=torch.uint8, device="cuda")
    dn_h = torch.empty(max(nbytes_down, 1), dtype=torch.uint8, pin_memory=True)
    dn_d = torch.empty(max(nbytes_down, 1), dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    with torch.cuda.stream(s1):
        up_d.copy_(up_h, non_blocking=True)
        e[0].record()
        for _ in range(reps):
            up_d.copy_(up_h, non_blocking=True)
        e[1].record()
    with torch.cuda.stream(s2):
        dn_h.copy_(dn_d, non_blocking=True)
        e[2].record()
        for _ in range(reps):
            dn_h.copy_(dn_d, non_blocking=True)
        e[3].record()
    torch.cuda.synchronize()
    return (reps * nbytes_up / (e[0].elapsed_time(e[1]) / 1e3) / 1e9,
            reps * nbytes_down / (e[2].elapsed_time(e[3]) / 1e3) / 1e9)


def run_b200(a):
    import torch
    import torch.distributed as dist

    from wavebreaking_b200 import _lib, detect, pipeline, spatial, synthetic

    world, rank, local = _setup_ranks()
    lib = _lib.get()
    lat, lon = synthetic.grid_coords(a.nlat, a.nlon)
    graphs = not a.no_graphs
    det = pipeline.Detector(lat, lon, levels=[2.0], passes=a.passes, graphs=graphs)
    T, K, W = a.batch, a.steps, a.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # inputs: every step (and rank) gets its own slab of consecutive hours, generated in HBM (untimed)
    # (a few distinct slabs are cycled: each is far larger than the 126 MB L2, so nothing is reused from cache)
    nslab = min(K + W, 4)
    slabs = []
    for s in range(nslab):
        hour0 = float((rank * nslab + s) * T)
        slabs.append(spatial.synth_pv(T, a.nlat, a.nlon, hour0=hour0, hour_step=1.0))
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    depth = n_resident = a.depth

    def timed_region(detector, inputs, k_steps, shared_stream, profile, depth=depth):
        """k_steps batches, `depth` in flight; returns (ms, per-kernel profile, kernel launches, per-batch counts,
        result of the last batch: valid until the detector runs again)."""
        n_in = len(inputs)
        # warm-up: every slot allocates its arenas on first use, and every (slot, buffer) combination is captured
        # into its CUDA graph on its second submission
        warm = max(W, 3 * depth * (n_in // math.gcd(n_in, depth)) if detector.graphs else 2 * depth)
        for res in detector.stream((inputs[s % n_in] for s in range(warm)), depth=depth, shared_stream=shared_stream):
            pass
        barrier()
        launches0 = lib.cdll.wbk_launch_count()
        g0 = detector.graph_kernel_launches
        lib.cdll.wbk_prof_reset()
        lib.cdll.wbk_prof_enable(1 if profile else 0)
        sampler.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        cnts = []
        for res in detector.stream((inputs[(warm + s) % n_in] for s in range(k_steps)), depth=depth,
                                   shared_stream=shared_stream):
            cnts.append(pipeline.summarize(res))
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1000.0
        e1.record()
        barrier()
        lib.cdll.wbk_prof_enable(0)
        launches = lib.cdll.wbk_launch_count() - launches0 + detector.graph_kernel_launches - g0
        # batches run on side streams: the host clock bounds the region
        return max(e0.elapsed_time(e1), wall_ms), (_lib.prof_read(lib) if profile else {}), launches, cnts, res

    # ---- headline region (value): every slot on its own stream, one CUDA graph per batch, so the latency-bound
    #      kernels of one batch overlap the FP64-bound smoothing of another
    log("inputs ready; device-resident leg")
    ms, _, launches, counts, last = timed_region(det, slabs, K, shared_stream=a.serial, profile=False)
    clocks = sampler.stop()
    log("device-resident leg done: {:.1f} ms for {} batches".format(ms, K))
    if a.dump_outputs is not None and rank == 0:
        nbytes = dump_outputs(last, a.dump_outputs)
        log("outputs of the last timed batch: {:.1f} MB in {}".format(nbytes / 1e6, a.dump_outputs))
    del last
    ms_max = _max_over_ranks(ms, world)
    value = world * K * T / (ms_max / 1000.0)
    # ---- the same batches on ONE stream with eager launches and CUDA events around every kernel: clean per-kernel
    #      durations for the roofline; its throughput is reported as value_single_stream
    det_prof = pipeline.Detector(lat, lon, levels=[2.0], passes=a.passes, graphs=False)
    k_prof = min(K, 20)
    sampler = ClockSampler(local)
    ms_ser, prof, _, counts_ser, _ = timed_region(det_prof, slabs, k_prof, shared_stream=True, profile=True, depth=min(depth, 3))
    value_serial = world * k_prof * T / (_max_over_ranks(ms_ser, world) / 1000.0)

    # per-time-step work statistics (device counters of the batches) for the algorithmic byte counts
    stats = {k: float(np.mean([c[k] for c in counts])) / T for k in ("points", "segments", "pairs")}

    # ---- roofline of the dominant kernel
    peak, peak_src = peaks()
    roof = None
    if prof:
        dom = max(prof.items(), key=lambda kv: kv[1][1])
        name, (n_l, tot_ms) = dom
        avg_ms = tot_ms / n_l
        by = algorithmic_bytes(name, a, stats)
        achieved = by / (avg_ms / 1000.0) / 1e9 if avg_ms > 0 else 0.0
        tot = sum(x[1] for x in prof.values())
        roof = {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": measured_traffic(name, a.batch), "peak_source": peak_src,
                "avg_launch_ms": avg_ms, "launches": n_l, "algorithmic_bytes_per_launch": by,
                "kernel_ms_share": {k: round(v[1] / tot, 4) for k, v in prof.items()},
                "kernel_us_per_time_step": {k: round(1000.0 * v[1] / v[0] / T, 3) for k, v in prof.items()},
                "device_busy_frac": tot / ms_ser,
                "measured_in": "second timed region: {} of the same batches on ONE CUDA stream with eager launches "
                               "(value_single_stream); the headline region replays one CUDA graph per batch on {} "
                               "streams".format(k_prof, n_resident),
                "note": "smooth_fused (wbk_smooth_impl.cuh) is bounded by the FP64 pipe before HBM: 5 passes x 7 DP ops "
                        "per cell on 64-column strips with a 5-column halo = 2.5 us per 721x1440 step at 64 DP "
                        "lanes/clk/SM, HBM floor 1.9 us (DESIGN.md 4)"}
    det_prof.close()
    # the later legs keep three batches in flight: release the slots of the device-resident leg (arenas, smoothed
    # fields and flag grids of `depth` batches) so that they run without memory pressure
    det.close()
    det = pipeline.Detector(lat, lon, levels=[2.0], passes=a.passes, graphs=graphs)
    torch.cuda.empty_cache()
    log("single-stream profile leg done (peak device memory {:.1f} GB)".format(torch.cuda.max_memory_allocated() / 1e9))

    # ---- end-to-end leg (host buffers): float32 field in pinned host memory -> bit-packed flag grids + tables
    #      (three batches in flight: the leg is bound by the host link, more slots only pin more host memory)
    e2e = None
    extras = {}
    depth = min(depth, 3)
    if not a.no_e2e:
        ncells = 3 * T * a.nlat * a.nlon
        host_in = [torch.empty((T, a.nlat, a.nlon), dtype=torch.float32, pin_memory=True) for _ in range(depth)]
        for i, h in enumerate(host_in):
            h.copy_(slabs[i % nslab])
        packed_host = [torch.empty(pipeline.packed_nbytes(ncells), dtype=torch.uint8, pin_memory=True) for _ in range(depth)]
        torch.cuda.synchronize()

        def e2e_region(detector, inputs, k_steps, **kw):
            warm = max(min(W, depth), 3 * depth if detector.graphs else 0)
            for r in detector.stream((inputs[s % depth] for s in range(warm)), depth=depth, **kw):
                pass
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_wall = time.perf_counter()
            e0.record()
            tab_bytes = 0
            for r in detector.stream((inputs[s % depth] for s in range(k_steps)), depth=depth, **kw):
                tab_bytes = sum(t.sums.nbytes + 11 * 4 * len(t) for t in r.tables.values()) \
                    + sum(t.rings.nbytes for t in r.tables.values() if t.rings is not None)
            torch.cuda.synchronize()
            e1.record()
            barrier()
            wall = time.perf_counter() - t_wall
            ems = _max_over_ranks(max(e0.elapsed_time(e1), wall * 1000.0), world)
            return world * k_steps * T / (ems / 1000.0), int(tab_bytes)

        log("e2e leg")
        v, tab_bytes = e2e_region(det, host_in, K, packed_host=packed_host)
        log("e2e leg done: {:.0f} steps/s".format(v))
        h2d, d2h = T * a.nlat * a.nlon * 4, packed_host[0].numel() + tab_bytes
        e2e = {"value": v, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(d2h),
               "result": "bit-packed flag grids (1 bit per cell, pipeline.unpack_flags) + event tables + ring vertices"}
        if not a.no_extras:
            # host link ceiling with all ranks copying at once, and what fraction of it the e2e leg reaches
            up, dn = link_test(h2d, int(d2h))
            up = -_max_over_ranks(-up, world)   # the slowest rank
            dn = -_max_over_ranks(-dn, world)
            per_rank = v / world / T * h2d / 1e9  # GB/s of field upload per rank (h2d is bytes per batch of T steps)
            e2e["roofline"] = {"bound": "host link (PCIe), H2D of the float32 field", "h2d_gbs_concurrent": up,
                               "d2h_gbs_concurrent": dn, "achieved_h2d_gbs": per_rank, "frac": per_rank / up,
                               "note": "measured in this run: every rank copies one step's bytes up and down at the "
                                       "same time on two streams (slowest rank)"}
            k_var = max(3, min(K, 20))
            # round-1 definition: dense int8 flag grids on the wire
            flags_host = [torch.empty((3, T, a.nlat, a.nlon), dtype=torch.int8, pin_memory=True) for _ in range(depth)]
            log("link test: {:.1f} / {:.1f} GB/s; e2e variants".format(up, dn))
            v8, _ = e2e_region(det, host_in, k_var, flags_host=flags_host)
            extras["e2e_int8_flags"] = {"value": v8, "unit": UNIT, "d2h_bytes_per_step": int(ncells + tab_bytes)}
            del flags_host
            # ERA5 files hold packed shorts: int16 field on the wire, decoded inside the smoothing loads
            lo, hi = float(slabs[0].min()), float(slabs[0].max())
            scale, offset = (hi - lo) / 65000.0, (hi + lo) / 2.0
            det16 = pipeline.Detector(lat, lon, levels=[2.0], passes=a.passes, graphs=graphs, packing=(scale, offset, None))
            host16 = [torch.empty((T, a.nlat, a.nlon), dtype=torch.int16, pin_memory=True) for _ in range(depth)]
            for i, h in enumerate(host16):
                h.copy_(torch.round((slabs[i % nslab].double() - offset) / scale).to(torch.int16))
            v16, _ = e2e_region(det16, host16, k_var, packed_host=packed_host)
            extras["e2e_int16_input"] = {"value": v16, "unit": UNIT, "h2d_bytes_per_step": T * a.nlat * a.nlon * 2,
                                         "note": "CF-packed shorts (scale_factor / add_offset) decoded to float64 in the "
                                                 "smoothing loads, as xarray decodes ERA5 NetCDF; not the float32 workload "
                                                 "of `value` / `e2e`"}
            det16.close()
            del host16

    # ---- the same workload through the drop-in API (reference call sequence on a Field of T time steps in ordinary,
    #      pageable host memory): smoothed field -> contours -> three indices -> three to_xarray grids read on the host
    if not a.no_extras and not a.no_e2e:
        import wavebreaking_b200 as wb
        from wavebreaking_b200 import compat

        det.close()
        torch.cuda.empty_cache()
        log("e2e through the drop-in API")
        tt = np.datetime64("2000-01-01T00", "ns") + np.arange(T) * np.timedelta64(3600 * 10**9, "ns")
        host_nps = [slabs[i % nslab].cpu().numpy() for i in range(3)]  # a different host array per pass: no reuse

        def api_pass(k=0):
            pv = compat.Field(host_nps[k % 3], ("time", "lat", "lon"), {"time": tt, "lat": lat, "lon": lon}, name="PV")
            sm = wb.calculate_smoothed_field(pv, a.passes)
            contours = wb.calculate_contours(sm, 2, original_coordinates=False)
            evs = [fn(sm, 2, contours=contours) for fn in (wb.calculate_streamers, wb.calculate_overturnings, wb.calculate_cutoffs)]
            grids = [np.asarray(wb.to_xarray(sm, ev).values) for ev in evs]
            return sum(len(ev) for ev in evs), grids

        api_pass(0)
        torch.cuda.synchronize()
        n_api = 3
        t_api = time.perf_counter()
        grids = None
        for k in range(n_api):
            del grids  # a user loop drops the previous result: its page-locked host blocks are recycled
            nev, grids = api_pass(k + 1)
        torch.cuda.synchronize()
        dt_api = _max_over_ranks((time.perf_counter() - t_api) * 1000.0, world) / 1000.0
        ncell = int(sum(np.count_nonzero(g) for g in grids))  # a check of the host grids, outside the timed region
        del grids
        extras["e2e_api"] = {"value": world * n_api * T / dt_api, "unit": UNIT, "events_per_pass": nev, "flagged_cells": ncell,
                             "calls": "calculate_smoothed_field -> calculate_contours -> calculate_streamers / overturnings / "
                                      "cutoffs(contours=) -> to_xarray x3 on a Field of {} time steps (pageable host memory in, "
                                      "frames + int8 grids on the host out)".format(T)}
        del host_nps
        log("e2e through the drop-in API done: {:.0f} steps/s".format(extras["e2e_api"]["value"]))

    # ---- stress line: a noisier field with 2-4x the contour points (SURVEY.md 8: real ERA5 sits there)
    if not a.no_extras:
        g = torch.Generator(device="cuda").manual_seed(20260101 + rank)
        noisy = []
        for sl in slabs[:2]:
            noise = torch.randn(sl.shape, generator=g, device="cuda", dtype=torch.float32)
            noisy.append(sl + 1.5 * noise)
        del noise
        k_st = max(3, min(K, 12))
        log("stress line")
        # (arenas grow to ~25 GB per slot on this field: three batches in flight)
        det.close()
        det = pipeline.Detector(lat, lon, levels=[2.0], passes=a.passes, graphs=graphs)
        ms_st, _, _, cnt_st, _ = timed_region(det, noisy, k_st, shared_stream=a.serial, profile=False, depth=min(n_resident, 3))
        det.close()
        log("stress line done")
        extras["stress"] = {"value": world * k_st * T / (_max_over_ranks(ms_st, world) / 1000.0), "unit": UNIT,
                            "recipe": "benchmark field + 1.5 PVU white noise per cell (before the 5 smoothing passes)",
                            "per_time_step": {k: float(np.mean([c[k] for c in cnt_st])) / T for k in
                                              ("points", "segments", "pairs", "contours", "streamers", "overturnings", "cutoffs")}}
        del noisy

    # ---- CPU baseline (rank 0, single GPU runs only)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        n = min(a.cpu_sample, T)
        raw_host = slabs[0][:n + 1].cpu().numpy()
        hours = np.arange(n + 1, dtype=np.float64)
        log("cpu baseline")
        cpu = cpu_baseline(a, raw_host[1:], hours[1:])

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "time_steps_per_step": T, "value_single_stream": value_serial,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(a), "clocks": clocks,
            "e2e": e2e, "gpu_launches": int(launches), "cuda_graphs": graphs, "roofline": roof, "cpu_baseline": cpu,
            "per_time_step": {k: float(np.mean([c[k] for c in counts])) / T
                              for k in ("streamers", "overturnings", "cutoffs", "contours", "split", "points", "segments",
                                        "pairs", "near")},
        }
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ decade + tracking
def run_decade_track(a):
    """BASELINE.json configs[4]: detection + to_xarray of consecutive hours sharded over the ranks, then
    track_events(by_overlap) on the streamers across the shard boundaries (halo of the event table)."""
    import torch
    import torch.distributed as dist

    from wavebreaking_b200 import _lib, pipeline, sharding, spatial, synthetic, tracking

    world, rank, local = _setup_ranks()
    lib = _lib.get()
    hours = a.hours if a.hours is not None else 8760 * world
    lat, lon = synthetic.grid_coords(a.nlat, a.nlon)
    det = pipeline.Detector(lat, lon, levels=[2.0], passes=a.passes, graphs=False, want_pieces=True)
    t0, t1 = sharding.shard_range(hours, rank, world)
    T = a.batch

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for r in det.stream((spatial.synth_pv(T, a.nlat, a.nlon, hour0=float(t0)) for _ in range(2)), depth=2):
        pass
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    sampler.mark()
    # The shard's field is generated in HBM chunk by chunk (up to 40 GB resident, untimed: a production run streams it
    # from storage; `value` of the main workload has the same "input resident in HBM" definition) and every chunk is
    # detected inside the timed region.
    chunk_batches = max(1, int(40e9 // (T * a.nlat * a.nlon * 4)))
    soups, dates, t_det = [], [], 0.0
    step0 = t0
    starts = list(range(t0, t1, T))
    for c0 in range(0, len(starts), chunk_batches):
        resident = [spatial.synth_pv(min(T, t1 - b0), a.nlat, a.nlon, hour0=float(b0), hour_step=1.0)
                    for b0 in starts[c0:c0 + chunk_batches]]
        torch.cuda.synchronize()
        tc = time.perf_counter()
        for res in det.stream(resident, depth=min(a.depth, 3)):
            soup, _ = pipeline.events_soup(res, "streamers", det)
            soups.append(soup)
            dates.append(step0 + res.tables["streamers"].job.astype(np.int64))
            step0 += res.ntime
        torch.cuda.synchronize()
        t_det += time.perf_counter() - tc
        del resident
    soup = tracking.PolygonSoup.concat(soups)
    hrs = np.concatenate(dates) if dates else np.zeros(0, dtype=np.int64)
    date = np.datetime64("2000-01-01T00", "ns") + hrs * np.timedelta64(3600 * 10**9, "ns")
    stats = {}
    barrier()
    t_tr0 = time.perf_counter()
    labels = sharding.track_sharded(date, "by_overlap", soup=soup, time_range=1, stats=stats)
    torch.cuda.synchronize()
    t_tr = time.perf_counter() - t_tr0
    barrier()
    t_tot = t_det + t_tr
    clocks = sampler.stop()
    tm = torch.tensor([t_tot, t_det, t_tr], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([len(labels), stats.get("pairs_in_range", 0), stats.get("candidates", 0), stats.get("links", 0),
                        int(labels.max()) + 1 if len(labels) else 0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        mx = cnt[4:].clone()
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        cnt[4] = mx[0]
    if rank == 0:
        t_tot, t_det, t_tr = (float(v) for v in tm)
        ev, inr, cand, links, ntracks = (int(v) for v in cnt)
        print(json.dumps({
            "metric": "time steps/sec, 0.25deg hourly detection + to_xarray + track_events(by_overlap) across shard boundaries",
            "value": hours / t_tot, "unit": UNIT, "n_gpus": world, "hours": hours, "higher_is_better": True, "scaling": "strong",
            "data": "synthetic", "dtype": "f64", "clocks": clocks,
            "seconds": {"total": t_tot, "detection": t_det, "tracking": t_tr},
            "tracking": {"events": ev, "pairs_in_range": inr, "candidate_pairs": cand, "links": links, "tracks": ntracks,
                         "events_per_s": ev / t_tr, "pairs_in_range_per_s": inr / t_tr,
                         "rank0_seconds": {k[2:]: round(v, 4) for k, v in stats.items() if k.startswith("t_")},
                         "exchange": "halo of the event table (first time_range hours of the next shard), union-find "
                                     "over the boundary components; no gather of the tables"},
            "config": {"workload": "synthetic ERA5-shaped 0.25deg ({}x{}) hourly PV, {} consecutive hours, full detection + "
                                   "to_xarray + track_events(streamers, by_overlap, time_range 1 h)".format(a.nlat, a.nlon, hours),
                       "parallelism": "time steps sharded over ranks; event-table halo for the tracking",
                       "timed": "detection of HBM-resident chunks (field generation excluded) + tracking; max over ranks"}}))
    if world > 1:
        dist.destroy_process_group()


def main():
    # stdout carries exactly ONE line (the JSON): everything libraries print there (the NCCL version banner ...) is
    # sent to stderr by pointing fd 1 at fd 2 for the run; the JSON line goes to the saved real stdout
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "decade-track":
        run_decade_track(a)
    else:
        run_b200(a)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
