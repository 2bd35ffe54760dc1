"""Cost of accumulating a monthly flag-frequency climatology on the device during Detector.stream.

    python tools/climatology_bench.py [--batch 296] [--batches 8] [--passes 3] [--depth 6] [--out DIR]

C25 workload: 721 x 1440, hourly synthetic PV generated in device memory (`batches` distinct slabs of `batch` steps,
together far larger than the 126 MB L2), levels [2.0], five smoothing passes, streamers + overturnings + cutoffs + the
three flag grids kept on the device.  Two arms on the headline configuration (`depth` slots on their own streams, one
CUDA graph per batch): without a climatology and with a 12-month FlagClimatology over a record that crosses month
boundaries.  The arms alternate `passes` times in the same process.  Then one eager run on one stream with CUDA events
around every kernel (wbk_prof_*) gives wbk_flag_counts' time per step and its achieved bandwidth (3 bytes read per cell
and step), set against a device-to-device copy measured in the same run and the 7.7 TB/s data-sheet figure.  The GPU
name and power limit are read in the same run.  Prints one JSON line; needs a CUDA device.
"""

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DATASHEET_GBS = 7700.0


def gpu_info():
    """name, power limit (W) and max SM clock of GPU 0 (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [p.strip() for p in out.split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as exc:  # noqa: BLE001
        import torch

        return dict(gpu=torch.cuda.get_device_name(0), power_limit="unknown ({})".format(exc))


def copy_peak_gbs(torch, nbytes=4 << 30, reps=10):
    """device-to-device copy: (read + written bytes) / time, best of `reps`."""
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2 * nbytes / (best / 1000.0) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=296, help="hourly time steps per batch")
    ap.add_argument("--batches", type=int, default=8, help="distinct input slabs; each timed region streams 3x this")
    ap.add_argument("--passes", type=int, default=3, help="alternations of the two arms")
    ap.add_argument("--depth", type=int, default=6, help="slots (batches in flight, one stream each)")
    ap.add_argument("--out", default=None, help="directory for climatology_bench.json")
    a = ap.parse_args()

    import numpy as np
    import torch

    from wavebreaking_b200 import _lib, pipeline, spatial, synthetic

    lib = _lib.get()
    nlat, nlon = 721, 1440
    ncells = nlat * nlon
    T, nb, depth = a.batch, a.batches, a.depth
    lat, lon = synthetic.grid_coords(nlat, nlon)
    slabs = [spatial.synth_pv(T, nlat, nlon, hour0=float(s * T), hour_step=1.0) for s in range(nb)]
    torch.cuda.synchronize()
    k = 3 * nb  # batches per timed region
    ntime = k * T
    dates = np.datetime64("2001-01-20T00", "h") + np.arange(ntime) * np.timedelta64(1, "h")
    groups = pipeline.groups_from_dates(dates, "month")
    months_crossed = int(len(np.unique(groups)))

    def region(det, clim, profile=False, shared_stream=False, d=depth):
        t0 = time.perf_counter()
        for _ in det.stream((slabs[s % nb] for s in range(k)), depth=d, shared_stream=shared_stream, climatology=clim):
            pass
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1000.0

    arms = {"plain": pipeline.Detector(lat, lon, levels=[2.0], graphs=True),
            "climatology": pipeline.Detector(lat, lon, levels=[2.0], graphs=True)}
    # warm-up: every (slot, slab) combination is captured into its CUDA graph on its second submission
    warm = 3 * depth * (nb // math.gcd(nb, depth))
    for name, det in arms.items():
        clim = pipeline.FlagClimatology(det, np.zeros(warm * T, dtype=np.int32)) if name == "climatology" else None
        for _ in det.stream((slabs[s % nb] for s in range(warm)), depth=depth, climatology=clim):
            pass
    torch.cuda.synchronize()
    ms = {name: [] for name in arms}
    for _ in range(a.passes):
        for name, det in arms.items():
            clim = pipeline.FlagClimatology(det, groups, ngroups=12) if name == "climatology" else None
            ms[name].append(region(det, clim))
            if clim is not None:
                assert int(clim.steps.sum()) == ntime
    for det in arms.values():
        det.close()
    rate = {name: [round(ntime / (v / 1000.0), 1) for v in ms[name]] for name in arms}
    best = {name: max(r) for name, r in rate.items()}

    # ---- eager, one stream, CUDA events around every kernel: wbk_flag_counts' device time
    det = pipeline.Detector(lat, lon, levels=[2.0], graphs=False)
    region(det, pipeline.FlagClimatology(det, groups, ngroups=12), shared_stream=True, d=3)
    lib.cdll.wbk_prof_reset()
    lib.cdll.wbk_prof_enable(1)
    clim = pipeline.FlagClimatology(det, groups, ngroups=12)
    region(det, clim, shared_stream=True, d=3)
    lib.cdll.wbk_prof_enable(0)
    prof = _lib.prof_read(lib)
    det.close()
    n_fc, ms_fc = prof["flag_counts"]
    us_per_step = ms_fc * 1000.0 / ntime
    bytes_per_step = 3 * ncells
    achieved = bytes_per_step / (us_per_step * 1e-6) / 1e9
    del slabs
    torch.cuda.empty_cache()
    peak = copy_peak_gbs(torch)
    res = dict(
        workload="C25 721x1440, batch {}, {} distinct slabs ({:.1f} GB of float32 input), {} batches per region, "
                 "depth {}, graphs".format(T, nb, nb * T * ncells * 4 / 1e9, k, depth),
        months_in_record=months_crossed, passes=a.passes,
        steps_per_s_plain=rate["plain"], steps_per_s_climatology=rate["climatology"],
        slowdown_best_pct=round(100.0 * (1.0 - best["climatology"] / best["plain"]), 2),
        flag_counts_launches=n_fc, flag_counts_us_per_step=round(us_per_step, 3),
        flag_counts_gbs=round(achieved, 1), copy_peak_gbs=round(peak, 1),
        frac_of_copy_peak=round(achieved / peak, 3), frac_of_datasheet=round(achieved / DATASHEET_GBS, 3),
        kernel_us_per_step={key: round(v[1] * 1000.0 / ntime, 2) for key, v in sorted(prof.items())},
        **gpu_info())
    print(json.dumps(res), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "climatology_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
