"""Throughput of Detector.stream on an anisotropic grid and on an isotropic grid of similar size.

    python tools/grid_shapes_bench.py [--batch 100] [--batches 8] [--depth 6] [--out DIR]

Shapes: 361 x 576 (MERRA-2, 0.625 x 0.5 degrees: flag grids with the elliptic to_xarray buffer) and 361 x 720
(0.5 degrees, isotropic).  Hourly synthetic PV generated in device memory, levels [2.0], five smoothing passes,
streamers + overturnings + cutoffs + the three flag grids.  Per shape it prints one JSON line: steps/s of the
headline configuration (`depth` slots on their own streams, one CUDA graph per batch) and the per-kernel device time
in us per time step from a second run on one stream with eager launches and CUDA events around every kernel
(wbk_prof_*).  Needs a CUDA device.
"""

import argparse
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [("merra2_0.625x0.5", 361, 576), ("iso_0.5", 361, 720)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=100, help="hourly time steps per batch")
    ap.add_argument("--batches", type=int, default=8, help="timed batches per shape")
    ap.add_argument("--depth", type=int, default=6, help="slots (batches in flight, one stream each)")
    ap.add_argument("--out", default=None, help="directory for grid_shapes_bench.json")
    a = ap.parse_args()

    import numpy as np
    import torch

    from wavebreaking_b200 import _lib, pipeline, spatial

    lib = _lib.get()
    props = torch.cuda.get_device_properties(0)
    results = []
    for name, nlat, nlon in SHAPES:
        lat = np.linspace(-90.0, 90.0, nlat)
        lon = np.arange(nlon) * (360.0 / nlon)
        T, K, depth = a.batch, a.batches, a.depth
        slabs = [spatial.synth_pv(T, nlat, nlon, hour0=float(s * T), hour_step=1.0) for s in range(4)]
        torch.cuda.synchronize()

        def region(det, k, shared_stream, profile, depth):
            n_in = len(slabs)
            warm = 3 * depth * (n_in // math.gcd(n_in, depth)) if det.graphs else 2 * depth
            for _ in det.stream((slabs[s % n_in] for s in range(warm)), depth=depth, shared_stream=shared_stream):
                pass
            torch.cuda.synchronize()
            lib.cdll.wbk_prof_reset()
            lib.cdll.wbk_prof_enable(1 if profile else 0)
            t0 = time.perf_counter()
            events = 0
            for res in det.stream((slabs[(warm + s) % n_in] for s in range(k)), depth=depth,
                                  shared_stream=shared_stream):
                events += sum(v for key, v in pipeline.summarize(res).items()
                              if key in ("streamers", "overturnings", "cutoffs"))
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1000.0
            lib.cdll.wbk_prof_enable(0)
            return ms, (_lib.prof_read(lib) if profile else {}), events

        det = pipeline.Detector(lat, lon, levels=[2.0], graphs=True)
        ms, _, events = region(det, K, False, False, depth)
        det.close()
        det = pipeline.Detector(lat, lon, levels=[2.0], graphs=False)
        _, prof, _ = region(det, K, True, True, min(depth, 3))
        det.close()
        steps = K * T
        results.append(dict(
            shape=name, nlat=nlat, nlon=nlon, dlon=float(lon[1] - lon[0]), dlat=float(lat[1] - lat[0]),
            batch=T, batches=K, depth=depth, steps_per_s=round(steps / (ms / 1000.0), 1),
            events_per_step=round(events / steps, 2),
            kernel_us_per_step={k: round(v[1] * 1000.0 / steps, 2) for k, v in sorted(prof.items())},
            gpu=props.name))
        print(json.dumps(results[-1]), flush=True)
        del slabs
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "grid_shapes_bench.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
