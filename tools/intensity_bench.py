"""Cost of the event intensity (momentum flux from u and v) in Detector.stream: C25-L.

    python tools/intensity_bench.py [--batch 296] [--batches 2] [--host-batches 2] [--passes 3] [--depth 4] [--out DIR]

C25-L workload (BASELINE.md, SURVEY.md 8(d)): 721 x 1440, hourly synthetic PV generated in device memory, levels
1.5 / 2 / 3 PVU, five smoothing passes, streamers + overturnings + cutoffs + the three flag grids kept on the device.
u and v are ``synth_pv`` fields of the seeds SEED + 1 and SEED + 2.  Two arms on the headline configuration (`depth`
slots on their own streams, one CUDA graph per batch): without intensity and with (u, v) items whose momentum flux is
computed on the device.  Both arms run on device-resident input (`batches` distinct slabs, several GB together, far
larger than the 126 MB L2) and on pinned-host input (`host-batches` slabs, uploaded by the stream); the arms alternate
`passes` times in the same process and share one Detector (its slots keep one captured graph per arm).  Four slots,
not the six of bench.py: with three levels the arenas of a 296-step slot take about 26 GB, so six slots plus the
inputs and the host arm's upload buffers would not fit in the 180 GB of a B200.  Then one eager run per arm on one
stream with CUDA events around every kernel (wbk_prof_*) gives the time per step of wbk_mflux and the event
rasteriser.  The GPU name, power limit and max SM clock are read in the same run.  Prints one JSON line; needs a CUDA
device.
"""

import argparse
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

LEVELS = [1.5, 2.0, 3.0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=296, help="hourly time steps per batch")
    ap.add_argument("--batches", type=int, default=2, help="distinct device-resident slabs")
    ap.add_argument("--host-batches", type=int, default=2, help="distinct pinned-host slabs")
    ap.add_argument("--passes", type=int, default=3, help="alternations of the arms")
    ap.add_argument("--depth", type=int, default=4, help="slots (batches in flight, one stream each)")
    ap.add_argument("--out", default=None, help="directory for intensity_bench.json")
    a = ap.parse_args()

    import torch

    from climatology_bench import gpu_info
    from wavebreaking_b200 import _lib, pipeline, spatial, synthetic

    info = gpu_info()
    lib = _lib.get()
    nlat, nlon = 721, 1440
    T, depth = a.batch, a.depth
    lat, lon = synthetic.grid_coords(nlat, nlon)

    def slab(s, seed=None):
        return spatial.synth_pv(T, nlat, nlon, hour0=float(s * T), hour_step=1.0, seed=seed)

    def inputs(n):
        pv = [slab(s) for s in range(n)]
        uv = [(slab(s, synthetic.SEED + 1), slab(s, synthetic.SEED + 2)) for s in range(n)]
        return pv, uv

    dev_pv, dev_uv = inputs(a.batches)
    host_pv, host_uv = inputs(a.host_batches)
    host_pv = [x.cpu().pin_memory() for x in host_pv]
    host_uv = [tuple(x.cpu().pin_memory() for x in p) for p in host_uv]
    torch.cuda.synchronize()
    sets = {"device": (dev_pv, dev_uv), "host": (host_pv, host_uv)}

    def region(det, where, inten, k, d=depth, shared_stream=False):
        pv, uv = sets[where]
        nb = len(pv)
        items = (uv[s % nb] for s in range(k)) if inten else None
        t0 = time.perf_counter()
        for _ in det.stream((pv[s % nb] for s in range(k)), depth=d, shared_stream=shared_stream, intensity=items):
            pass
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1000.0

    det = pipeline.Detector(lat, lon, levels=LEVELS, graphs=True)
    arms = [(where, inten) for where in sets for inten in (False, True)]
    # warm-up: every (slot, slab, arm) combination is captured into its CUDA graph on its second submission
    for where, inten in arms:
        nb = len(sets[where][0])
        region(det, where, inten, 3 * depth * (nb // math.gcd(nb, depth)))
    ms = {key: [] for key in arms}
    steps = {}
    for _ in range(a.passes):
        for where, inten in arms:
            nb = len(sets[where][0])
            k = 6 * depth * nb // math.gcd(nb, depth)
            steps[(where, inten)] = k * T
            ms[(where, inten)].append(region(det, where, inten, k))
    replays = det.graph_replays
    det.close()
    torch.cuda.empty_cache()

    def name(key):
        return "{}_{}".format(key[0], "uv" if key[1] else "plain")

    rate = {name(key): [round(steps[key] / (v / 1000.0), 1) for v in ms[key]] for key in arms}
    slowdown = {where: round(100.0 * (1.0 - max(rate[where + "_uv"]) / max(rate[where + "_plain"])), 2)
                for where in sets}

    # ---- eager, one stream, CUDA events around every kernel: device time per step of the kernels of each arm
    per_step = {}
    for inten in (False, True):
        det = pipeline.Detector(lat, lon, levels=LEVELS, graphs=False)
        k = 2 * len(dev_pv)
        region(det, "device", inten, k, d=3, shared_stream=True)
        lib.cdll.wbk_prof_reset()
        lib.cdll.wbk_prof_enable(1)
        region(det, "device", inten, k, d=3, shared_stream=True)
        lib.cdll.wbk_prof_enable(0)
        prof = _lib.prof_read(lib)
        det.close()
        per_step["uv" if inten else "plain"] = {key: round(v[1] * 1000.0 / (k * T), 3) for key, v in sorted(prof.items())}
    res = dict(
        workload="C25-L 721x1440, levels {}, batch {}, {} device slabs ({:.1f} GB of float32 PV + u + v), {} pinned-host "
                 "slabs, depth {}, graphs".format(LEVELS, T, len(dev_pv), 3 * len(dev_pv) * T * nlat * nlon * 4 / 1e9,
                                                  len(host_pv), depth),
        passes=a.passes, steps_per_region={name(key): v for key, v in steps.items()},
        steps_per_s=rate, slowdown_best_pct=slowdown, graph_replays=replays,
        mflux_us_per_step=per_step["uv"].get("mflux"),
        mflux_gbs=round(3 * nlat * nlon * 4 / (per_step["uv"]["mflux"] * 1e-6) / 1e9, 1) if "mflux" in per_step["uv"]
        else None,
        events_raster_us_per_step={arm: per_step[arm].get("events_raster") for arm in per_step},
        kernel_us_per_step=per_step, **info)
    print(json.dumps(res), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "intensity_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
