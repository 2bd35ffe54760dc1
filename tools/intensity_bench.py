"""Cost of the event intensity (momentum flux from u and v) in Detector.stream, float32 and CF-packed int16: C25-L.

    python tools/intensity_bench.py [--batch 296] [--batches 2] [--host-batches 2] [--passes 3] [--depth 4] [--out DIR]

C25-L workload (BASELINE.md, SURVEY.md 8(d)): 721 x 1440, hourly synthetic PV generated in device memory, levels
1.5 / 2 / 3 PVU, five smoothing passes, streamers + overturnings + cutoffs + the three flag grids kept on the device.
u and v are ``synth_pv`` fields of the seeds SEED + 1 and SEED + 2.  Arms on the headline configuration (`depth` slots
on their own streams, one CUDA graph per batch): float32 PV without intensity ("plain"), float32 PV with float32
(u, v) items whose momentum flux is computed on the device ("uv"), and PV, u and v packed on the host side as int16
with a fixed scale / offset each (ERA5's storage type, decoded in the smoothing loads and in wbk_mflux: "packed").
Every arm runs on device-resident input (`batches` distinct slabs, several GB together, far larger than the 126 MB
L2) and on pinned-host input (`host-batches` slabs, uploaded by the stream).  Four slots, not the six of bench.py:
with three levels the arenas of a 296-step slot take about 26 GB, so six slots plus the inputs and the host arm's
upload buffers would not fit in the 180 GB of a B200 -- nor do two Detectors of four slots, and the packed arms need
a Detector with the packings.  So the arms run in two groups, each with one Detector whose slots keep one captured
graph per arm: group "float" alternates plain and uv, group "packed" alternates plain and packed, `passes` times
each; plain, in both groups, ties them together.  Then one eager run per arm on one stream with CUDA events around
every kernel (wbk_prof_*) gives the time per step of wbk_mflux (float32 and int16 u, v) and of the event rasteriser,
also with a single float32 and a single packed int16 intensity field.  The GPU name, power limit and max SM clock
are read in the same run.  Prints one JSON line; needs a CUDA device.
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
# CF packings (scale_factor, add_offset, _FillValue) of the packed arms: int16 covers the synthetic fields' range.  No
# contour level is a decoded value (level - offset is no multiple of scale): the flat plateaus of a quantised field
# would otherwise lie exactly on a level and send whole steps to the sequential contour linker
PK_PV = (3.7e-4, 0.0123, None)
PK_U = (4.5e-4, 0.25, None)
PK_V = (5.0e-4, -0.5, None)
PK_F = (4.5e-4, 0.0, None)


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
    ncell = nlat * nlon

    def slab(s, seed=None):
        return spatial.synth_pv(T, nlat, nlon, hour0=float(s * T), hour_step=1.0, seed=seed)

    def pack(x, pk):
        return torch.round((x.double() - pk[1]) / pk[0]).clamp(-32766, 32766).to(torch.int16)

    def inputs(n):
        pv = [slab(s) for s in range(n)]
        uv = [(slab(s, synthetic.SEED + 1), slab(s, synthetic.SEED + 2)) for s in range(n)]
        ppv = [pack(x, PK_PV) for x in pv]
        puv = [(pack(u, PK_U), pack(v, PK_V)) for u, v in uv]
        return dict(plain=(pv, None), uv=(pv, uv), packed=(ppv, puv))

    def pinned(arms):
        def pin(x):
            return tuple(pin(y) for y in x) if isinstance(x, tuple) else x.cpu().pin_memory()

        return {k: (pin(tuple(pv)), None if it is None else pin(tuple(it))) for k, (pv, it) in arms.items()}

    sets = {"device": inputs(a.batches), "host": pinned(inputs(a.host_batches))}
    torch.cuda.synchronize()

    def region(det, where, arm, k, d=depth, shared_stream=False):
        pv, it = sets[where][arm]
        nb = len(pv)
        items = (it[s % nb] for s in range(k)) if it is not None else None
        t0 = time.perf_counter()
        for _ in det.stream((pv[s % nb] for s in range(k)), depth=d, shared_stream=shared_stream, intensity=items):
            pass
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1000.0

    def detector(group, **kw):
        pk = dict(packing=PK_PV, intensity_packing=(PK_U, PK_V)) if group == "packed" else {}
        return pipeline.Detector(lat, lon, levels=LEVELS, **pk, **kw)

    groups = {"float": ("plain", "uv"), "packed": ("plain", "packed")}
    rate, steps, replays = {}, {}, {}
    for group, names in groups.items():
        det = detector(group, graphs=True)
        arms = [(where, arm) for where in sets for arm in names]
        # warm-up: every (slot, slab, arm) combination is captured into its CUDA graph on its second submission
        for where, arm in arms:
            nb = len(sets[where][arm][0])
            region(det, where, arm, 3 * depth * (nb // math.gcd(nb, depth)))
        ms = {key: [] for key in arms}
        for _ in range(a.passes):
            for where, arm in arms:
                nb = len(sets[where][arm][0])
                k = 6 * depth * nb // math.gcd(nb, depth)
                steps["{}_{}_{}".format(group, where, arm)] = k * T
                ms[(where, arm)].append(region(det, where, arm, k))
        replays[group] = det.graph_replays
        det.close()
        del det
        torch.cuda.empty_cache()
        for (where, arm), v in ms.items():
            key = "{}_{}_{}".format(group, where, arm)
            rate[key] = [round(steps[key] / (t / 1000.0), 1) for t in v]
    best = {key: max(v) for key, v in rate.items()}
    vs_plain = {"{}_{}_{}".format(g, where, arm): round(best["{}_{}_{}".format(g, where, arm)] /
                                                        best["{}_{}_plain".format(g, where)], 4)
                for g, names in groups.items() for where in sets for arm in names if arm != "plain"}

    # ---- eager, one stream, CUDA events around every kernel: device time per step of the kernels of each arm; the
    # single-field arms compare the rasteriser's float32 and packed int16 intensity reads
    dev = sets["device"]
    fields = [slab(s, synthetic.SEED + 3) for s in range(a.batches)]
    dev["field_f32"] = (dev["plain"][0], fields)
    dev["field_i16"] = (dev["plain"][0], [pack(x, PK_F) for x in fields])
    per_step = {}
    for arm, kw in (("plain", {}), ("uv", {}), ("packed", dict(packing=PK_PV, intensity_packing=(PK_U, PK_V))),
                    ("field_f32", {}), ("field_i16", dict(intensity_packing=PK_F))):
        det = pipeline.Detector(lat, lon, levels=LEVELS, graphs=False, **kw)
        k = 2 * a.batches
        region(det, "device", arm, k, d=3, shared_stream=True)
        lib.cdll.wbk_prof_reset()
        lib.cdll.wbk_prof_enable(1)
        region(det, "device", arm, k, d=3, shared_stream=True)
        lib.cdll.wbk_prof_enable(0)
        prof = _lib.prof_read(lib)
        det.close()
        per_step[arm] = {key: round(v[1] * 1000.0 / (k * T), 3) for key, v in sorted(prof.items())}

    def gbs(arm, nbytes):
        us = per_step[arm].get("mflux")
        return round(nbytes * ncell / (us * 1e-6) / 1e9, 1) if us else None

    res = dict(
        workload="C25-L 721x1440, levels {}, batch {}, {} device slabs ({:.1f} GB of float32 PV + u + v, {:.1f} GB "
                 "packed), {} pinned-host slabs, depth {}, graphs".format(
                     LEVELS, T, a.batches, 12 * a.batches * T * ncell / 1e9, 6 * a.batches * T * ncell / 1e9,
                     a.host_batches, depth),
        packings=dict(pv=PK_PV, u=PK_U, v=PK_V, field=PK_F),
        passes=a.passes, steps_per_region=steps, steps_per_s=rate, best_over_plain_same_group=vs_plain,
        graph_replays=replays,
        # float32 u, v: 4 + 4 B read and 4 B written per cell; int16: 2 + 2 B read and 8 B (float64 flux) written
        mflux_us_per_step={"f32": per_step["uv"].get("mflux"), "i16": per_step["packed"].get("mflux")},
        mflux_gbs_at_12_bytes_per_cell={"f32": gbs("uv", 12), "i16": gbs("packed", 12)},
        events_raster_us_per_step={arm: per_step[arm].get("events_raster") for arm in per_step},
        kernel_us_per_step=per_step, **info)
    print(json.dumps(res), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "intensity_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
