"""Cost of tracking streamers while Detector.stream runs, against tracking after detection on the host.

    python tools/track_stream_bench.py [--batch 296] [--batches 8] [--steps 17760] [--passes 2] [--depth 6] [--out DIR]

C25 workload: 721 x 1440, hourly synthetic PV generated in device memory (`batches` distinct slabs of `batch` steps,
cycled over a record of `steps` hourly dates, at least two years), levels [2.0], five smoothing passes, CUDA graphs,
`depth` slots on their own streams, want_pieces=True in every arm.  Three arms alternate `passes` times in one process:

  (a) Detector.stream alone;
  (b) pipeline.events_soup after every batch, all polygons kept on the host, tracking.track_columnar at the end;
  (c) Detector.stream(trackers=[EventTracker(streamers, by_overlap, time_range=1)]): polygons of the last hour on the
      device, linked batch by batch, labels at the end.

The labels of (b) and (c) must be equal.  (a) and (c) also run once with all slots on one shared stream.  Then one
eager run of (c) on one stream with CUDA events around every kernel (wbk_prof_*) gives wbk_track_append's device time.
The GPU name and power limit are read in the same run.  Prints one JSON line; needs a CUDA device.
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

from climatology_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=296, help="hourly time steps per batch")
    ap.add_argument("--batches", type=int, default=8, help="distinct input slabs, cycled over the record")
    ap.add_argument("--steps", type=int, default=60 * 296, help="hourly steps of the record (>= 2 x 8760)")
    ap.add_argument("--passes", type=int, default=2, help="alternations of the three arms")
    ap.add_argument("--depth", type=int, default=6, help="slots (batches in flight, one stream each)")
    ap.add_argument("--out", default=None, help="directory for r3_track_stream_bench.json")
    a = ap.parse_args()

    import numpy as np
    import torch

    from wavebreaking_b200 import _lib, pipeline, spatial, synthetic, tracking

    lib = _lib.get()
    nlat, nlon = 721, 1440
    T, nb, depth = a.batch, a.batches, a.depth
    k = -(-a.steps // T)
    lat, lon = synthetic.grid_coords(nlat, nlon)
    slabs = [spatial.synth_pv(T, nlat, nlon, hour0=float(s * T), hour_step=1.0) for s in range(nb)]
    torch.cuda.synchronize()
    ntime = k * T
    dates = synthetic.time_axis(ntime, 1)

    def batches():
        return (slabs[s % nb] for s in range(k))

    def arm_plain(det, **kw):
        for _ in det.stream(batches(), depth=depth, **kw):
            pass
        return None

    def arm_host(det, **kw):
        soups, steps, t = [], [], 0
        for res in det.stream(batches(), depth=depth, **kw):
            soup, _ = pipeline.events_soup(res, "streamers", det)
            soups.append(soup)
            steps.append(t + res.tables["streamers"].job.astype(np.int64))
            t += res.ntime
        labels, _ = tracking.track_columnar(dates[np.concatenate(steps)], "by_overlap",
                                            soup=tracking.PolygonSoup.concat(soups), time_range=1)
        return labels

    trackers = []

    def arm_device(det, **kw):
        tr = pipeline.EventTracker(det, dates, "streamers", time_range=1)
        for _ in det.stream(batches(), depth=depth, trackers=[tr], **kw):
            pass
        trackers.append(tr)
        return tr.labels()

    arms = {"stream": arm_plain, "host_tracking": arm_host, "stream_tracker": arm_device}
    # one Detector for the three arms: they differ only in what happens after every batch is collected
    det = pipeline.Detector(lat, lon, levels=[2.0], graphs=True, want_pieces=True)
    # warm-up: every (slot, slab) combination is captured into its CUDA graph on its second submission
    warm = 3 * depth * (nb // math.gcd(nb, depth))
    for _ in det.stream((slabs[s % nb] for s in range(warm)), depth=depth):
        pass
    torch.cuda.synchronize()
    ms = {name: [] for name in arms}
    labels = {}
    for _ in range(a.passes):
        for name, fn in arms.items():
            t0 = time.perf_counter()
            labels[name] = fn(det)
            torch.cuda.synchronize()
            ms[name].append((time.perf_counter() - t0) * 1000.0)
    assert np.array_equal(labels["host_tracking"], labels["stream_tracker"])
    tr = trackers[-1]
    # all slots on one shared stream: the tracker's read-backs run on its own stream, not behind the queued batches
    shared = {}
    for name in ("stream", "stream_tracker"):
        t0 = time.perf_counter()
        arms[name](det, shared_stream=True)
        torch.cuda.synchronize()
        shared[name] = round(ntime / (time.perf_counter() - t0), 1)
    det.close()
    rate = {name: [round(ntime / (v / 1000.0), 1) for v in ms[name]] for name in arms}
    best = {name: max(r) for name, r in rate.items()}

    # ---- eager, one stream, CUDA events around every kernel: wbk_track_append's device time
    det = pipeline.Detector(lat, lon, levels=[2.0], graphs=False, want_pieces=True)
    lib.cdll.wbk_prof_reset()
    lib.cdll.wbk_prof_enable(1)
    arm_device(det, shared_stream=True)
    lib.cdll.wbk_prof_enable(0)
    prof = _lib.prof_read(lib)
    det.close()
    n_ap, ms_ap = prof["track_append"]
    host_ms = np.asarray(tr.host_ms)
    res = dict(
        workload="C25 721x1440, batch {}, {} distinct slabs cycled over {} hourly steps ({} batches), depth {}, graphs, "
                 "want_pieces; streamers tracked by_overlap, time_range 1 h".format(T, nb, ntime, k, depth),
        passes=a.passes, events=int(tr.n_events), tracks=int(labels["stream_tracker"].max() + 1),
        stats=tr.stats,
        steps_per_s_stream=rate["stream"], steps_per_s_host_tracking=rate["host_tracking"],
        steps_per_s_stream_tracker=rate["stream_tracker"],
        tracker_vs_stream_best_pct=round(100.0 * (1.0 - best["stream_tracker"] / best["stream"]), 2),
        steps_per_s_shared_stream=shared["stream"], steps_per_s_shared_stream_tracker=shared["stream_tracker"],
        tracker_vs_host_tracking_speedup=round(best["stream_tracker"] / best["host_tracking"], 2),
        track_append_launches=n_ap, track_append_ms_total=round(ms_ap, 3),
        track_append_us_per_batch=round(ms_ap * 1000.0 / k, 2),
        tracker_host_ms_per_batch=dict(mean=round(float(host_ms.mean()), 3), median=round(float(np.median(host_ms)), 3),
                                       max=round(float(host_ms.max()), 3)),
        kernel_ms_total={key: round(v[1], 3) for key, v in sorted(prof.items())},
        labels_equal=True, **gpu_info())
    print(json.dumps(res), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "r3_track_stream_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
