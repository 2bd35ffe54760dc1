"""The reference arm of bench.py (the oracle port on the host cores) prints the JSON line of the bench contract;
checked on a coarse grid so that it runs in seconds.  The output dump of the CUDA arm (--dump-outputs) is checked on
the emulator build and, on a GPU, by two runs of the benchmark that must write identical arrays."""

import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=600, cwd=ROOT, env=env)
    assert res.returncode == 0, res.stderr[-2000:]
    return res.stdout.strip().splitlines()


def test_reference_arm_json_line():
    lines = _run("--impl", "reference", "--nlat", "46", "--nlon", "90", "--steps", "1", "--warmup", "1")
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["higher_is_better"] is True and d["unit"] == "time steps/s" and d["value"] > 0
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None
    cpu = d["cpu_baseline"]
    assert cpu["kind"] == "port" and cpu["cores"] >= 1 and cpu["value"] == d["value"] and cpu["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert set(d["config"]) == {"workload", "l2", "parallelism"}  # no per-arm keys: both arms print the same config


def test_reference_arm_other_ranks_exit_quietly():
    """under torchrun only rank 0 runs the CPU arm; the other ranks exit 0 without output"""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29999")
    assert _run("--impl", "reference", "--gpus", "2", "--nlat", "46", "--nlon", "90", "--steps", "1", env=env) == []


def _load_bench():
    write_bytecode = sys.dont_write_bytecode
    spec = importlib.util.spec_from_file_location("wbk_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.dont_write_bytecode = write_bytecode  # bench.py turns bytecode caches off for its own process only
    return mod


def _small_batch():
    from wavebreaking_b200 import pipeline, spatial, synthetic

    lat, lon = synthetic.grid_coords(46, 90)
    raw = synthetic.pv_field(46, 90, np.arange(3) * 6.0)
    return pipeline.Detector(lat, lon, levels=[2.0]).run_batch(spatial.to_device(raw))


def _read_dump(path):
    return {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}


def test_dump_outputs_writes_the_batch_emu(emu, tmp_path):
    bench = _load_bench()
    from wavebreaking_b200 import detect

    res = _small_batch()
    nbytes = bench.dump_outputs(res, str(tmp_path))
    got = _read_dump(tmp_path)
    assert nbytes == sum(v.nbytes for v in got.values()) <= bench.DUMP_MAX_BYTES
    assert all(v.dtype in (np.float32, np.float64) and v.size for v in got.values())
    assert "near" not in got and res.near_total == 0  # no rows, not written: counted instead
    assert got["counts"].tolist() == [3, res.contours.ncontours, res.contours.npoints, *map(len, res.tables.values()),
                                      res.n_split, 0]
    flags = res.flags.numpy()
    assert np.array_equal(got["flags_sample"], flags.reshape(-1))  # small enough to be written whole
    h = res.contours.host()
    assert np.array_equal(got["contour_points"], np.c_[h["x"], h["y"]])
    assert np.array_equal(got["contours"][:, 4], np.diff(h["pt_off"]))
    for kind in detect.KINDS:
        t = res.tables[kind]
        if len(t) == 0:  # (no overturnings in this batch)
            assert not any(k.startswith(kind) for k in got), kind
            continue
        assert got[kind + "_events"].shape == (len(t), 17)
        assert np.array_equal(got[kind + "_events"][:, 11:], t.sums)
        if kind != "overturnings":
            assert np.array_equal(got[kind + "_ring_points"], np.concatenate(list(t.rings)))
    assert len(res.tables["streamers"]) > 0 and len(res.tables["cutoffs"]) > 0


def test_dump_outputs_samples_large_arrays_emu(emu, tmp_path, monkeypatch):
    """Arrays over their cap keep the same seeded, sorted sample of rows on every run."""
    bench = _load_bench()
    caps = dict(bench.DUMP_CAPS, flags_sample=1000, contour_points=50)
    monkeypatch.setattr(bench, "DUMP_CAPS", caps)
    res = _small_batch()
    bench.dump_outputs(res, str(tmp_path / "a"))
    bench.dump_outputs(res, str(tmp_path / "b"))
    a, b = _read_dump(tmp_path / "a"), _read_dump(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    keep = bench._sample_rows(res.flags.numel(), 1000)
    assert len(keep) == 1000 and np.all(np.diff(keep) > 0)
    assert np.array_equal(a["flags_sample"], res.flags.numpy().reshape(-1)[keep])
    assert a["contour_points"].shape == (50, 2)


def test_dump_outputs_needs_the_cuda_arm():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 2 and "--dump-outputs" in res.stderr


@pytest.mark.gpu
def test_bench_dump_is_reproducible_gpu(tmp_path):
    """Two runs with the same arguments time the given number of steps and write identical outputs."""
    args = ["--steps", "3", "--warmup", "1", "--batch", "4", "--nlat", "181", "--nlon", "360", "--no-cpu", "--no-e2e",
            "--no-extras"]
    for run in ("a", "b"):
        lines = _run(*args, "--dump-outputs", str(tmp_path / run))
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
    a, b = _read_dump(tmp_path / "a"), _read_dump(tmp_path / "b")
    assert "flags_sample" in a and a.keys() == b.keys()
    for k in a:
        assert a[k].size and np.array_equal(a[k], b[k]), k
    assert a["flags_sample"].shape == (3 * 4 * 181 * 360,) and a["flags_sample"].sum() > 0
