"""Input streaming for the detection path: field files -> pinned host batches -> ``Detector.stream``.

SURVEY.md 8(f).4: the reference loads a whole NetCDF file through xarray and re-sorts descending latitudes with
``sortby`` on every call (utils/data_utils.py:196-213).  Here a (time, lat, lon) array on disk -- a ``.npy`` file or a
raw little-endian binary, both memory-mapped; NetCDF readers are not part of this image -- is read in batches of
time steps by a background thread into a ring of pinned host buffers, so the file read of batch k+1 overlaps the
upload and the kernels of batch k.  Descending coordinates are handled on the device by ``Detector`` (``wbk_flip``),
never by re-sorting the file.
"""

import threading
import queue

import numpy as np
import torch

from . import _lib


def open_field(path, shape=None, dtype=np.float32):
    """Memory-map a (time, lat, lon) field: ``.npy`` (shape / dtype from the header) or raw binary (given)."""
    if str(path).endswith(".npy"):
        arr = np.load(path, mmap_mode="r")
    else:
        if shape is None:
            raise ValueError("shape is required for raw binary fields")
        arr = np.memmap(path, dtype=dtype, mode="r", shape=tuple(shape))
    if arr.ndim != 3:
        raise ValueError("expected a (time, lat, lon) array, got shape {}".format(arr.shape))
    if arr.dtype not in (np.float32, np.float64):
        raise TypeError("field dtype has to be float32 or float64, got {}".format(arr.dtype))
    return arr


def iter_batches(field, batch, depth=3, start=0, stop=None, intensity=None):
    """Yield pinned host tensors ``field[t : t + batch]`` in time order, read ahead by a background thread.

    ``depth + 1`` pinned buffers rotate, so a yielded tensor stays valid while the next ``depth`` batches are
    produced -- exactly the lifetime ``Detector.stream(depth=depth)`` needs for its asynchronous uploads.
    ``intensity``: an array shaped like ``field``, or a pair ``(u, v)`` of them; then every item is the pair
    ``(batch, item)`` with ``item`` the same steps of the intensity (a tensor, or a pair of tensors), read by the same
    thread into the same ring slot as the batch, so it stays valid exactly as long.
    """
    stop = field.shape[0] if stop is None else min(stop, field.shape[0])
    if batch < 1:
        raise ValueError("batch has to be positive")
    pin = _lib.get().is_cuda
    arrays = [field]
    if intensity is not None:
        arrays += list(intensity) if isinstance(intensity, (tuple, list)) else [intensity]
    nbuf = depth + 2
    bufs = [[torch.empty((batch,) + tuple(a.shape[1:]), dtype=torch.float32 if a.dtype == np.float32 else torch.float64,
                         pin_memory=pin) for a in arrays] for _ in range(nbuf)]
    free = queue.Queue()
    for b in range(nbuf):
        free.put(b)
    ready = queue.Queue(maxsize=nbuf)

    def reader():
        try:
            for t0 in range(start, stop, batch):
                b = free.get()
                n = min(batch, stop - t0)
                for buf, a in zip(bufs[b], arrays):
                    np.copyto(buf.numpy()[:n], a[t0:t0 + n])
                ready.put((b, n))
            ready.put(None)
        except BaseException as exc:  # surfaced in the consumer
            ready.put(exc)

    th = threading.Thread(target=reader, daemon=True)
    th.start()
    held = []
    while True:
        item = ready.get()
        if item is None:
            break
        if isinstance(item, BaseException):
            raise item
        b, n = item
        held.append(b)
        if len(held) > depth + 1:  # the oldest buffer is no longer referenced by an in-flight batch
            free.put(held.pop(0))
        views = [buf[:n] for buf in bufs[b]]
        if intensity is None:
            yield views[0]
        else:
            yield views[0], (views[1] if len(views) == 2 else tuple(views[1:]))
    th.join()


def detect_file(path, lat, lon, batch=296, depth=3, shape=None, dtype=np.float32, gmax_nx="full", climatology=None,
                trackers=None, intensity=None, **detector_kwargs):
    """Run the whole detection path over a field file; yields ``(t0, BatchResult)`` per batch in time order.

    ``gmax_nx``: see ``Detector.stream`` (the reference's global ``exp_lon.max()``).  ``climatology``: a
    ``pipeline.FlagClimatology`` for the same grid; the flag grids of every batch are added to it on the device.
    ``trackers``: a list of ``pipeline.EventTracker`` for the same grid, which track the events of every batch.
    ``intensity``: the path of an intensity field, or a pair of paths ``(u_path, v_path)`` whose momentum flux is the
    intensity (see ``Detector.stream``); opened like ``path`` (same ``shape`` / ``dtype`` for raw binary files) and
    stored like the field."""
    from . import pipeline

    field = open_field(path, shape=shape, dtype=dtype)
    inten = None
    if intensity is not None:
        paths = tuple(intensity) if isinstance(intensity, (tuple, list)) else (intensity,)
        if len(paths) not in (1, 2):
            raise ValueError("intensity is a path or a pair of paths (u_path, v_path)")
        inten = tuple(open_field(p, shape=shape, dtype=dtype) for p in paths)
        for p, a in zip(paths, inten):
            if a.shape != field.shape:
                raise ValueError("intensity file {} has shape {}, the field {}".format(p, a.shape, field.shape))
        inten = inten if len(inten) == 2 else inten[0]
    det = pipeline.Detector(lat, lon, **detector_kwargs)
    batches, items = iter_batches(field, batch, depth=depth, intensity=inten), None
    if inten is not None:
        pending = []  # the intensity item of the batch the stream took last (it asks for both in step)

        def fields(pairs):
            for b, it in pairs:
                pending.append(it)
                yield b

        batches, items = fields(batches), iter(lambda: pending.pop(0), None)
    t0 = 0
    for res in det.stream(batches, depth=depth, gmax_nx=gmax_nx, climatology=climatology, trackers=trackers,
                          intensity=items):
        yield t0, res
        t0 += res.ntime
