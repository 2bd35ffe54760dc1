"""B200-native drop-in for the per-time-step detection path of skaderli/WaveBreaking.

Same public names as ``wavebreaking/__init__.py:19-34`` (plotting is out of scope).  The CUDA library
``libwbk.so`` is required: there is no CPU fallback (``wavebreaking_b200._lib.get`` raises without it).
"""

__version__ = "0.1.0"

_API = ("calculate_momentum_flux", "calculate_smoothed_field", "to_xarray", "track_events", "event_tracking",
        "calculate_contours", "calculate_streamers", "calculate_overturnings", "calculate_cutoffs", "combine_shared", "flag_frequency")


def __getattr__(name):  # lazy: importing the package must not need torch / a GPU
    if name in _API:
        from . import api

        return getattr(api, name)
    raise AttributeError(name)


__all__ = list(_API)
