"""b200-robot-tick: B200-native batched control tick (vehicle / IMU update / arm
interpolation) of the Roboken-FMSKF robot-controller firmware.

The arithmetic lives in hand-written CUDA for sm_100a behind the C-ABI of
include/robotick.h (librobotick_b200.so).  This package is the thin host side: ctypes
binding, state layout helpers, synthetic streams and torch-owned device buffers.
"""
from . import _cabi, layout, streams  # noqa: F401
from ._cabi import RobotickError, default_params, load  # noqa: F401

__all__ = ["_cabi", "layout", "streams", "RobotickError", "default_params", "load"]


def __getattr__(name):
    # torch-dependent modules are imported lazily so that layout/streams stay light.  import_module, not `from . import`:
    # the latter first probes this module for the attribute, which would call __getattr__ again.
    import importlib

    if name in ("vehicle", "VehicleBatch"):
        _v = importlib.import_module(".vehicle", __name__)
        return _v if name == "vehicle" else _v.VehicleBatch
    if name in ("planner", "VehiclePlanner", "CostMap", "CostToGo", "inflation_table"):
        _p = importlib.import_module(".planner", __name__)
        return _p if name == "planner" else getattr(_p, name)
    raise AttributeError(name)
