"""camlasercalibratool_b200 -- B200-native (sm_100a) camera<-laser extrinsic solve.

The product is libclc_b200.so (C ABI in include/clc_b200.h, CUDA in csrc/).  This package holds the build recipe,
the ctypes binding and a Python mirror of the reference's solver interface (api.py).  Nothing here falls back to
the CPU: importing is cheap, but every numeric call needs the CUDA library and a B200.
"""
from . import _build  # noqa: F401
from .api import (  # noqa: F401
    CamLaserCalClosedSolution,
    CamLaserCalibration,
    LineFittingCeres,
    ClcError,
    Comm,
    Group,
    Oberserve,
    Problem,
    T_to_pose7,
    comm_unique_id,
    debug_pack,
    default_options,
    launch_count,
    marshal,
    pose7_to_T,
    problems_from_scans,
    shard_range,
    upload_stats,
)

__all__ = [
    "CamLaserCalClosedSolution", "CamLaserCalibration", "LineFittingCeres", "ClcError", "Comm", "Group", "Oberserve", "Problem", "T_to_pose7",
    "comm_unique_id", "default_options", "launch_count", "marshal", "pose7_to_T", "shard_range", "debug_pack", "upload_stats",
    "problems_from_scans",
]
