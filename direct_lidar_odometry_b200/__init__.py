"""direct_lidar_odometry_b200 — B200-native (sm_100a) NanoGICP registration hot path of Direct LiDAR Odometry.

    from direct_lidar_odometry_b200 import NanoGICP
    gicp = NanoGICP(device=0)            # raises if the CUDA library / a GPU is missing: no CPU fallback

The compute lives in csrc/ (hand-written CUDA behind the C ABI of include/nanogicp_c.h);
`NanoGICP` mirrors the reference class nano_gicp::NanoGICP member for member.
"""
from . import synth  # noqa: F401  (pure numpy)
from . import pointcloud2  # noqa: F401  (plain data + field mapping, no ROS)

__all__ = ["NanoGICP", "NanoGICPError", "CovarianceView", "KeyframeStore", "align_batch", "fitness_batch", "imu_prior", "synth", "pointcloud2", "lib_path"]


def __getattr__(name):
    if name in ("NanoGICP", "NanoGICPError", "CovarianceView", "KeyframeStore", "align_batch", "fitness_batch", "imu_prior"):
        from . import nanogicp
        return getattr(nanogicp, name)
    if name == "lib_path":
        from ._lib import LIB_PATH
        return LIB_PATH
    raise AttributeError(name)
