"""bodyslam_b200 -- B200-native (sm_100a) implementation of BodySLAM's depth->3D hot path.

Drop-in surface (same names / signatures as the reference):
  MDEM : colorize, process_image, process_images, DepthEstimator, MDEMInterface,
         compute_median_scale_factor                       (bodyslam_b200.mdem)
  3DM  : TSDF, RGBD, update_map_after_pg, get_o3d_intrinsic, pixel_to_3d,
         compute_curr_estimate_global_pose                 (bodyslam_b200.tsdf / .slam_utils)
Everything downstream of the predicted depth tensor runs in hand-written CUDA kernels reached
through the C ABI in include/bodyslam_b200.h (libbodyslam_b200.so).  There is no CPU fallback.
"""
__version__ = "0.1.0"

from . import _lib  # noqa: F401
from .geometry import PinholeCameraIntrinsic, PointCloud, RGBDImage, TriangleMesh  # noqa: F401


def __getattr__(name):  # lazy: keep `import bodyslam_b200` light and torch-free until used
    import importlib

    table = {
        "TSDF": "tsdf", "MAP": "tsdf", "DenseTSDFVolume": "tsdf",
        "RGBD": "slam_utils", "update_map_after_pg": "slam_utils", "get_o3d_intrinsic": "slam_utils",
        "compute_curr_estimate_global_pose": "slam_utils", "pixel_to_3d": "slam_utils",
        "colorize": "mdem", "process_image": "mdem", "process_images": "mdem", "DepthEstimator": "mdem",
        "MDEMInterface": "mdem", "compute_median_scale_factor": "mdem",
        "ShardedTSDF": "sharding",
        "RaycastingScene": "raycasting",
    }
    if name in table:
        return getattr(importlib.import_module(f"{__name__}.{table[name]}"), name)
    raise AttributeError(name)
