"""nvsf_b200 — B200-native (sm_100a) ray-rendering hot path of NVSF.

Importable as ``nvsf_b200`` (shim at the repository root) or via
``importlib.import_module("selfsupervised-nvsf_b200")``.

Sub-modules
    raymarching   drop-in for reference ``nvsf.nerf.raymarching.raymarching``
    field         NeRFNetwork: density / color / flow / run / render of the reference model on the GPU
                  kernels, plus the occupancy-grid update and the march_rays* render loops (run_cuda)
    rays          get_lidar_rays / get_rays (reference dataset_utils.py) generated on the device, error-map
                  guided sampling and update_error_map
    dist          ray sharding + flat-buffer gradient all-reduce (one process per GPU)
    optim         Adam over the flat parameter / gradient buffers (CUDA kernel)
    losses        lidar_loss / rgb_loss of the reference's train_step, loss + derivative in one kernel
    chamfer       drop-in for reference ``nvsf.nerf.chamfer3D.dist_chamfer_3D`` (chamfer_3DDist)
    metrics       evaluation on the device: lidar_points (range image -> point cloud), range_image (point cloud ->
                  range image, the images_lidar ground truth), LidarMeter / CameraMeter
    mesh          mesh extraction: marching_cubes on the device (drop-in for mcubes) and write_ply
    _lib          ctypes binding of the C ABI (include/nvsf_b200.h)
    build         compiles csrc/*.cu into libnvsf_b200.so with nvcc (sm_100a)
"""
from . import _lib  # noqa: F401
from . import raymarching  # noqa: F401
from . import field  # noqa: F401
from . import rays  # noqa: F401
from . import dist  # noqa: F401
from . import optim  # noqa: F401
from . import losses  # noqa: F401
from . import chamfer  # noqa: F401
from . import metrics  # noqa: F401
from . import mesh  # noqa: F401
from .field import NeRFNetwork  # noqa: F401

__version__ = "0.1.0"
