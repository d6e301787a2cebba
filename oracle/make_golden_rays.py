"""TEST INFRASTRUCTURE (build container only): golden vectors for ray generation.

Imports the reference's own nvsf/nerf/dataset/dataset_utils.py by file path, unchanged (stubs for
the modules it imports at the top but does not use in get_lidar_rays / get_rays: torch_ema,
trimesh, matplotlib, nvsf.lib), runs get_lidar_rays / get_rays on CPU for seeded poses and pixel
selections, and stores inputs + outputs in tests/golden/rays_ref.npz.

    python -m oracle.make_golden_rays
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

REF = "/root/reference/nvsf/nerf/dataset/dataset_utils.py"
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden", "rays_ref.npz")


def import_dataset_utils():
    def stub(name, **attrs):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = []
            sys.modules[name] = m
        for k, v in attrs.items():
            setattr(sys.modules[name], k, v)
        return sys.modules[name]

    stub("torch_ema", ExponentialMovingAverage=object)
    stub("trimesh")
    stub("matplotlib")
    stub("matplotlib.pyplot")
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    stub("nvsf")
    stub("nvsf.lib", convert=stub("nvsf.lib.convert"), tools=stub("nvsf.lib.tools"))
    spec = importlib.util.spec_from_file_location("ref_dataset_utils", REF)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def pose(seed):
    rng = np.random.default_rng(seed)
    from scipy.spatial.transform import Rotation
    P = np.eye(4, dtype=np.float32)
    P[:3, :3] = Rotation.from_euler("zyx", rng.uniform(-np.pi, np.pi, 3) * [1.0, 0.1, 0.1]).as_matrix()
    P[:3, 3] = rng.uniform(-0.3, 0.3, 3)
    return P


def main():
    du = import_dataset_utils()
    out = {}
    # KITTI-360 shapes (SURVEY.md §8d): LiDAR 66x1030, fov_up 2.0, fov 26.9, 360 deg; camera 376x1408
    lidar_K, lidar_K_hoz = [2.0, 26.9], [180.0, 360.0]
    cam_K = np.array([[552.554261, 0, 682.049453], [0, 552.554261, 238.769549], [0, 0, 1]], np.float32)
    for tag, seed in (("a", 0), ("b", 1)):
        P = pose(seed)
        out[f"pose_{tag}"] = P
        Pt = torch.from_numpy(P)[None]
        r = du.get_lidar_rays(Pt, lidar_K, lidar_K_hoz, 66, 1030, -1)
        out[f"lidar_full_{tag}_o"], out[f"lidar_full_{tag}_d"] = r["rays_o"][0].numpy(), r["rays_d"][0].numpy()
        torch.manual_seed(seed)
        r = du.get_lidar_rays(Pt, lidar_K, lidar_K_hoz, 66, 1030, 4096)
        out[f"lidar_batch_{tag}_inds"] = r["inds"][0].numpy()
        out[f"lidar_batch_{tag}_o"], out[f"lidar_batch_{tag}_d"] = r["rays_o"][0].numpy(), r["rays_d"][0].numpy()
        torch.manual_seed(seed)
        r = du.get_rays(Pt, cam_K, 376, 1408, 4096)
        out[f"cam_batch_{tag}_inds"] = r["inds"][0].numpy()
        out[f"cam_batch_{tag}_o"], out[f"cam_batch_{tag}_d"] = r["rays_o"][0].numpy(), r["rays_d"][0].numpy()
        torch.manual_seed(seed)
        r = du.get_rays(Pt, cam_K, 376, 1408, 4096, patch_size=8)
        out[f"cam_patch_{tag}_inds"] = r["inds"][0].numpy()
        out[f"cam_patch_{tag}_d"] = r["rays_d"][0].numpy()
    # a small full camera image (all pixels, row-major)
    r = du.get_rays(torch.from_numpy(out["pose_a"])[None], cam_K, 47, 176, -1)
    out["cam_small_full_d"] = r["rays_d"][0].numpy()
    # origins are the pose translation broadcast: one copy is enough; one full LiDAR frame too, and of
    # that frame the pixels of a checkerboard (every row and column, half the bytes: the file stays < 1 MB)
    for k in [k for k in out if k.endswith("_o") and k != "lidar_batch_a_o"] + ["lidar_full_b_d"]:
        del out[k]
    out["lidar_full_a_inds"] = np.flatnonzero(np.add.outer(np.arange(66), np.arange(1030)) % 2 == 0).astype(np.int32)
    out["lidar_full_a_d"] = out["lidar_full_a_d"][out["lidar_full_a_inds"]]
    out["lidar_K"], out["lidar_K_hoz"], out["cam_K"] = np.float32(lidar_K), np.float32(lidar_K_hoz), cam_K
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
