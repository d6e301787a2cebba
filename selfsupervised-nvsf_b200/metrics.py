"""Evaluation of rendered frames on the device: the synthesized LiDAR scan (range image -> point cloud) and
the per-frame meters of the reference's evaluation (Trainer.evaluate_one_epoch / test_step, trainer.py:817-903,
1458-1846, meters nvsf/lib/error_matrices.py, conversion nvsf/lib/convert.py), over C ABI Part 6 (csrc/eval.cu).

The reference copies every rendered frame to the host and scores it with numpy; here a frame's scoring is a
fixed sequence of kernels in the current stream that writes one metric row to device memory, so evaluation
reads nothing back per frame.  ``summary()`` is the one host read of an epoch.  The metric definitions are
DESIGN.md §3.5; they restate the LiDAR-NeRF / LiDAR4D meters (parity unpinned: the reference's nvsf/lib is not
in this repository).  GPU tensors only; no CPU fallback.
"""
import math

import torch

from . import _lib
from ._lib import NvsfError, check, ptr, stream_ptr

LIDAR_METRICS = ("depth_rmse", "depth_medae", "depth_psnr", "depth_ssim",
                 "intensity_rmse", "intensity_medae", "intensity_psnr", "intensity_ssim",
                 "raydrop_rmse", "raydrop_acc", "raydrop_f1",
                 "chamfer", "fscore", "points_pred", "points_gt")
CAMERA_METRICS = ("psnr", "ssim")


def _frame(t, H, W, C, what):
    """`t` as a contiguous fp32 [H*W*C] view (any shape with H*W*C elements, e.g. [H,W,C] or [1,H*W,C])."""
    if not torch.is_tensor(t) or not t.is_cuda:
        raise NvsfError(f"{what}: GPU tensors only")
    if t.numel() != H * W * C:
        raise NvsfError(f"{what}: {tuple(t.shape)} does not hold a {H}x{W}x{C} frame")
    return t.detach().to(torch.float32).reshape(-1).contiguous()


def _fovs(intrinsics, intrinsics_hoz):
    """(fov_up, fov, fov_hoz) in degrees, as get_lidar_rays reads them."""
    return float(intrinsics[0]), float(intrinsics[1]), float(intrinsics_hoz[1])


@torch.no_grad()
@_lib.device_guard
def lidar_points(depth, intrinsics, intrinsics_hoz, scale=1.0, raydrop=None, intensity=None, raydrop_threshold=0.5):
    """Range image -> point cloud in the sensor frame (convert.py): depth [H,W] (e.g. render_frame(...,
    cal_lidar_color=True)["depth_lidar"]); optional raydrop probability and intensity [H,W] (its
    ["image_lidar"][..., 0] / [..., 1]).  Pixels whose depth * (raydrop > raydrop_threshold) is non-zero become
    rows get_lidar_rays(identity).rays_d * (depth / scale), in row-major pixel order (np.where order), with the
    intensity as a 4th column when given.  Returns (points [H*W, 3|4] — rows past the count are zero,
    count — int32 device scalar); nothing is read back to the host."""
    if depth.dim() < 2:
        raise NvsfError("lidar_points: depth must be [H, W]")
    H, W = int(depth.shape[-2]), int(depth.shape[-1])
    d = _frame(depth, H, W, 1, "lidar_points depth")
    r = None if raydrop is None else _frame(raydrop, H, W, 1, "lidar_points raydrop")
    it = None if intensity is None else _frame(intensity, H, W, 1, "lidar_points intensity")
    L = _lib.lib()
    wb = L.nvsf_lidar_points_workspace_bytes(H, W)
    if wb == 0:
        raise NvsfError(f"lidar_points: frame {H}x{W} out of range")
    points = torch.empty(H * W, 3 if it is None else 4, dtype=torch.float32, device=d.device)
    count = torch.empty((), dtype=torch.int32, device=d.device)
    ws = torch.empty(wb, dtype=torch.uint8, device=d.device)
    check(L.nvsf_lidar_points(ptr(d), ptr(r), float(raydrop_threshold), ptr(it), H, W, *_fovs(intrinsics, intrinsics_hoz),
                              float(scale), ptr(points), ptr(count), ptr(ws), wb, stream_ptr()), "lidar_points")
    return points, count


def summarize(rows, names, process_group=None):
    """{name: mean over frames} of `rows` [frames, len(names)].  When torch.distributed is initialized the
    per-metric sums and the frame count are all-reduced over `process_group` (default: the world), so every
    rank gets the mean over all ranks' frames.  One host read."""
    K = len(names)
    acc = torch.zeros(K + 1, dtype=torch.float64, device=rows.device)
    if rows.shape[0]:
        acc[:K] = rows.to(torch.float64).sum(0)
        acc[K] = rows.shape[0]
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(acc, group=process_group)
    vals = acc.tolist()
    frames = vals[K]
    return {k: (vals[i] / frames if frames else math.nan) for i, k in enumerate(names)}


class _Meter:
    names = ()

    def __init__(self, H, W, ws_bytes_fn, device):
        self.H, self.W = int(H), int(W)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        wb = ws_bytes_fn(self.H, self.W) if self.H > 0 and self.W > 0 else 0
        if wb == 0:
            raise NvsfError(f"{type(self).__name__}: frame {H}x{W} out of range")
        # one workspace for every update: updates of one meter run in one stream, one after another
        self._ws = torch.empty(wb, dtype=torch.uint8, device=self.device)
        self._rows = []

    def _new_row(self):
        row = torch.empty(len(self.names), dtype=torch.float32, device=self.device)
        self._rows.append(row)
        return row

    def frame_results(self):
        """Device tensor [frames, K] of the rows stored by update(), columns `names`."""
        if not self._rows:
            return torch.empty(0, len(self.names), dtype=torch.float32, device=self.device)
        return torch.stack(self._rows)

    def summary(self, process_group=None):
        """{metric: mean over frames} (all ranks' frames under torch.distributed; see summarize)."""
        return summarize(self.frame_results(), self.names, process_group)

    def reset(self):
        self._rows = []


class LidarMeter(_Meter):
    """Per-frame LiDAR metrics of a full range image (DESIGN.md §3.5): depth and intensity RMSE / MedAE /
    PSNR / SSIM, ray-drop RMSE / accuracy / F1, Chamfer distance and F-score of the synthesized vs the
    ground-truth point cloud, and the two point counts.  intrinsics / intrinsics_hoz are get_lidar_rays's
    (fov_up, fov) pairs in degrees; scale is the scene scale the depths are divided by."""
    names = LIDAR_METRICS

    def __init__(self, H, W, intrinsics, intrinsics_hoz, scale, max_depth=80.0, fscore_threshold=0.05, device=None):
        super().__init__(H, W, _lib.lib().nvsf_eval_lidar_workspace_bytes, device)
        self.fovs = _fovs(intrinsics, intrinsics_hoz)
        self.scale, self.max_depth, self.fscore_threshold = float(scale), float(max_depth), float(fscore_threshold)

    @torch.no_grad()
    @_lib.device_guard
    def update(self, depth_lidar, image_lidar, images_lidar):
        """Score one frame: depth_lidar [H,W] and image_lidar [H,W,2] (raydrop probability, intensity) as
        render_frame returns them, images_lidar [H,W,3] = ground truth (raydrop mask, intensity, depth) as
        lidar_loss takes it.  Enqueues the work in the current stream, stores the row and returns it ([K]
        device tensor); no host synchronisation."""
        H, W = self.H, self.W
        d = _frame(depth_lidar, H, W, 1, "LidarMeter depth_lidar")
        im = _frame(image_lidar, H, W, 2, "LidarMeter image_lidar")
        gt = _frame(images_lidar, H, W, 3, "LidarMeter images_lidar")
        if d.device != self.device or im.device != self.device or gt.device != self.device:
            raise NvsfError(f"LidarMeter: inputs must be on {self.device}")
        row = self._new_row()
        check(_lib.lib().nvsf_eval_lidar(ptr(d), ptr(im), ptr(gt), H, W, *self.fovs, self.scale, self.max_depth,
                                         self.fscore_threshold, ptr(row), ptr(self._ws), self._ws.numel(),
                                         stream_ptr()), "LidarMeter.update")
        return row


class CameraMeter(_Meter):
    """Per-frame camera PSNR (-10 log10 MSE on [0, 1]) and SSIM (mean of the per-channel SSIMs, data range 1)
    of [H,W,3] images."""
    names = CAMERA_METRICS

    def __init__(self, H, W, device=None):
        super().__init__(H, W, _lib.lib().nvsf_eval_camera_workspace_bytes, device)

    @torch.no_grad()
    @_lib.device_guard
    def update(self, pred, gt):
        """Score one frame: pred, gt [H,W,3].  Enqueues the work, stores the row and returns it ([2])."""
        p = _frame(pred, self.H, self.W, 3, "CameraMeter pred")
        g = _frame(gt, self.H, self.W, 3, "CameraMeter gt")
        if p.device != self.device or g.device != self.device:
            raise NvsfError(f"CameraMeter: inputs must be on {self.device}")
        row = self._new_row()
        check(_lib.lib().nvsf_eval_camera(ptr(p), ptr(g), self.H, self.W, ptr(row), ptr(self._ws), self._ws.numel(),
                                          stream_ptr()), "CameraMeter.update")
        return row
