"""Ray generation on the device: the reference's ``get_lidar_rays`` / ``get_rays``
(nvsf/nerf/dataset/dataset_utils.py:369-536, 539-687) with the same arguments and result dict.

Pixel selection (which ids to render) stays a torch RNG call exactly like the reference's
(`torch.randint(0, H*W, [N])`, so a seeded run picks the same pixels); turning pixel ids and a pose
into origins and directions is one kernel launch per pose (`nvsf_get_lidar_rays` /
`nvsf_get_rays`) instead of ~20 ATen launches over [B, H*W] meshgrids.

Error-map guided selection (`use_error_map=True`, torch-ngp's convention; DESIGN.md §3.5): per pose,
`nvsf_error_map_sample` draws N distinct coarse cells of the [res*res] map with probability
proportional to it and one jittered pixel in each, from exponential and uniform draws of torch's CUDA
generator; `update_error_map` folds the per-ray loss back into the trainer's maps
(map = 0.1 * map + 0.9 * loss).  Neither reads anything back to the host, so a training step that
uses them stays free of host syncs and can be captured in a CUDA graph.
"""
import math

import torch

from . import _lib
from ._lib import NvsfError, check, ptr, stream_ptr


def _patch(patch_size):
    if isinstance(patch_size, int):
        return patch_size, patch_size
    if len(patch_size) == 1:
        return patch_size[0], patch_size[0]
    return tuple(patch_size)


def _select(H, W, N, patch_size, device):
    """Pixel ids [n] (int64) or None for the full image in row-major order."""
    if N <= 0:
        return None
    N = min(N, H * W)
    ph, pw = _patch(patch_size)
    if ph > 1:  # random patches, top-left corners may repeat (dataset_utils.py:444-465)
        num_patch = N // (ph * pw)
        inds_x = torch.randint(0, W - pw, size=[num_patch], device=device)
        inds_y = torch.randint(0, H - ph, size=[num_patch], device=device)
        oy, ox = torch.meshgrid(torch.arange(ph, device=device), torch.arange(pw, device=device), indexing="ij")
        rows = inds_y[:, None] + oy.reshape(1, -1)
        cols = inds_x[:, None] + ox.reshape(1, -1)
        return (rows * W + cols).reshape(-1)
    return torch.randint(0, H * W, size=[N], device=device)


def _error_map_select(error_map, B, H, W, N, dev):
    """torch-ngp's error-map branch: inds [B,N] and inds_coarse [B,N] (ascending cells per row)."""
    L = _lib.lib()
    N = min(N, H * W)
    if error_map.dim() != 2 or error_map.shape[0] != B:
        raise NvsfError(f"get_rays: error_map must be [B={B}, res*res], got {list(error_map.shape)}")
    R = error_map.shape[1]
    res = math.isqrt(R)
    if res * res != R:
        raise NvsfError(f"get_rays: error_map has {R} cells per map, not a square number")
    if N > R:
        raise NvsfError(f"get_rays: N={N} distinct cells cannot be drawn from a map of {R} cells")
    w = error_map.detach().to(dev, torch.float32).contiguous()
    expo = torch.empty(B, R, dtype=torch.float32, device=dev).exponential_()
    jitter = torch.rand(B, N, 2, dtype=torch.float32, device=dev)
    inds_coarse = torch.empty(B, N, dtype=torch.int64, device=dev)
    inds = torch.empty(B, N, dtype=torch.int64, device=dev)
    for b in range(B):
        check(L.nvsf_error_map_sample(ptr(w[b]), ptr(expo[b]), ptr(jitter[b]), res, N, H, W, ptr(inds_coarse[b]),
                                      ptr(inds[b]), stream_ptr()), "error_map_sample")
    return inds, inds_coarse


def _generate(kind, poses, scalars, H, W, N, patch_size, error_map, use_error_map):
    L = _lib.lib()
    if not poses.is_cuda:
        poses = poses.cuda()
    poses = poses.detach().to(torch.float32).contiguous()
    dev = poses.device
    B = poses.shape[0]
    if use_error_map and N > 0:
        if error_map is None or _patch(patch_size)[0] > 1:
            raise NotImplementedError("error-map guided sampling needs an error_map and single-pixel sampling "
                                      "(patch_size 1)")
        inds, inds_coarse = _error_map_select(error_map, B, H, W, N, dev)
        n, rows = inds.shape[1], inds
    else:
        sel = _select(H, W, N, patch_size, dev)
        n = H * W if sel is None else sel.shape[0]
        rows, inds_coarse = [sel] * B, None
        inds = (torch.arange(H * W, device=dev) if sel is None else sel).expand([B, n])
    rays_o = torch.empty(B, n, 3, dtype=torch.float32, device=dev)
    rays_d = torch.empty(B, n, 3, dtype=torch.float32, device=dev)
    fn = L.nvsf_get_lidar_rays if kind == "lidar" else L.nvsf_get_rays
    for b in range(B):
        check(fn(ptr(poses[b]), ptr(rows[b]), n, H, W, *scalars, ptr(rays_o[b]), ptr(rays_d[b]), stream_ptr()),
              f"get_{kind}_rays")
    out = {"rays_o": rays_o, "rays_d": rays_d, "inds": inds}
    if inds_coarse is not None:
        out["inds_coarse"] = inds_coarse
    return out


@torch.no_grad()
def get_lidar_rays(poses, intrinsics, intrinsics_hoz, H, W, N=-1, patch_size=1, error_map=None,
                   use_error_map=False):
    """poses [B,4,4] lidar2world; intrinsics = (fov_up, fov) and intrinsics_hoz = (fov_up, fov) in
    degrees -> {'rays_o' [B,n,3], 'rays_d' [B,n,3], 'inds' [B,n]}.

    With N > 0, `use_error_map=True` and `error_map` [B, res*res] (one map per pose, ideally on the
    device), the N pixels are drawn from N distinct coarse cells with probability proportional to the
    map (torch-ngp's error-map sampling) and the dict also holds 'inds_coarse' [B,N], the cells in
    ascending order per row (not in draw order: the drawn set has the same distribution).  The draws
    are torch.empty(B, R).exponential_() and then torch.rand(B, N, 2) from the current CUDA generator."""
    fov_up, fov = float(intrinsics[0]), float(intrinsics[1])
    fov_hoz = float(intrinsics_hoz[1])
    return _generate("lidar", poses, (fov_up, fov, fov_hoz), H, W, N, patch_size, error_map, use_error_map)


@torch.no_grad()
def get_rays(poses, intrinsics, H, W, N=-1, patch_size=1, error_map=None, use_error_map=False):
    """poses [B,4,4] cam2world; intrinsics = 3x3 (or 3x4) pinhole matrix.  Error-map sampling as
    get_lidar_rays."""
    fx, fy = float(intrinsics[0][0]), float(intrinsics[1][1])
    cx, cy = float(intrinsics[0][2]), float(intrinsics[1][2])
    return _generate("camera", poses, (fx, fy, cx, cy), H, W, N, patch_size, error_map, use_error_map)


@torch.no_grad()
def update_error_map(error_maps, index, inds_coarse, loss):
    """torch-ngp's error-map update after the loss head, in place and without a host sync: for each
    batch row b, error_maps[index[b], c] = 0.1 * error_maps[index[b], c] + 0.9 * loss[b, j] at the cells
    c = inds_coarse[b, j] that row was drawn from.

    error_maps [F, R] fp32 contiguous CUDA tensor (one map per training frame); index: the frames of the
    batch (data['index']: host ints, distinct); inds_coarse [B, N] as get_lidar_rays / get_rays return it;
    loss [B, N] per ray (lidar_loss as is, rgb_loss(...).mean(-1) for the camera)."""
    if not (isinstance(error_maps, torch.Tensor) and error_maps.is_cuda and error_maps.dtype == torch.float32
            and error_maps.dim() == 2 and error_maps.is_contiguous()):
        raise NvsfError("update_error_map: error_maps must be a contiguous [F, R] float32 CUDA tensor")
    if isinstance(index, torch.Tensor):
        if index.is_cuda:
            raise NvsfError("update_error_map: index must be host ints (data['index']), not a CUDA tensor")
        index = index.reshape(-1).tolist()
    elif isinstance(index, int):
        index = [index]
    index = [int(i) for i in index]
    F, R = error_maps.shape
    if len(set(index)) != len(index) or any(i < 0 or i >= F for i in index):
        raise NvsfError(f"update_error_map: index {index} must be distinct frames in [0, {F})")
    B = len(index)
    if inds_coarse.dim() != 2 or inds_coarse.shape[0] != B or tuple(loss.shape) != tuple(inds_coarse.shape):
        raise NvsfError(f"update_error_map: inds_coarse {list(inds_coarse.shape)} and loss {list(loss.shape)} "
                        f"must both be [B={B}, N]")
    if inds_coarse.device != error_maps.device or loss.device != error_maps.device:
        raise NvsfError("update_error_map: error_maps, inds_coarse and loss must be on the same device")
    ic = inds_coarse.to(torch.int64).contiguous()
    e = loss.detach().to(torch.float32).contiguous()
    N = ic.shape[1]
    L = _lib.lib()
    for b, f in enumerate(index):
        check(L.nvsf_error_map_update(ptr(error_maps[f]), R, ptr(ic[b]), N, ptr(e[b]), stream_ptr()),
              "error_map_update")
