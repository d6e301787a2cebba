"""TEST INFRASTRUCTURE — float64 numpy / scipy restatement of the evaluation metrics (DESIGN.md §3.5): range
image -> point cloud (nvsf/lib/convert.py) and the LiDAR / camera meters of nvsf/lib/error_matrices.py as the
LiDAR-NeRF / LiDAR4D meters NVSF's evaluation derives from define them.  PARITY UNPINNED: the reference's
nvsf/lib sources are not in this repository.

The images the metrics see (masked, scaled, clamped depths and intensities, and their differences) are formed
in float32, as the renderer's outputs and the device pass form them, so medians and counts compare exactly.  The
point clouds are float32 too: the contract defines a point as the fp32 beam direction times the fp32 range, and
the squared distance of two nearby points 70 m out keeps only a few bits of fp32 coordinates, so a float64 cloud
would differ from it by more than 1e-5 at a single point.  The directions take their angles in fp32 in the
device's operation order and their sines / cosines in float64, rounded once.  Sums, means, SSIM and nearest
neighbours are float64.  SSIM follows skimage.metrics.structural_similarity's defaults (7x7 uniform window,
K1 = 0.01, K2 = 0.03, sample covariance, 3-pixel crop) on scipy.ndimage.uniform_filter.

Only tests/ and tools/bench_eval.py import this module.
"""
import numpy as np
from scipy import ndimage
from scipy.spatial import cKDTree

f32 = np.float32


def lidar_dirs(H, W, intrinsics, intrinsics_hoz):
    """[H*W, 3] float32 beam directions of get_lidar_rays at the identity pose, row-major pixels
    (dataset_utils.py:512-530): angles in fp32 in the order nvsf_get_lidar_rays evaluates them, sin / cos of
    those angles in float64 rounded to fp32, the products cos a cos b / cos a sin b in fp32."""
    p = np.arange(H * W, dtype=np.int64)
    i, j = (p % W).astype(f32), (p // W).astype(f32)
    fov_up, fov, fov_hoz = f32(intrinsics[0]), f32(intrinsics[1]), f32(intrinsics_hoz[1])
    pi = f32(np.pi)
    beta = -(i - f32(W) * f32(0.5)) / f32(W) * fov_hoz / f32(180) * pi
    alpha = (fov_up - j / f32(H) * fov) / f32(180) * pi
    a, b = alpha.astype(np.float64), beta.astype(np.float64)
    ca, sa, cb, sb = (v.astype(f32) for v in (np.cos(a), np.sin(a), np.cos(b), np.sin(b)))
    return np.stack([ca * cb, ca * sb, sa], -1)


def lidar_points(depth, intrinsics, intrinsics_hoz, scale=1.0, raydrop=None, intensity=None, raydrop_threshold=0.5):
    """points [count, 3|4] of the pixels whose depth * (raydrop > threshold) is non-zero, row-major: direction
    times depth / scale in fp32 (returned as float64, with the intensity as a 4th column when given)."""
    H, W = depth.shape[-2:]
    d = np.asarray(depth, f32).reshape(-1)
    if raydrop is not None:
        d = d * (np.asarray(raydrop, f32).reshape(-1) > raydrop_threshold).astype(f32)
    keep = np.nonzero(d != 0)[0]
    r = d[keep] / f32(scale)
    pts = (lidar_dirs(H, W, intrinsics, intrinsics_hoz)[keep] * r[:, None]).astype(np.float64)
    if intensity is not None:
        pts = np.concatenate([pts, np.asarray(intensity, f32).reshape(-1)[keep, None].astype(np.float64)], 1)
    return pts


def ssim(x, y, data_range):
    """skimage.metrics.structural_similarity(x, y, data_range=data_range) of 2-D images (defaults); NaN for
    images smaller than the 7x7 window (skimage raises there)."""
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    if min(x.shape) < 7:
        return float("nan")
    win, pad = 7, 3
    cov = win * win / (win * win - 1.0)
    ux, uy = ndimage.uniform_filter(x, win), ndimage.uniform_filter(y, win)
    uxx, uyy, uxy = (ndimage.uniform_filter(a, win) for a in (x * x, y * y, x * y))
    vx, vy, vxy = cov * (uxx - ux * ux), cov * (uyy - uy * uy), cov * (uxy - ux * uy)
    R = float(data_range)
    C1, C2 = (0.01 * R) ** 2, (0.03 * R) ** 2
    S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2))
    return float(S[pad:-pad, pad:-pad].mean())


def psnr(mse, peak):
    return float("inf") if mse == 0 else float(10 * np.log10(peak * peak / mse))


def fscore(p, r):
    return 0.0 if p + r == 0 else 2 * p * r / (p + r)


def chamfer(pred_pts, gt_pts, threshold=0.05):
    """(chamfer = mean d1 + mean d2, fscore of precision mean(d1 < t) / recall mean(d2 < t)) on squared
    nearest-neighbour distances; (+inf, 0) when either cloud is empty."""
    if len(pred_pts) == 0 or len(gt_pts) == 0:
        return float("inf"), 0.0
    d1 = cKDTree(gt_pts).query(pred_pts)[0] ** 2
    d2 = cKDTree(pred_pts).query(gt_pts)[0] ** 2
    return float(d1.mean() + d2.mean()), fscore(float((d1 < threshold).mean()), float((d2 < threshold).mean()))


def lidar_metrics(depth_lidar, image_lidar, images_lidar, intrinsics, intrinsics_hoz, scale, max_depth=80.0,
                  fscore_threshold=0.05):
    """LidarMeter's row as a dict: depth_lidar [H,W], image_lidar [H,W,2] (raydrop probability, intensity),
    images_lidar [H,W,3] (raydrop mask, intensity, depth)."""
    dh = np.asarray(depth_lidar, f32)
    H, W = dh.shape[-2:]
    dh = dh.reshape(H, W)
    im = np.asarray(image_lidar, f32).reshape(H, W, 2)
    gt = np.asarray(images_lidar, f32).reshape(H, W, 3)
    r, it, dt = gt[..., 0], gt[..., 1], gt[..., 2]
    mh = (im[..., 0] > 0.5).astype(f32)
    P, G = (dh * mh) / f32(scale), (dt * r) / f32(scale)
    Pc, Gc = np.clip(P, f32(1e-3), f32(max_depth)), np.clip(G, f32(1e-3), f32(max_depth))
    Ip, Ig = np.clip(im[..., 1] * mh, f32(1e-6), f32(1)), np.clip(it * r, f32(1e-6), f32(1))
    ed, ei = Gc - Pc, Ig - Ip
    mse_d, mse_i = np.mean(ed.astype(np.float64) ** 2), np.mean(ei.astype(np.float64) ** 2)
    pos, tpos = mh != 0, r > 0.5
    tp, fp, fn = np.sum(pos & tpos), np.sum(pos & ~tpos), np.sum(~pos & tpos)
    prec = tp / (tp + fp) if tp + fp else 0.0
    rec = tp / (tp + fn) if tp + fn else 0.0
    pp = lidar_points(P, intrinsics, intrinsics_hoz)
    pg = lidar_points(G, intrinsics, intrinsics_hoz)
    ch, fs = chamfer(pp, pg, fscore_threshold)
    return {
        "depth_rmse": float(np.sqrt(mse_d)), "depth_medae": float(np.median(np.abs(ed))),
        "depth_psnr": psnr(mse_d, float(max_depth)),
        "depth_ssim": ssim(Pc, Gc, float(Gc.max()) - float(Gc.min())),
        "intensity_rmse": float(np.sqrt(mse_i)), "intensity_medae": float(np.median(np.abs(ei))),
        "intensity_psnr": psnr(mse_i, 1.0),
        "intensity_ssim": ssim(Ip, Ig, float(Ig.max()) - float(Ig.min())),
        "raydrop_rmse": float(np.sqrt(np.mean((r.astype(np.float64) - mh) ** 2))),
        "raydrop_acc": float(np.mean(pos == tpos)), "raydrop_f1": fscore(float(prec), float(rec)),
        "chamfer": ch, "fscore": fs, "points_pred": float(len(pp)), "points_gt": float(len(pg)),
    }


def camera_metrics(pred, gt):
    """CameraMeter's row: PSNR = -10 log10(MSE), SSIM = mean of the per-channel SSIMs (data range 1)."""
    p, g = np.asarray(pred, f32), np.asarray(gt, f32)
    mse = np.mean((p - g).astype(np.float64) ** 2)
    return {"psnr": psnr(mse, 1.0), "ssim": float(np.mean([ssim(p[..., c], g[..., c], 1.0) for c in range(3)]))}
