"""TEST INFRASTRUCTURE — numpy restatement of point cloud -> range image (metrics.range_image, DESIGN.md §3.5), the
inverse of metrics_oracle.lidar_points and the projection that builds every images_lidar ground truth.  PARITY
UNPINNED: the reference's nvsf/lib/convert.py is not in this repository; this restates its per-point loop with the
pixel convention of get_lidar_rays.

Every step is float64 from the fp32 inputs, in the contract's order, each operation rounded on its own (numpy and
Python never contract a multiply-add); depth is rounded to fp32 once.  Two forms: `range_image_loop`, the literal
per-point loop (math.atan2, Python's round = half to even), for small clouds, and `range_image`, vectorised (keep,
then np.lexsort by pixel, depth bits, index and take the first of each pixel).  Both call the host's atan2, so they
agree bit for bit; the device's double atan2 (within 2 ulp) can land elsewhere only for a point within ~1e-13 px of
a half-integer column or row.

Only tests/ and tools/bench_range_image.py import this module.
"""
import math

import numpy as np

f32 = np.float32
DEG = 180.0 / math.pi


def _fovs(intrinsics, intrinsics_hoz):
    return float(f32(intrinsics[0])), float(f32(intrinsics[1])), float(f32(intrinsics_hoz[1]))


def _offsets(points, offsets):
    return [0, len(points)] if offsets is None else [int(o) for o in offsets]


def _pose(poses, b):
    """(R [3][3], t [3]) of scan b as float64 of the fp32 pose, or None."""
    if poses is None:
        return None
    p = np.asarray(poses, f32).reshape(-1, 4, 4)[b].astype(np.float64)
    return p[:3, :3], p[:3, 3]


def _finish(images, index, offsets):
    return (images[0], index[0]) if offsets is None else (images, index)


def range_image_loop(points, H, W, intrinsics, intrinsics_hoz, scale=1.0, max_depth=80.0, offsets=None, poses=None):
    """(images [B,H,W,3] fp32, index [B,H,W] int64) — [H,W,3] / [H,W] without offsets — by the per-point loop."""
    pts = np.asarray(points, f32)
    offs = _offsets(pts, offsets)
    B, C = len(offs) - 1, pts.shape[1]
    fov_up, fov, fh = _fovs(intrinsics, intrinsics_hoz)
    md, sc = f32(max_depth), f32(scale)
    images = np.zeros((B, H, W, 3), f32)
    index = np.full((B, H, W), -1, np.int64)
    best = np.zeros((B, H, W), f32)
    for b in range(B):
        pose = _pose(poses, b)
        for g in range(offs[b], offs[b + 1]):
            x, y, z = (float(v) for v in pts[g, :3])
            if pose is not None:
                R, t = (v.tolist() for v in pose)
                dx, dy, dz = x - t[0], y - t[1], z - t[2]
                x, y, z = ((R[0][k] * dx + R[1][k] * dy) + R[2][k] * dz for k in range(3))
            xy2 = x * x + y * y
            s = xy2 + z * z
            with np.errstate(over="ignore"):
                d = f32(math.sqrt(s)) if math.isfinite(s) else f32(math.nan)
            if not (d > 0 and d < md):
                continue
            beta, alpha = math.atan2(y, x) * DEG, math.atan2(z, math.sqrt(xy2)) * DEG
            c = round(((0.5 * fh - beta) / fh) * W)
            r = round(((fov_up - alpha) / fov) * H)
            if not (0 <= r < H and 0 <= c < W):
                continue
            if index[b, r, c] < 0 or best[b, r, c] > d:   # the reference's strict `pano[r, c] > dist`
                best[b, r, c] = d
                index[b, r, c] = g
                images[b, r, c] = (1.0, pts[g, 3] if C == 4 else 0.0, d * sc)
    return _finish(images, index, offsets)


def range_image(points, H, W, intrinsics, intrinsics_hoz, scale=1.0, max_depth=80.0, offsets=None, poses=None):
    """The same as range_image_loop, vectorised."""
    pts = np.asarray(points, f32)
    offs = _offsets(pts, offsets)
    B, C = len(offs) - 1, pts.shape[1]
    fov_up, fov, fh = _fovs(intrinsics, intrinsics_hoz)
    counts = np.diff(offs)
    scan = np.repeat(np.arange(B), counts)
    q = pts[:, :3].astype(np.float64)
    if poses is not None:
        P = np.asarray(poses, f32).reshape(-1, 4, 4).astype(np.float64)[scan]
        d = q - P[:, :3, 3]
        q = np.stack([(P[:, 0, k] * d[:, 0] + P[:, 1, k] * d[:, 1]) + P[:, 2, k] * d[:, 2] for k in range(3)], 1)
    x, y, z = q[:, 0], q[:, 1], q[:, 2]
    with np.errstate(over="ignore", invalid="ignore"):
        xy2 = x * x + y * y
        depth = np.sqrt(xy2 + z * z).astype(f32)
        keep = (depth > 0) & (depth < f32(max_depth))
        beta = np.arctan2(y, x) * DEG
        alpha = np.arctan2(z, np.sqrt(xy2)) * DEG
        c = np.rint(((0.5 * fh - beta) / fh) * W)
        r = np.rint(((fov_up - alpha) / fov) * H)
        keep &= (c >= 0) & (c < W) & (r >= 0) & (r < H)
    g = np.nonzero(keep)[0]
    pix = scan[g] * (H * W) + r[g].astype(np.int64) * W + c[g].astype(np.int64)
    order = np.lexsort((g, depth[g].view(np.uint32), pix))
    pix, g = pix[order], g[order]
    first = np.ones(len(pix), bool)
    first[1:] = pix[1:] != pix[:-1]
    pix, g = pix[first], g[first]
    images = np.zeros((B * H * W, 3), f32)
    index = np.full(B * H * W, -1, np.int64)
    images[pix, 0] = 1.0
    if C == 4:
        images[pix, 1] = pts[g, 3]
    images[pix, 2] = depth[g] * f32(scale)
    index[pix] = g
    return _finish(images.reshape(B, H, W, 3), index.reshape(B, H, W), offsets)
