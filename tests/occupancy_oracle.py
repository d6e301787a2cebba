"""TEST INFRASTRUCTURE — numpy fp32 restatement of the occupancy-grid maintenance beyond the full update
(DESIGN.md §3.5 "Untrained cells and the partial update"): the coverage tests of nvsf_grid_coverage_camera /
_lidar with the kernel's operation order, nvsf_grid_apply_marks, the draw hash of nvsf_grid_draws and torch-ngp's
partial update.  Built on oracle/scene_oracle.py (cell points, the full grid update).  Parity unpinned: the
reference has no such routine.  Only tests may import this module."""
import numpy as np

from oracle.scene_oracle import grid_cell_points, grid_update

f32 = np.float32


# ------------------------------------------------------------------------ untrained-cell marking
def _sensor_points(C, H, bound, pose):
    """(p [n,3] = R^T (x - t) of every cell centre, margin m [n]) in fp32, each product / sum rounded alone."""
    x = grid_cell_points(C, H, bound)
    P = np.asarray(pose, f32)
    d = x - P[:3, 3][None, :]
    p = np.empty_like(d)
    for a in range(3):
        p[:, a] = (P[0, a] * d[:, 0] + P[1, a] * d[:, 1]) + P[2, a] * d[:, 2]
    bc = np.array([min(2 ** c, bound) for c in range(C)], f32)
    m = np.repeat(f32(2) * bc / f32(H), H ** 3)
    return p, m


def camera_slopes(fx, fy, cx, cy, img_H, img_W):
    """(sl, sr, st, sb): computed in float64 from the fp32 intrinsics, rounded to fp32 once."""
    fx, fy, cx, cy = (float(f32(v)) for v in (fx, fy, cx, cy))
    return (f32(-cx / fx), f32((img_W - cx) / fx), f32(-cy / fy), f32((img_H - cy) / fy))


def lidar_constants(fov_up, fov, fov_hoz):
    """(s_lo, s_up, wedge, n1, n2) as nvsf_grid_coverage_lidar prepares them (wedge 0 / 1 / 2 = none /
    intersection / union of the two half-planes)."""
    up, fv, hoz = float(f32(fov_up)), float(f32(fov)), float(f32(fov_hoz))
    deg = np.pi / 180.0
    s_lo, s_up = f32(np.tan((up - fv) * deg)), f32(np.tan(up * deg))
    if hoz >= 360.0:
        return s_lo, s_up, 0, None, None
    h = 0.5 * hoz * deg
    sh, ch = np.sin(h), np.cos(h)
    return s_lo, s_up, (1 if hoz <= 180.0 else 2), (f32(sh), f32(ch)), (f32(sh), f32(-ch))


def grid_coverage_camera(C, H, bound, poses, fx, fy, cx, cy, img_H, img_W, covered=None):
    """Covered mask [C*H^3] (bool) of nvsf_grid_coverage_camera, OR-ed into `covered`."""
    sl, sr, st, sb = camera_slopes(fx, fy, cx, cy, img_H, img_W)
    out = np.zeros(C * H ** 3, bool) if covered is None else np.asarray(covered, bool).copy()
    for pose in np.asarray(poses, f32).reshape(-1, 4, 4):
        p, m = _sensor_points(C, H, bound, pose)
        z = p[:, 2]
        ok = (z > 0) & (p[:, 0] > sl * z - m) & (p[:, 0] < sr * z + m) & (p[:, 1] > st * z - m) & (p[:, 1] < sb * z + m)
        out |= ok
    return out


def grid_coverage_lidar(C, H, bound, poses, fov_up, fov, fov_hoz, near, far, covered=None):
    """Covered mask [C*H^3] (bool) of nvsf_grid_coverage_lidar, OR-ed into `covered`."""
    s_lo, s_up, wedge, n1, n2 = lidar_constants(fov_up, fov, fov_hoz)
    near, far = f32(near), f32(far)
    out = np.zeros(C * H ** 3, bool) if covered is None else np.asarray(covered, bool).copy()
    for pose in np.asarray(poses, f32).reshape(-1, 4, 4):
        p, m = _sensor_points(C, H, bound, pose)
        xy = p[:, 0] * p[:, 0] + p[:, 1] * p[:, 1]
        r = np.sqrt(xy + p[:, 2] * p[:, 2])
        rho = np.sqrt(xy)
        ok = (r > near - m) & (r < far + m) & (p[:, 2] > s_lo * rho - m) & (p[:, 2] < s_up * rho + m)
        if wedge:
            in1 = (n1[0] * p[:, 0] + n1[1] * p[:, 1]) > -m
            in2 = (n2[0] * p[:, 0] + n2[1] * p[:, 1]) > -m
            ok &= (in1 & in2) if wedge == 1 else (in1 | in2)
        out |= ok
    return out


def apply_marks(grid, bitfield, covered):
    """nvsf_grid_apply_marks -> (grid, bitfield, n_marked)."""
    g = np.asarray(grid, f32).reshape(-1).copy()
    cov = np.asarray(covered, bool).reshape(-1)
    g[~cov] = f32(-1)
    g[cov & (g < 0)] = f32(0)
    bf = np.asarray(bitfield, np.uint8) & np.packbits(cov, bitorder="little")
    return g, bf, int((~cov).sum())


# ------------------------------------------------------------------------ partial update (torch-ngp)
_M64 = (1 << 64) - 1


def splitmix64(x):
    """splitmix64 on uint64 arrays (wrapping arithmetic)."""
    z = np.asarray(x, np.uint64) + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def grid_draws(C, H, seed, iteration, grid):
    """The C*H^3/2 cells of nvsf_grid_draws (int32, -1 for an occupied slot of a cascade with no cell > 0)."""
    H3 = H ** 3
    Q = H3 // 4
    g = np.asarray(grid, f32).reshape(C, H3)
    key = splitmix64(splitmix64(np.array([int(seed) & _M64], np.uint64)) ^ np.uint64(int(iteration) & _M64))
    out = np.empty((C, 2 * Q), np.int64)
    s = np.arange(2 * Q, dtype=np.uint64)
    for c in range(C):
        hi = splitmix64(key ^ ((np.uint64(c) << np.uint64(32)) | s)) >> np.uint64(32)
        out[c, :Q] = c * H3 + ((hi[:Q] * np.uint64(H3)) >> np.uint64(32)).astype(np.int64)
        occ = np.nonzero(g[c] > 0)[0]
        if occ.size:
            out[c, Q:] = c * H3 + occ[((hi[Q:] * np.uint64(occ.size)) >> np.uint64(32)).astype(np.int64)]
        else:
            out[c, Q:] = -1
    return out.reshape(-1).astype(np.int32)


def scatter_max(n, cells, vals):
    """tmp [n] = -1, then tmp[cells[r]] = max(tmp[cells[r]], vals[r]) for cells[r] >= 0."""
    tmp = np.full(n, f32(-1))
    cells = np.asarray(cells, np.int64)
    keep = cells >= 0
    np.maximum.at(tmp, cells[keep], np.asarray(vals, f32)[keep])
    return tmp


def cell_points_list(C, H, bound, cells, noise=None):
    """Points of the listed cells (the origin for a negative id); noise rows by list position."""
    cells = np.asarray(cells, np.int64)
    allp = grid_cell_points(C, H, bound)
    out = np.zeros((cells.size, 3), f32)
    ok = cells >= 0
    out[ok] = allp[cells[ok]]
    if noise is not None:
        half = np.array([min(2 ** c, bound) for c in range(C)], f32)[cells[ok] // H ** 3] / f32(H)
        out[ok] = out[ok] + (np.asarray(noise, f32)[ok] * f32(2) - f32(1)) * half[:, None]
    return out


def partial_update(grid, cells, vals, decay, density_thresh):
    """torch-ngp's partial update given the drawn cells and their values sigma * density_scale (max over the
    times): -> grid_update's (grid, mean, thresh, bitfield)."""
    g = np.asarray(grid, f32).reshape(-1)
    return grid_update(g, scatter_max(g.size, cells, vals), decay, density_thresh)
