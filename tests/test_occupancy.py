"""CPU: the untrained-cell marking and partial-update oracle (tests/occupancy_oracle.py) against float64 geometry
and torch-ngp's own camera formula, the statistics of the partial-update draws, and the C ABI's argument checks
that return before any launch."""
import ctypes
import importlib
import math

import numpy as np
import pytest

import occupancy_oracle as SO

f32 = np.float32
C, H, BOUND = 2, 16, 2.0


def _pose(yaw, t, cam=False):
    c, s = math.cos(yaw), math.sin(yaw)
    R = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    if cam:  # columns = (right, down, forward): the camera looks along the yawed +x axis
        R = R @ np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])
    P = np.eye(4)
    P[:3, :3], P[:3, 3] = R, t
    return P.astype(f32)


def _f64_points(pose):
    x = SO.grid_cell_points(C, H, BOUND).astype(np.float64)
    P = pose.astype(np.float64)
    p = (x - P[:3, 3]) @ P[:3, :3]
    bc = np.array([min(2 ** c, BOUND) for c in range(C)])
    return p, np.repeat(2 * bc / H, H ** 3)


def test_camera_coverage_matches_float64_geometry_away_from_the_margin():
    fx, fy, cx, cy, Hi, Wi = 55.0, 55.0, 68.2, 23.9, 38, 141   # off-centre principal point, like KITTI-360
    pose = _pose(0.7, (0.1, -0.2, 0.05), cam=True)
    got = SO.grid_coverage_camera(C, H, BOUND, pose[None], fx, fy, cx, cy, Hi, Wi)
    p, m = _f64_points(pose)
    z = p[:, 2]
    terms = [z, p[:, 0] - (-cx / fx * z - m), (Wi - cx) / fx * z + m - p[:, 0],
             p[:, 1] - (-cy / fy * z - m), (Hi - cy) / fy * z + m - p[:, 1]]
    want = np.all([t > 0 for t in terms], axis=0)
    clear = np.all([np.abs(t) > 1e-4 for t in terms], axis=0)
    assert clear.mean() > 0.99 and 0.05 < want.mean() < 0.95
    np.testing.assert_array_equal(got[clear], want[clear])


@pytest.mark.parametrize("fov_hoz", [360.0, 90.0, 250.0])
def test_lidar_coverage_matches_float64_geometry_away_from_the_margin(fov_hoz):
    fov_up, fov, near, far = 2.0, 26.9, 0.0109, 0.868
    pose = _pose(-0.4, (0.2, 0.1, -0.03))
    got = SO.grid_coverage_lidar(C, H, BOUND, pose[None], fov_up, fov, fov_hoz, near, far)
    p, m = _f64_points(pose)
    r, rho = np.linalg.norm(p, axis=1), np.linalg.norm(p[:, :2], axis=1)
    s_up, s_lo = math.tan(math.radians(fov_up)), math.tan(math.radians(fov_up - fov))
    terms = [r - (near - m), far + m - r, p[:, 2] - (s_lo * rho - m), s_up * rho + m - p[:, 2]]
    want = np.all([t > 0 for t in terms], axis=0)
    if fov_hoz < 360:
        h = math.radians(fov_hoz / 2)
        d1 = p[:, 0] * math.sin(h) + p[:, 1] * math.cos(h) + m
        d2 = p[:, 0] * math.sin(h) - p[:, 1] * math.cos(h) + m
        want &= ((d1 > 0) & (d2 > 0)) if fov_hoz <= 180 else ((d1 > 0) | (d2 > 0))
        terms += [d1, d2]
        # the wedge as an azimuth interval, for points clear of both edges
        phi = np.degrees(np.arctan2(p[:, 1], p[:, 0]))
        inside = np.abs(phi) < fov_hoz / 2
        far_from_edges = (np.abs(d1 - m) > 2 * m) & (np.abs(d2 - m) > 2 * m) & (rho > 4 * m)
        base = np.all([t > 0 for t in terms[:4]], axis=0)
        np.testing.assert_array_equal(got[far_from_edges & base], inside[far_from_edges & base])
    clear = np.all([np.abs(t) > 1e-4 for t in terms], axis=0)
    assert clear.mean() > 0.99 and 0.001 < want.mean() < 0.95
    np.testing.assert_array_equal(got[clear], want[clear])


def test_centred_camera_equals_torch_ngp_formula():
    """cx = W/2, cy = H/2: the frustum test is torch-ngp's |x| < cx/fx * z + 2h, |y| < cy/fy * z + 2h, z > 0, bit
    for bit in fp32 (the slopes are then exact negatives, and fl(-a - m) = -fl(a + m))."""
    Wi, Hi, fx, fy = 140, 38, 50.3, 50.3
    cx, cy = f32(Wi / 2), f32(Hi / 2)
    poses = np.stack([_pose(0.3, (0.0, 0.1, 0.0), cam=True), _pose(2.0, (-0.3, 0.2, 0.1), cam=True)])
    got = SO.grid_coverage_camera(C, H, BOUND, poses, fx, fy, cx, cy, Hi, Wi)
    want = np.zeros_like(got)
    for P in poses:
        p, m = SO._sensor_points(C, H, BOUND, P)
        ax, ay = f32(cx) / f32(fx), f32(cy) / f32(fy)
        want |= (p[:, 2] > 0) & (np.abs(p[:, 0]) < ax * p[:, 2] + m) & (np.abs(p[:, 1]) < ay * p[:, 2] + m)
    np.testing.assert_array_equal(got, want)


def test_coverage_accumulates_as_a_union():
    poses = np.stack([_pose(0.3 * k, (0.05 * k, 0.0, 0.0)) for k in range(3)])
    args = (2.0, 26.9, 120.0, 0.01, 0.8)
    one = SO.grid_coverage_lidar(C, H, BOUND, poses, *args)
    acc = SO.grid_coverage_lidar(C, H, BOUND, poses[:1], *args)
    acc = SO.grid_coverage_lidar(C, H, BOUND, poses[1:], *args, covered=acc)
    np.testing.assert_array_equal(one, acc)


def test_apply_marks():
    rng = np.random.default_rng(0)
    n = C * H ** 3
    grid = rng.random(n, dtype=np.float32)
    grid[:10] = -1
    cov = rng.random(n) < 0.6
    cov[:5] = True
    bf = np.packbits(grid > 0.3, bitorder="little")
    g, b, k = SO.apply_marks(grid, bf, cov)
    assert k == int((~cov).sum())
    assert (g[~cov] == -1).all() and (g[:5] == 0).all() and np.array_equal(g[10:][cov[10:]], grid[10:][cov[10:]])
    assert (g[5:10][cov[5:10]] == 0).all()   # a covered mark becomes 0
    np.testing.assert_array_equal(b, np.packbits((grid > 0.3) & cov, bitorder="little"))


def test_splitmix64_reference_values():
    # the first outputs of splitmix64 seeded with 0 (Vigna's reference generator: state += golden, then mix)
    z = SO.splitmix64(np.array([0, 0x9E3779B97F4A7C15], np.uint64))
    assert [int(v) for v in z] == [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4]


def test_partial_draw_statistics():
    rng = np.random.default_rng(1)
    n, H3 = C * H ** 3, H ** 3
    grid = np.zeros(n, np.float32)
    occ = rng.random(n) < 0.03
    grid[occ] = rng.random(occ.sum(), dtype=np.float32) + 0.01
    grid[rng.random(n) < 0.1] = -1
    d = SO.grid_draws(C, H, 5, 17, grid).reshape(C, -1)
    Q = H3 // 4
    assert d.shape == (C, 2 * Q)
    for c in range(C):
        assert (d[c] >= c * H3).all() and (d[c] < (c + 1) * H3).all()
        assert (grid[d[c, Q:]] > 0).all()
        # uniform draws: about (1 - e^{-1/4}) of the cascade's cells are hit, and every cell can be
        assert abs(np.unique(d[c, :Q]).size / H3 - (1 - math.exp(-0.25))) < 0.02
        occ_c = np.nonzero(grid[c * H3:(c + 1) * H3] > 0)[0] + c * H3
        hits = np.bincount(np.searchsorted(occ_c, d[c, Q:]), minlength=occ_c.size)
        assert hits.min() > 0 and hits.max() < 4 * Q / occ_c.size   # Q draws spread over every occupied cell
    np.testing.assert_array_equal(d.reshape(-1), SO.grid_draws(C, H, 5, 17, grid))      # the same key repeats
    assert (SO.grid_draws(C, H, 5, 18, grid) != d.reshape(-1)).mean() > 0.9                # another iteration
    assert (SO.grid_draws(C, H, 6, 17, grid) != d.reshape(-1)).mean() > 0.9                # another seed
    empty = SO.grid_draws(C, H, 5, 17, np.zeros(n, np.float32)).reshape(C, -1)
    assert (empty[:, Q:] == -1).all() and (empty[:, :Q] >= 0).all()


def test_partial_update_touches_only_drawn_cells():
    rng = np.random.default_rng(2)
    n = C * H ** 3
    grid = rng.random(n, dtype=np.float32)
    grid[:50] = -1
    cells = np.array([3, 3, 7, 20, -1, 60], np.int32)
    vals = np.array([0.5, 2.0, 0.0, 5.0, 9.0, 3.0], np.float32)
    g, mean, thresh, bits = SO.partial_update(grid, cells, vals, 0.9, 0.01)
    want = grid.copy()
    want[60] = max(grid[60] * f32(0.9), f32(3.0))   # cells 3, 7, 20 are marked (-1): untouched
    np.testing.assert_array_equal(g, want)
    tmp = SO.scatter_max(n, cells, vals)
    assert tmp[3] == 2.0 and tmp[20] == 5.0 and tmp[60] == 3.0 and (tmp[np.setdiff1d(np.arange(n), cells)] == -1).all()


# ------------------------------------------------------------------------------------------------------ C ABI
def _lib():
    pkg = importlib.import_module("selfsupervised-nvsf_b200")
    importlib.import_module("selfsupervised-nvsf_b200.build").build()
    return pkg._lib.lib()


def test_cabi_argument_checks():
    L = _lib()
    fake = ctypes.c_void_p(1 << 20)   # never dereferenced: every check below returns before a launch
    lid = lambda *a: L.nvsf_grid_coverage_lidar(2, 128, 2.0, fake, 4, *a, fake, None)
    assert lid(90.0, 10.0, 360.0, 0.01, 0.8) == -1      # fov_up >= 90
    assert lid(2.0, 92.0, 360.0, 0.01, 0.8) == -1       # fov_up - fov <= -90
    assert lid(2.0, 0.0, 360.0, 0.01, 0.8) == -1        # fov <= 0
    assert lid(2.0, 26.9, 0.0, 0.01, 0.8) == -1         # fov_hoz outside (0, 360]
    assert lid(2.0, 26.9, 360.5, 0.01, 0.8) == -1
    assert lid(2.0, 26.9, 360.0, 0.9, 0.8) == -1        # far <= near
    assert lid(2.0, 26.9, 360.0, -0.1, 0.8) == -1
    assert L.nvsf_grid_coverage_lidar(2, 128, 2.0, None, 4, 2.0, 26.9, 360.0, 0.01, 0.8, fake, None) == -1
    assert L.nvsf_grid_coverage_lidar(2, 128, 2.0, fake, 4, 2.0, 26.9, 360.0, 0.01, 0.8, ctypes.c_void_p((1 << 20) + 2),
                                      None) == -1     # covered not 4-byte aligned
    assert L.nvsf_grid_coverage_lidar(1, 2, 2.0, fake, 4, 2.0, 26.9, 360.0, 0.01, 0.8, fake, None) == -1  # 8 cells
    assert L.nvsf_grid_coverage_lidar(2, 128, 2.0, fake, 0, 90.0, 0.0, 0.0, 0.0, 0.0, fake, None) == 0  # B == 0
    cam = lambda fx, fy, cx, h, w: L.nvsf_grid_coverage_camera(2, 128, 2.0, fake, 4, fx, fy, cx, 20.0, h, w, fake, None)
    assert cam(0.0, 50.0, 10.0, 30, 40) == -1 and cam(50.0, -1.0, 10.0, 30, 40) == -1
    assert cam(50.0, 50.0, float("nan"), 30, 40) == -1 and cam(50.0, 50.0, 10.0, 0, 40) == -1
    assert L.nvsf_grid_apply_marks(fake, fake, fake, 12, fake, None) == -1          # n not a multiple of 8
    assert L.nvsf_grid_apply_marks(fake, None, fake, 16, fake, None) == -1
    wb = L.nvsf_grid_cell_list_workspace_bytes(2 * 128 ** 3)
    assert wb >= 2 * 128 ** 3 // 1024 * 4
    assert L.nvsf_grid_cell_list(fake, 2, 128 ** 3, 0, fake, fake, fake, wb - 4, None) == -2
    assert L.nvsf_grid_cell_list(fake, 2, 128 ** 3, 2, fake, fake, fake, wb, None) == -1
    assert L.nvsf_grid_draws(2, 6, 0, 0, fake, fake, fake, None) == -1               # H3 not a multiple of 4
    assert L.nvsf_grid_draws(2, 128 ** 3, 0, 0, None, fake, fake, None) == -1
    assert L.nvsf_grid_scatter_max(None, 8, fake, fake, 4, None) == -1
    assert L.nvsf_grid_scatter_max(None, 8, None, None, 0, None) == 0
    assert L.nvsf_grid_cell_points_list(2, 1, 2.0, fake, 4, None, 0, fake, None) == -1
    assert L.nvsf_grid_cell_points_list(2, 128, 2.0, None, 4, None, 0, fake, None) == -1
