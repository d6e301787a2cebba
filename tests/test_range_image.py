"""Point cloud -> range image (metrics.range_image, csrc/eval.cu k_range_scatter / k_range_resolve, C ABI Part 6)
against the numpy restatement (oracle/range_image_oracle.py).

CPU: the literal per-point loop equals the vectorised oracle on constructed clouds (exact-depth ties, order,
max_depth, non-finite points, the seam with y = +-0.0, rows just outside the field of view, empty scans, poses);
the round trip lidar_points -> range_image; the C ABI's argument checks.  GPU: images and index bit-exact against
the oracle; ragged batches with poses equal single calls; repeatability and input-order independence; round trips
with the renderer, get_lidar_rays and LidarMeter; one pixel under 1 M points; malformed input."""
import importlib
import math
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import metrics_oracle as MO
from oracle import range_image_oracle as RO

gpu = pytest.mark.gpu
K, K_HOZ = (2.0, 26.9), (180.0, 360.0)   # tests/golden/rays_ref.npz lidar_K / lidar_K_hoz
H_FULL, W_FULL = 66, 1030
f32 = np.float32


def _pkg():
    return importlib.import_module("selfsupervised-nvsf_b200")


def _rigid(rng):
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    p = np.eye(4, dtype=f32)
    p[:3, :3] = q
    p[:3, 3] = rng.normal(0, 5, 3)
    return p


def _random_cloud(rng, n, fov_up=2.0, fov=26.9, near=1.0, far=90.0, channels=4):
    """n points spread over the frustum of the frame (and a little outside it), depths in [near, far)."""
    b = np.radians(rng.uniform(-180, 180, n))
    a = np.radians(rng.uniform(fov_up - fov - 1, fov_up + 1, n))
    d = rng.uniform(near, far, n)
    pts = np.stack([d * np.cos(a) * np.cos(b), d * np.cos(a) * np.sin(b), d * np.sin(a), rng.random(n)], 1)
    return pts[:, :channels].astype(f32)


def _constructed(channels=4, H=8, W=16, fov_up=10.0, fov=20.0, max_depth=80.0):
    """Hand-built points of the frame (H, W, (fov_up, fov), 360 deg).  Directions use exact angles (0, +-90, 180
    deg) or rows at least 0.1 px from a rounding boundary.  Returns (points, what each one tests)."""
    below = float(np.nextafter(f32(max_depth), f32(0)))
    nan, inf = float("nan"), float("inf")

    def at_row(r_real, d=5.0, beta_deg=45.0):   # a point whose exact row coordinate is r_real
        a = math.radians(fov_up - r_real * fov / H)
        b = math.radians(beta_deg)
        return [d * math.cos(a) * math.cos(b), d * math.cos(a) * math.sin(b), d * math.sin(a)]

    rows = [
        ([5.0, 0.0, 0.0], "farther first"), ([2.0, 0.0, 0.0], "nearer later wins"),
        ([3.0, 3.0, 0.0], "tie: lowest index"), ([3.0, 3.0, 0.0], "tie: loses"), ([3.0, 3.0, 0.0], "tie: loses"),
        ([0.0, max_depth, 0.0], "depth == max_depth: dropped"), ([0.0, -below, 0.0], "next float below: kept"),
        ([0.0, 0.0, 0.0], "zero: dropped"), ([nan, 1.0, 0.0], "nan: dropped"), ([1.0, nan, nan], "nan"),
        ([inf, 0.0, 0.0], "inf: dropped"), ([-inf, 1.0, 2.0], "-inf"), ([1.0, 1.0, inf], "inf z"),
        ([-3.0, 0.0, 0.0], "seam y = +0: c = 0"), ([-4.0, -0.0, 0.0], "seam y = -0: c = W, dropped"),
        (at_row(-0.6), "row -1: dropped"), (at_row(-0.4), "row 0"), (at_row(H - 0.6), "row H-1"),
        (at_row(H - 0.4), "row H: dropped"), (at_row(3.0, 7.0, -90.0), "beta = -90"),
    ]
    pts = np.array([p for p, _ in rows], np.float64).astype(f32)
    if channels == 4:
        pts = np.concatenate([pts, (np.arange(len(pts), dtype=f32)[:, None] + 1) / 64], 1)
    return pts, [w for _, w in rows]


CASE_FRAME = dict(H=8, W=16, intrinsics=(10.0, 20.0), intrinsics_hoz=(180.0, 360.0))


# ---------------------------------------------------------------------------------------------- CPU
def _loop_eq_vec(pts, H, W, intrinsics, intrinsics_hoz, **kw):
    a_img, a_idx = RO.range_image_loop(pts, H, W, intrinsics, intrinsics_hoz, **kw)
    b_img, b_idx = RO.range_image(pts, H, W, intrinsics, intrinsics_hoz, **kw)
    assert np.array_equal(a_img.view(np.uint32), b_img.view(np.uint32))
    assert np.array_equal(a_idx, b_idx)
    return a_img, a_idx


@pytest.mark.parametrize("channels", [3, 4])
def test_oracle_loop_equals_vectorised_on_constructed_cases(channels):
    pts, _ = _constructed(channels)
    img, idx = _loop_eq_vec(pts, **CASE_FRAME, scale=0.5)
    H, W = CASE_FRAME["H"], CASE_FRAME["W"]
    r0, c0 = H // 2, W // 2            # beta = 0, alpha = 0: column W/2, row H/2
    assert idx[r0, c0] == 1 and img[r0, c0, 2] == f32(1.0)             # the nearer, later point
    assert idx[r0, 6] == 2                                             # beta = 45: column 6, lowest of the ties
    assert idx[r0, 4] == -1                                            # depth == max_depth (beta = 90)
    assert idx[r0, 12] == 6                                            # the float below max_depth (beta = -90)
    assert idx[r0, 0] == 13                                            # y = +0.0 lands on column 0
    assert 14 not in idx and 15 not in idx and 18 not in idx           # y = -0.0 (c = W), rows -1 and H
    assert idx[0, 6] == 16 and idx[H - 1, 6] == 17
    assert not np.isin(np.arange(7, 13), idx).any()                    # zero, NaN, inf
    if channels == 4:
        assert img[r0, 6, 1] == pts[2, 3] and img[r0, c0, 1] == pts[1, 3]
    hit = idx >= 0
    assert (img[hit, 0] == 1).all() and not img[~hit].any()


def test_oracle_loop_equals_vectorised_on_scans_with_poses():
    rng = np.random.default_rng(3)
    case, _ = _constructed(4)
    counts = [40, 0, 300, 0, 25]
    offs = np.concatenate([[0], np.cumsum(counts)])
    pts = np.concatenate([_random_cloud(rng, offs[-1], 10.0, 20.0, 1.0, 30.0), case])
    offs = list(offs[:-1]) + [offs[-1] + len(case)]    # the constructed points go to the last scan
    poses = np.stack([_rigid(rng) for _ in counts])
    img, idx = _loop_eq_vec(pts, **CASE_FRAME, offsets=offs, poses=poses, scale=2.0, max_depth=25.0)
    assert img.shape == (5, 8, 16, 3) and idx.shape == (5, 8, 16)
    assert (idx[1] == -1).all() and (idx[3] == -1).all()
    for b in (0, 2, 4):
        assert (idx[b] >= 0).sum() > 0 and ((idx[b] < 0) | ((idx[b] >= offs[b]) & (idx[b] < offs[b + 1]))).all()
    # the pose only moves the points: sensor-frame points, taken to the world and projected at the pose, give the
    # image of the sensor-frame points without a pose
    g = slice(offs[2], offs[3])
    R, t = poses[2][:3, :3].astype(np.float64), poses[2][:3, 3].astype(np.float64)
    world = (pts[g, :3].astype(np.float64) @ R.T + t).astype(f32)
    _, idx_w = RO.range_image(np.concatenate([world, pts[g, 3:]], 1), **CASE_FRAME, poses=poses[2], max_depth=25.0)
    _, idx_s = RO.range_image(pts[g], **CASE_FRAME, max_depth=25.0)
    assert (idx_s >= 0).sum() > 20 and np.array_equal(idx_w, idx_s)


@pytest.mark.parametrize("fov_hoz", [360.0, 90.0])
def test_oracle_round_trip_from_lidar_points(fov_hoz):
    """lidar_points(D) -> range_image gives back mask and intensity exactly and the depth to rtol 5e-7.  The bound:
    D / scale is rounded once, the fp32 beam direction has |d| = 1 +- 1.5 ulp, each fp32 coordinate product and
    |p| are rounded once, and depth32 * scale once more: under 4 ulp, each at most 2^-23 relative (4.8e-7).
    At 360 deg column 0 lies on the seam: its fp32 angle 0.5 * 360 / 180 * pi_f32 overshoots pi, so its point
    has y < 0 and beta = -180 deg + 5e-6 deg, which rounds to c = W and is dropped."""
    H, W, scale = 16, 64, f32(0.37)
    rng = np.random.default_rng(int(fov_hoz))
    D = rng.uniform(1, 70, (H, W)).astype(f32)
    D[rng.random((H, W)) < 0.2] = 0
    it = rng.random((H, W)).astype(f32)
    pts = MO.lidar_points(D, K, (0.0, fov_hoz), scale=scale, intensity=it)
    img, _ = _loop_eq_vec(pts.astype(f32), H, W, K, (0.0, fov_hoz), scale=scale, max_depth=1e4)
    mask = D != 0
    if fov_hoz == 360.0:
        assert not img[:, 0].any()
        mask[:, 0] = False
    assert np.array_equal(img[..., 0] == 1, mask)
    assert np.array_equal(img[..., 1], np.where(mask, it, 0))
    np.testing.assert_allclose(img[..., 2], np.where(mask, D, 0), rtol=5e-7, atol=0)


def test_cabi_argument_checks():
    """Checks that return before anything touches the device (the pointers are never dereferenced)."""
    L = _pkg()._lib.lib()
    assert L.nvsf_range_image_workspace_bytes(3, H_FULL, W_FULL) == 3 * H_FULL * W_FULL * 8
    assert L.nvsf_range_image_workspace_bytes(1, 1 << 14, 1 << 13) == 0
    assert L.nvsf_range_image_workspace_bytes(1, 0, 5) == 0
    fake = 1 << 20
    wb = L.nvsf_range_image_workspace_bytes(2, 4, 5)
    args = [fake, 4, fake, 2, 10, None, 4, 5, 2.0, 26.9, 360.0, 1.0, 80.0, fake, None, fake, wb, None]
    for i, bad in ((1, 5), (1, 2), (2, None), (3, 65536), (4, 10), (6, 0), (6, 1 << 24), (13, None), (15, None),
                   (15, fake + 4)):
        a = list(args)
        a[i] = bad
        if i == 4:
            a[0] = None     # points may be NULL only when every scan is empty
        assert L.nvsf_range_image(*a) == -1, (i, bad)
    a = list(args)
    a[16] = wb - 1
    assert L.nvsf_range_image(*a) == -2
    a = list(args)
    a[3] = 0                # no scans: nothing to do
    assert L.nvsf_range_image(*a) == 0


# ---------------------------------------------------------------------------------------------- GPU
def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _dirty(*nbytes):
    """Leave NaN-patterned blocks of these sizes in the caching allocator, so that the next allocations of these
    sizes (outputs, workspace) start with garbage."""
    for n in nbytes:
        torch.full((n // 4,), float("nan"), device="cuda")


def _check_equal(img, idx, want_img, want_idx):
    assert torch.equal(img.cpu().view(torch.int32), torch.from_numpy(want_img).view(torch.int32))
    assert torch.equal(idx.cpu(), torch.from_numpy(want_idx))


def _dense_cloud(seed, channels, n=200_000, dups=2000):
    """~2 points per pixel at 66 x 1030 (some beyond 80 m or outside the frame), then `dups` exact copies of
    earlier points with other intensities (exact-depth ties), then the constructed cases."""
    rng = np.random.default_rng(seed)
    pts = _random_cloud(rng, n, channels=4)
    src = rng.integers(0, n, dups)
    cp = pts[src].copy()
    cp[:, 3] = rng.random(dups)
    pts = np.concatenate([pts, cp])
    case, _ = _constructed(4)
    pts = np.concatenate([pts, case * f32([4, 4, 1, 1])])   # (seam, zero, non-finite cases in this frame too)
    return pts[:, :channels].copy(), src


@gpu
@pytest.mark.parametrize("channels,scale", [(3, 1.0), (4, 1.0), (4, 0.37), (3, 2.5)])
def test_bit_exact_vs_oracle(channels, scale):
    pkg = _pkg()
    pts, _ = _dense_cloud(channels * 10 + int(scale * 10), channels)
    n_px = H_FULL * W_FULL
    _dirty(n_px * 12, n_px * 8, n_px * 8)
    img, idx = pkg.metrics.range_image(_dev(pts), H_FULL, W_FULL, K, K_HOZ, scale=scale, return_index=True)
    want_img, want_idx = RO.range_image(pts, H_FULL, W_FULL, K, K_HOZ, scale=scale)
    assert img.shape == (H_FULL, W_FULL, 3) and idx.shape == (H_FULL, W_FULL) and idx.dtype == torch.int64
    _check_equal(img, idx, want_img, want_idx)
    assert 0.5 < (want_idx >= 0).mean() < 1.0
    only = pkg.metrics.range_image(_dev(pts), H_FULL, W_FULL, K, K_HOZ, scale=scale)
    assert torch.equal(only.view(torch.int32), img.view(torch.int32))


@gpu
def test_ragged_batch_with_poses_equals_single_calls_and_oracle():
    pkg = _pkg()
    rng = np.random.default_rng(16)
    counts = rng.integers(1000, 20000, 16)
    counts[3], counts[7] = 0, 70_000
    offs = [0] + np.cumsum(counts).tolist()
    poses = np.stack([_rigid(rng) for _ in counts])
    clouds = []
    for b, c in enumerate(counts):
        p = _random_cloud(rng, int(c))
        R, t = poses[b][:3, :3], poses[b][:3, 3]
        clouds.append(np.concatenate([(p[:, :3] @ R.T + t).astype(f32), p[:, 3:]], 1))
    pts = np.concatenate(clouds)
    img, idx = pkg.metrics.range_image(_dev(pts), H_FULL, W_FULL, K, K_HOZ, scale=0.5, offsets=offs,
                                       poses=_dev(poses), return_index=True)
    want_img, want_idx = RO.range_image(pts, H_FULL, W_FULL, K, K_HOZ, scale=0.5, offsets=offs, poses=poses)
    assert img.shape == (16, H_FULL, W_FULL, 3)
    _check_equal(img, idx, want_img, want_idx)
    assert (want_idx[3] == -1).all() and (want_idx[7] >= 0).sum() > 0.45 * H_FULL * W_FULL
    for b in range(16):
        one, one_idx = pkg.metrics.range_image(_dev(clouds[b]), H_FULL, W_FULL, K, K_HOZ, scale=0.5,
                                               poses=_dev(poses[b]), return_index=True)
        assert torch.equal(one.view(torch.int32), img[b].view(torch.int32))
        assert torch.equal(torch.where(one_idx >= 0, one_idx + offs[b], one_idx), idx[b])
    # offsets as a CPU tensor
    again = pkg.metrics.range_image(_dev(pts), H_FULL, W_FULL, K, K_HOZ, scale=0.5, offsets=torch.tensor(offs),
                                    poses=_dev(poses))
    assert torch.equal(again.view(torch.int32), img.view(torch.int32))


@gpu
def test_repeatable_and_independent_of_input_order():
    pkg = _pkg()
    pts, src = _dense_cloud(7, 4)
    n = len(pts)
    x = _dev(pts)
    n_px = H_FULL * W_FULL
    _dirty(n_px * 12, n_px * 8, n_px * 8)
    a, ia = pkg.metrics.range_image(x, H_FULL, W_FULL, K, K_HOZ, return_index=True)
    _dirty(n_px * 12, n_px * 8, n_px * 8)
    b, ib = pkg.metrics.range_image(x, H_FULL, W_FULL, K, K_HOZ, return_index=True)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)) and torch.equal(ia, ib)
    perm = torch.from_numpy(np.random.default_rng(8).permutation(n)).cuda()
    c, ic = pkg.metrics.range_image(x[perm], H_FULL, W_FULL, K, K_HOZ, return_index=True)
    assert torch.equal(c[..., 0], a[..., 0]) and torch.equal(c[..., 2], a[..., 2])
    # the same point wins wherever its depth is the pixel's unique minimum: ties only come from the copies
    n_case = len(_constructed()[0])
    tied = np.zeros(n, bool)
    tied[src] = True
    tied[n - n_case - len(src):] = True     # the copies and the constructed cases
    ia_h, ic_h = ia.cpu().numpy(), ic.cpu().numpy()
    hit = ia_h >= 0
    unique = hit.copy()
    unique[hit] = ~tied[ia_h[hit]]
    assert unique.sum() > 0.9 * hit.sum()
    assert np.array_equal(perm.cpu().numpy()[ic_h[unique]], ia_h[unique])
    assert torch.equal(c[..., 1][torch.from_numpy(unique).cuda()], a[..., 1][torch.from_numpy(unique).cuda()])


def _model_and_frame():
    import field_cases as FC
    pkg = _pkg()
    S = FC.S
    model = pkg.NeRFNetwork(time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND,
                            min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    model.load_flat_params(FC.oracle_params())
    model.eval()
    g = np.load(os.path.join(GOLDEN, "rays_ref.npz"))
    pose = torch.from_numpy(g["pose_a"]).clone()
    pose[:3, 3] *= 0.2
    f = model.render_frame(pose, g["lidar_K"], H_FULL, W_FULL, 0.3, cal_lidar_color=True,
                           intrinsics_hoz=g["lidar_K_hoz"])
    f["image_lidar"][..., 0] += 0.3    # the untrained ray-drop head stays below 0.5 (see test_metrics.py)
    return pkg, S, g, pose.float().cuda(), f


@gpu
def test_round_trips_with_the_renderer_and_rays():
    pkg, S, g, pose, f = _model_and_frame()
    Kl, Kh = g["lidar_K"], g["lidar_K_hoz"]
    depth, raydrop, inten = f["depth_lidar"], f["image_lidar"][..., 0], f["image_lidar"][..., 1]
    pts, count = pkg.metrics.lidar_points(depth, Kl, Kh, S.SCALE, raydrop=raydrop, intensity=inten)
    pts = pts[:int(count)]
    img, idx = pkg.metrics.range_image(pts, H_FULL, W_FULL, Kl, Kh, scale=S.SCALE, max_depth=1e4,
                                       return_index=True)
    mask = (depth * (raydrop > 0.5).float()) != 0
    assert not img[:, 0].any()              # column 0 of a 360 deg frame is on the seam (see the CPU round trip)
    mask[:, 0] = False
    assert 0 < int(mask.sum()) < H_FULL * W_FULL - H_FULL
    assert torch.equal(img[..., 0] == 1, mask)
    assert torch.equal(img[..., 1], torch.where(mask, inten, 0.0))
    torch.testing.assert_close(img[..., 2], torch.where(mask, depth, 0.0), rtol=5e-7, atol=0)
    # the same points in world coordinates, projected at the pose: the same pixels, the same winners
    R, t = pose[:3, :3], pose[:3, 3]
    world = torch.cat([(R[None] * pts[:, None, :3]).sum(-1) + t, pts[:, 3:]], 1)
    img_w, idx_w = pkg.metrics.range_image(world, H_FULL, W_FULL, Kl, Kh, scale=S.SCALE, max_depth=1e4, poses=pose,
                                           return_index=True)
    assert torch.equal(idx_w[:, 1:], idx[:, 1:])
    torch.testing.assert_close(img_w[:, 1:], img[:, 1:], rtol=1e-5, atol=0)
    # get_lidar_rays: rays_o + rays_d * t lands on the ray's own pixel
    rays = pkg.rays.get_lidar_rays(pose[None], Kl, Kh, H_FULL, W_FULL, -1)
    tt = 1.0 + 59.0 * torch.rand(H_FULL * W_FULL, 1, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    p = rays["rays_o"][0] + rays["rays_d"][0] * tt
    _, idx_r = pkg.metrics.range_image(p, H_FULL, W_FULL, Kl, Kh, poses=pose, return_index=True)
    inds = rays["inds"][0].reshape(H_FULL, W_FULL)
    assert torch.equal(idx_r[:, 1:], inds[:, 1:])
    assert ((idx_r[:, 0] == inds[:, 0]) | (idx_r[:, 0] == -1)).all()


@gpu
def test_lidar_meter_reads_the_layout():
    pkg, S, g, pose, f = _model_and_frame()
    Kl, Kh = g["lidar_K"], g["lidar_K_hoz"]
    f["image_lidar"][:, 0, 0] = 0.0         # no return on the seam column, which range_image cannot give back
    depth, raydrop, inten = f["depth_lidar"], f["image_lidar"][..., 0], f["image_lidar"][..., 1]
    pts, count = pkg.metrics.lidar_points(depth, Kl, Kh, S.SCALE, raydrop=raydrop, intensity=inten)
    gt = pkg.metrics.range_image(pts[:int(count)], H_FULL, W_FULL, Kl, Kh, scale=S.SCALE, max_depth=1e4)
    meter = pkg.metrics.LidarMeter(H_FULL, W_FULL, Kl, Kh, S.SCALE)
    row = dict(zip(pkg.metrics.LIDAR_METRICS, meter.update(depth, f["image_lidar"], gt).tolist()))
    assert row["raydrop_acc"] == 1.0 and row["raydrop_f1"] == 1.0 and row["intensity_rmse"] == 0.0
    # the depths differ by the round trip's < 4 ulp (a few 1e-6 m at 80 m)
    assert row["depth_rmse"] < 1e-4 and row["chamfer"] < 1e-7 and row["fscore"] == 1.0
    assert row["points_pred"] == row["points_gt"] == int(count)


@gpu
def test_one_pixel_under_a_million_points():
    pkg = _pkg()
    n = 1 << 20
    rng = np.random.default_rng(6)
    d = rng.uniform(1.0, 50.0, n).astype(f32)
    ties = [500_000, 123_457, 1_048_575, 777, 65_536]
    d[ties] = f32(0.75)
    pts = np.zeros((n, 4), f32)
    pts[:, 0] = d
    pts[:, 3] = rng.random(n)
    img, idx = pkg.metrics.range_image(_dev(pts), H_FULL, W_FULL, K, K_HOZ, return_index=True)
    r, c = round(2.0 / 26.9 * H_FULL), W_FULL // 2
    assert int(idx[r, c]) == 777 and int((idx >= 0).sum()) == 1
    assert img[r, c].tolist() == [1.0, float(pts[777, 3]), 0.75]


@gpu
def test_malformed_input_raises():
    pkg = _pkg()
    M, E = pkg.metrics, pkg._lib.NvsfError
    x = torch.rand(100, 4, device="cuda")
    pose = torch.eye(4, device="cuda")
    bad = [
        dict(points=x.cpu()), dict(points=x[:, :2].contiguous()), dict(points=torch.rand(100, 5, device="cuda")),
        dict(points=x.double()), dict(points=x[None]),
        dict(offsets=[0, 50]), dict(offsets=[1, 100]), dict(offsets=[0, 60, 40, 100]), dict(offsets=[0]),
        dict(offsets=torch.tensor([0, 100], device="cuda")), dict(offsets=[0, "x", 100]),
        dict(poses=pose.cpu()), dict(poses=torch.eye(4, device="cuda")[None].repeat(2, 1, 1)),
        dict(poses=torch.eye(3, device="cuda")), dict(offsets=[0, 50, 100], poses=pose),
        dict(H=0), dict(W=-3), dict(H=1 << 14, W=1 << 13),
    ]
    for kw in bad:
        args = dict(points=x, H=H_FULL, W=W_FULL)
        args.update(kw)
        with pytest.raises(E):
            M.range_image(args.pop("points"), args.pop("H"), args.pop("W"), K, K_HOZ, **args)
    # through the C ABI: a short workspace
    L, P = pkg._lib.lib(), pkg._lib.ptr
    off = torch.tensor([0, 100], dtype=torch.int64, device="cuda")
    img = torch.empty(H_FULL, W_FULL, 3, device="cuda")
    wb = L.nvsf_range_image_workspace_bytes(1, H_FULL, W_FULL)
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
    args = [P(x), 4, P(off), 1, 100, None, H_FULL, W_FULL, 2.0, 26.9, 360.0, 1.0, 80.0, P(img), None, P(ws), wb, None]
    assert L.nvsf_range_image(*args) == 0
    args[16] = wb - 8
    assert L.nvsf_range_image(*args) == -2
    torch.cuda.synchronize()
