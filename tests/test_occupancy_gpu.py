"""GPU: untrained-cell marking (NeRFNetwork.mark_untrained_grid, csrc/scene.cu k_grid_coverage /
k_grid_apply_marks) bit for bit against tests/occupancy_oracle.py; the full update over the trainable-cell list
against the all-cells update; torch-ngp's partial update against the oracle fed the model's own sigmas; the
"ngp" schedule; the occupancy state round trip; and run_cuda on marked grids."""
import io

import numpy as np
import pytest

import field_cases as FC
from conftest import assert_bits_equal

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

S = FC.S
K = np.array([[S.CAM_FX, 0, S.CAM_CX], [0, S.CAM_FY, S.CAM_CY], [0, 0, 1]])
LIDAR_INTR = (S.LIDAR_FOV_UP, S.LIDAR_FOV)


def host(t):
    return t.detach().cpu().numpy()


def lidar_pose(seed):
    R, t = S.random_pose(seed)
    P = np.eye(4)
    P[:3, :3], P[:3, 3] = R, t
    return P.astype(np.float32)


def camera_pose(seed):
    R, t = S.random_pose(seed + 100)
    P = np.eye(4)
    P[:3, :3], P[:3, 3] = R @ np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]]), t
    return P.astype(np.float32)


def poses(fn, seeds):
    return np.stack([fn(s) for s in seeds])


@pytest.fixture(scope="module")
def model(pkg):
    m = pkg.NeRFNetwork(time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND,
                        min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    m.load_flat_params(FC.oracle_params())
    return m.eval()


@pytest.fixture(scope="module")
def SO():
    import occupancy_oracle
    return occupancy_oracle


def fresh_grid(model, lidar=True, updates=1):
    model._grid = {}
    for k in range(updates):
        model.update_extra_state(0.5, cal_lidar_color=lidar, perturb=False)
    return model


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------------------------ marking
CASES = {
    "camera": [dict(camera_poses=(0, 1, 2))],
    "lidar_360": [dict(lidar_poses=(0, 1, 2), hoz=360.0)],
    "lidar_narrow_wedge": [dict(lidar_poses=(3, 4), hoz=90.0)],
    "lidar_wide_wedge": [dict(lidar_poses=(5, 6), hoz=250.0)],
    "accumulated": [dict(lidar_poses=(7,), hoz=360.0), dict(camera_poses=(8, 9)), dict(lidar_poses=(10, 11),
                                                                                       hoz=180.0),
                    dict(camera_poses=(12,), lidar_poses=(13,), hoz=360.0)],
}


@pytest.mark.parametrize("case", list(CASES))
def test_marks_match_oracle(model, SO, case):
    C, H = model.cascade, model.grid_size
    n = C * H ** 3
    fresh_grid(model)
    grid = host(model.density_grid(True)).reshape(-1)
    bf = host(model.density_bitfield(True))
    assert bf.any()
    stats = host(model._grid[True]["stats"]).copy()
    cov = np.zeros(n, bool)
    for call in CASES[case]:
        kw, cam, lid = {}, call.get("camera_poses"), call.get("lidar_poses")
        if cam:
            P = poses(camera_pose, cam)
            kw.update(camera_poses=dev(P), intrinsics=K, H=S.CAM_H, W=S.CAM_W)
            cov = SO.grid_coverage_camera(C, H, S.BOUND, P, K[0, 0], K[1, 1], K[0, 2], K[1, 2], S.CAM_H, S.CAM_W,
                                          covered=cov)
        if lid:
            P = poses(lidar_pose, lid)
            kw.update(lidar_poses=dev(P), intrinsics_lidar=LIDAR_INTR, intrinsics_hoz_lidar=(0.0, call["hoz"]))
            cov = SO.grid_coverage_lidar(C, H, S.BOUND, P, *LIDAR_INTR, call["hoz"], S.MIN_NEAR_LIDAR,
                                         S.LIDAR_MAX_DEPTH, covered=cov)
        got = int(model.mark_untrained_grid(cal_lidar_color=True, **kw))
        grid, bf, k = SO.apply_marks(grid, bf, cov)   # a cell a later call covers is restored to 0
        eg, ebf = grid, bf
        assert got == k and 0 < k < n
        assert_bits_equal(host(model.density_grid(True)).reshape(-1), eg, f"{case}: density grid")
        np.testing.assert_array_equal(host(model.density_bitfield(True)), ebf)
    np.testing.assert_array_equal(host(model._grid[True]["stats"]), stats)   # stats wait for the next update
    st = model._grid[True]
    want_list = np.nonzero(eg >= 0)[0]
    np.testing.assert_array_equal(host(st["trainable"]), want_list)
    assert not host(model.density_grid(False)).any()   # the camera grid is separate state


def test_mark_argument_errors(model, pkg):
    fresh_grid(model)
    with pytest.raises(pkg._lib.NvsfError):
        model.mark_untrained_grid(cal_lidar_color=True)
    with pytest.raises(pkg._lib.NvsfError):
        model.mark_untrained_grid(lidar_poses=dev(poses(lidar_pose, (0,))), intrinsics_lidar=LIDAR_INTR,
                                  cal_lidar_color=True)
    with pytest.raises(pkg._lib.NvsfError):
        model.mark_untrained_grid(lidar_poses=dev(poses(lidar_pose, (0,))), intrinsics_lidar=(90.0, 10.0),
                                  intrinsics_hoz_lidar=(0, 360.0), cal_lidar_color=True)
    with pytest.raises(pkg._lib.NvsfError):
        model.mark_untrained_grid(camera_poses=dev(np.zeros((2, 3, 4), np.float32)), intrinsics=K, H=10, W=10)


# ------------------------------------------------------------------------------------------------ updates
def mark_lidar(model, seeds=(0, 1), lidar=True):
    return model.mark_untrained_grid(lidar_poses=dev(poses(lidar_pose, seeds)), intrinsics_lidar=LIDAR_INTR,
                                     intrinsics_hoz_lidar=(0.0, 360.0), cal_lidar_color=lidar)


def grid_tuple(model, lidar=True):
    st = model._grid[lidar]
    return st["density_grid"].clone(), st["density_bitfield"].clone(), st["stats"].clone()


def test_full_update_with_marks_equals_all_cells(model):
    C, H = model.cascade, model.grid_size
    n = C * H ** 3
    fresh_grid(model)
    mark_lidar(model)
    assert model._grid[True]["trainable"] is not None
    saved = model.occupancy_state_dict()
    noise = torch.rand(n, 3, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    model.update_extra_state([0.2, 0.7], cal_lidar_color=True, decay=0.8, noise=noise)
    a = grid_tuple(model)
    model.load_occupancy_state_dict(saved)
    model._grid[True]["trainable"] = None          # force the all-cells path on the same marked grid
    model.update_extra_state([0.2, 0.7], cal_lidar_color=True, decay=0.8, noise=noise)
    b = grid_tuple(model)
    for x, y, what in zip(a, b, ("grid", "bitfield", "stats")):
        assert torch.equal(x, y), what
    assert (a[0] < 0).any() and a[1].any()


def test_partial_update_matches_oracle(model, SO):
    from oracle import raymarching_oracle as RO
    C, H = model.cascade, model.grid_size
    fresh_grid(model, updates=2)
    mark_lidar(model)
    st = model._grid[True]
    st["iter_density"] = 21
    grid0 = host(st["density_grid"]).reshape(-1).copy()
    seed, times, decay = 1234, [0.1, 0.9], 0.9
    draws = SO.grid_draws(C, H, seed, 21, grid0)
    np.testing.assert_array_equal(host(model._partial_draws(st, seed)), draws)
    assert (draws[draws >= 0] < C * H ** 3).all() and (grid0[draws[draws >= 0]] >= -1).all()
    noise = torch.rand(draws.size, 3, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    model.update_extra_state(times, cal_lidar_color=True, decay=decay, noise=noise, mode="partial", seed=seed)
    assert st["iter_density"] == 22
    xyz = SO.cell_points_list(C, H, S.BOUND, draws, host(noise))
    with torch.no_grad():
        sig = [host(model._density_raw(dev(xyz), t, True)[0]) * np.float32(model.density_scale) for t in times]
    vals = np.maximum(sig[0], sig[1])
    eg, mean, _, _ = SO.partial_update(grid0, draws, vals, decay, model.density_thresh)
    g = host(st["density_grid"]).reshape(-1)
    assert_bits_equal(g, eg, "grid after the partial update")
    stats = host(st["stats"])
    assert abs(stats[0] - mean) <= 1e-6 * mean
    np.testing.assert_array_equal(host(st["density_bitfield"]), RO.packbits(eg, stats[1]))
    drawn = np.zeros(g.size, bool)
    drawn[draws[draws >= 0]] = True
    assert_bits_equal(g[~drawn], grid0[~drawn], "cells not drawn are neither decayed nor refreshed")
    live = drawn & (grid0 >= 0)
    assert live.sum() > 1000 and (g[live] != grid0[live]).mean() > 0.5


def test_ngp_schedule_switches_at_16(model):
    C, H = model.cascade, model.grid_size
    n = C * H ** 3
    fresh_grid(model)
    st = model._grid[True]
    g = torch.Generator("cuda").manual_seed(6)
    noise_full = torch.rand(n, 3, device="cuda", generator=g)
    noise_part = torch.rand(n // 2, 3, device="cuda", generator=g)
    for it, mode, noise in ((15, "full", noise_full), (16, "partial", noise_part)):
        st["iter_density"] = it
        saved = model.occupancy_state_dict()
        model.update_extra_state(0.4, cal_lidar_color=True, noise=noise, mode="ngp", seed=3)
        a = grid_tuple(model)
        model.load_occupancy_state_dict(saved)
        model.update_extra_state(0.4, cal_lidar_color=True, noise=noise, mode=mode, seed=3)
        b = grid_tuple(model)
        assert all(torch.equal(x, y) for x, y in zip(a, b)), (it, mode)
        assert st["iter_density"] == it + 1


# ------------------------------------------------------------------------------------------------ state and rendering
def test_occupancy_state_round_trip(model):
    fresh_grid(model, updates=2)
    mark_lidar(model)
    model.update_extra_state(0.3, cal_lidar_color=True, perturb=True)
    buf = io.BytesIO()
    torch.save(model.occupancy_state_dict(), buf)
    keys = set(model.state_dict().keys())
    o, d = S.lidar_rays(2048, seed=7)
    kw = dict(cal_lidar_color=True, dt_gamma=S.DT_GAMMA, T_thresh=1e-2)
    a = model.run_cuda(dev(o)[None], dev(d)[None], 0.3, **kw)
    want = {k: v.clone() for k, v in model._grid[True].items() if torch.is_tensor(v)}
    model._grid = {}
    buf.seek(0)
    model.load_occupancy_state_dict(torch.load(buf, map_location="cpu"))
    for k, v in want.items():
        assert torch.equal(model._grid[True][k], v), k
    assert model._grid[True]["iter_density"] == 3 and set(model.state_dict().keys()) == keys
    b = model.run_cuda(dev(o)[None], dev(d)[None], 0.3, **kw)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_load_rejects_a_grid_of_another_size(model, pkg):
    fresh_grid(model)
    sd = model.occupancy_state_dict()
    sd["lidar"]["density_grid"] = sd["lidar"]["density_grid"][:, :-8]
    with pytest.raises(pkg._lib.NvsfError):
        model.load_occupancy_state_dict(sd)


def test_run_cuda_on_marked_grid_equals_oracle_marked_bitfield(model, SO):
    C, H = model.cascade, model.grid_size
    fresh_grid(model, lidar=False)
    bf = host(model.density_bitfield(False))
    P = poses(camera_pose, (20, 21))
    model.mark_untrained_grid(camera_poses=dev(P), intrinsics=K, H=S.CAM_H, W=S.CAM_W, cal_lidar_color=False)
    cov = SO.grid_coverage_camera(C, H, S.BOUND, P, K[0, 0], K[1, 1], K[0, 2], K[1, 2], S.CAM_H, S.CAM_W)
    _, ebf, _ = SO.apply_marks(np.zeros(C * H ** 3, np.float32), bf, cov)
    o, d = S.camera_rays(4096, seed=22)
    kw = dict(cal_lidar_color=False, dt_gamma=S.DT_GAMMA, T_thresh=1e-2)
    a = model.run_cuda(dev(o)[None], dev(d)[None], 0.5, **kw)
    na = model.last_run_cuda_samples
    b = model.run_cuda(dev(o)[None], dev(d)[None], 0.5, density_bitfield=dev(ebf), **kw)
    assert na == model.last_run_cuda_samples
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_central_rays_of_a_training_camera_are_unchanged_by_marks(model, pkg):
    """Every cell a sample of these rays falls in is covered: a sample x at depth z >= 0.1 on a ray through the
    middle half of the image lies at least (slope range / 4) * z >= 0.064 inside the frustum, while its cell
    centre is at most sqrt(3) half-cells (0.027 in the coarser cascade, whose points are >= 0.7 from the camera)
    away from x, and the test widens the frustum by two half-cells."""
    fresh_grid(model, lidar=False, updates=2)
    P = camera_pose(30)
    tP = dev(P)[None]
    r = pkg.rays.get_rays(tP, K, S.CAM_H, S.CAM_W, -1)
    rows, cols = np.meshgrid(np.arange(S.CAM_H // 4, 3 * S.CAM_H // 4, 3), np.arange(S.CAM_W // 4, 3 * S.CAM_W // 4, 3),
                             indexing="ij")
    idx = torch.from_numpy((rows * S.CAM_W + cols).reshape(-1)).cuda()
    d = r["rays_d"][0, idx]
    o = r["rays_o"][0, idx] + 0.1 * d
    kw = dict(cal_lidar_color=False, dt_gamma=S.DT_GAMMA, T_thresh=1e-4)
    before_bits = model.density_bitfield(False).clone()
    a = model.run_cuda(o[None], d[None], 0.5, **kw)
    na = model.last_run_cuda_samples
    marked = int(model.mark_untrained_grid(camera_poses=tP, intrinsics=K, H=S.CAM_H, W=S.CAM_W))
    assert marked > 0 and not torch.equal(before_bits, model.density_bitfield(False))
    b = model.run_cuda(o[None], d[None], 0.5, **kw)
    assert na == model.last_run_cuda_samples and na > 0
    for k in a:
        assert torch.equal(a[k], b[k]), k
