"""GPU parity of the callers either side of the marcher (SURVEY.md §8f): ray generation,
NeRFNetwork.color as a standalone operator, occupancy-grid update, alive-list compaction and the
march_rays* render loops (run_cuda), each against its CPU oracle and — where the reference has
the function — against golden outputs of the reference itself.

Tolerances: ray directions 2e-6 absolute (fp32 sin/cos/normalise); anything through the fp16
MLPs 1e-2 relative (BASELINE.json north_star); integer/bit results exact."""
import ctypes
import os

import numpy as np
import pytest

import field_cases as FC
from conftest import GOLDEN, assert_bits_equal

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

S = FC.S


def host(t):
    return t.detach().float().cpu().numpy()


def close(a, b, rtol, atol, what):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    err = np.abs(a - b) - (atol + rtol * np.abs(b))
    assert (err <= 0).all(), f"{what}: worst excess {err.max():.3e}, max abs err {np.abs(a - b).max():.3e}"


@pytest.fixture(scope="module")
def model(pkg):
    m = pkg.NeRFNetwork(time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND,
                        min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    m.load_flat_params(FC.oracle_params())
    return m.eval()


@pytest.fixture(scope="module")
def orc():
    from oracle.field_oracle import FieldOracle
    return FieldOracle(FC.oracle_config(), FC.oracle_params())


@pytest.fixture(scope="module")
def SO():
    from oracle import scene_oracle
    return scene_oracle


# ------------------------------------------------------------------------------ ray generation
@pytest.fixture(scope="module")
def gold_rays():
    return np.load(os.path.join(GOLDEN, "rays_ref.npz"))


def test_get_lidar_rays_vs_reference(pkg, gold_rays, SO):
    g = gold_rays
    P = torch.from_numpy(g["pose_a"])[None].cuda()
    r = pkg.rays.get_lidar_rays(P, g["lidar_K"], g["lidar_K_hoz"], 66, 1030, -1)
    assert r["rays_o"].shape == (1, 67980, 3) and r["inds"].shape == (1, 67980)
    np.testing.assert_allclose(host(r["rays_d"])[0][g["lidar_full_a_inds"]], g["lidar_full_a_d"], rtol=0, atol=2e-6)
    assert (host(r["rays_o"])[0] == g["pose_a"][:3, 3]).all()
    _, od = SO.get_lidar_rays(g["pose_a"], g["lidar_K"], g["lidar_K_hoz"], 66, 1030)
    np.testing.assert_allclose(host(r["rays_d"])[0], od, rtol=0, atol=1e-6)
    # explicit pixel ids through the C ABI (the batch the reference drew with torch.randint)
    L = pkg._lib.lib()
    for tag in ("a", "b"):
        inds = torch.from_numpy(g[f"lidar_batch_{tag}_inds"]).cuda()
        pose = torch.from_numpy(g[f"pose_{tag}"]).cuda()
        o = torch.empty(4096, 3, device="cuda"); d = torch.empty(4096, 3, device="cuda")
        assert L.nvsf_get_lidar_rays(pose.data_ptr(), inds.data_ptr(), 4096, 66, 1030, 2.0, 26.9, 360.0,
                                     o.data_ptr(), d.data_ptr(), None) == 0
        np.testing.assert_allclose(host(d), g[f"lidar_batch_{tag}_d"], rtol=0, atol=2e-6)
    np.testing.assert_array_equal(host(o), np.broadcast_to(g["pose_b"][:3, 3], (4096, 3)))


def test_get_rays_vs_reference(pkg, gold_rays):
    g = gold_rays
    L = pkg._lib.lib()
    for tag in ("a", "b"):
        for kind in ("batch", "patch"):
            inds = torch.from_numpy(g[f"cam_{kind}_{tag}_inds"]).cuda()
            pose = torch.from_numpy(g[f"pose_{tag}"]).cuda()
            o = torch.empty(4096, 3, device="cuda"); d = torch.empty(4096, 3, device="cuda")
            K = g["cam_K"]
            assert L.nvsf_get_rays(pose.data_ptr(), inds.data_ptr(), 4096, 376, 1408, float(K[0, 0]), float(K[1, 1]),
                                   float(K[0, 2]), float(K[1, 2]), o.data_ptr(), d.data_ptr(), None) == 0
            np.testing.assert_allclose(host(d), g[f"cam_{kind}_{tag}_d"], rtol=0, atol=2e-6)
    r = pkg.rays.get_rays(torch.from_numpy(g["pose_a"])[None], g["cam_K"], 47, 176, -1)
    np.testing.assert_allclose(host(r["rays_d"])[0], g["cam_small_full_d"], rtol=0, atol=2e-6)
    nrm = np.linalg.norm(host(r["rays_d"])[0], axis=-1)
    np.testing.assert_allclose(nrm, 1.0, atol=1e-6)


def test_get_rays_sampling_matches_reference_rng(pkg):
    """N > 0 draws pixel ids with the reference's torch.randint call; patches are contiguous."""
    P = torch.eye(4)[None].cuda()
    torch.manual_seed(3)
    r = pkg.rays.get_rays(P, np.eye(3, dtype=np.float32) * 500, 376, 1408, 1024)
    torch.manual_seed(3)
    want = torch.randint(0, 376 * 1408, size=[1024], device="cuda")
    assert torch.equal(r["inds"][0], want) and r["rays_d"].shape == (1, 1024, 3)
    r = pkg.rays.get_lidar_rays(P, [2.0, 26.9], [180.0, 360.0], 66, 1030, 1024, patch_size=[2, 8])
    inds = host(r["inds"])[0].astype(np.int64).reshape(-1, 2, 8)
    assert (np.diff(inds, axis=2) == 1).all() and (inds[:, 1] - inds[:, 0] == 1030).all()
    with pytest.raises(NotImplementedError):
        pkg.rays.get_rays(P, np.eye(3), 8, 8, 4, use_error_map=True)


def test_render_frame_from_pose_equals_render_of_generated_rays(pkg, model, gold_rays, orc):
    """render_frame (pose in, image out; rays generated on the device in the renderer's stream) == render() of
    the rays the reference's generator produces for that pose (golden), and == the CPU oracle on a few rays."""
    g = gold_rays
    H, W, Sn, t = 6, 40, 64, 0.3
    for lidar in (True, False):
        pose = torch.from_numpy(g["pose_a"])
        if lidar:
            out = model.render_frame(pose, g["lidar_K"], H, W, t, cal_lidar_color=True,
                                     intrinsics_hoz=g["lidar_K_hoz"], num_steps=Sn)
            r = pkg.rays.get_lidar_rays(pose[None].cuda(), g["lidar_K"], g["lidar_K_hoz"], H, W, -1)
            keys = ("depth_lidar", "image_lidar")
        else:
            out = model.render_frame(pose, g["cam_K"], H, W, t, num_steps=Sn)
            r = pkg.rays.get_rays(pose[None].cuda(), g["cam_K"], H, W, -1)
            keys = ("depth", "image")
        ref = model.render(r["rays_o"], r["rays_d"], t, cal_lidar_color=lidar, staged=True, num_steps=Sn)
        assert out[keys[0]].shape == (H, W) and out[keys[1]].shape == (H, W, 2 if lidar else 3)
        assert torch.equal(out[keys[0]].reshape(-1), ref[keys[0]].reshape(-1))
        assert torch.equal(out[keys[1]].reshape(H * W, -1), ref[keys[1]].reshape(H * W, -1))
        if lidar:
            with torch.no_grad():
                e = orc.run(r["rays_o"][0, :32].cpu(), r["rays_d"][0, :32].cpu(), t, True, num_steps=Sn)
            close(host(out[keys[0]]).reshape(-1)[:32], e["depth"].numpy(), 1e-2, 1e-4, "render_frame depth vs oracle")


# ------------------------------------------------------------------------------ color operator
@pytest.mark.parametrize("lidar", [True, False])
def test_color_vs_oracle(model, orc, lidar):
    n = 1000  # not a multiple of 32: ragged last tile
    rng = np.random.default_rng(5)
    x = ((rng.random((n, 3), dtype=np.float32) * 2 - 1) * np.float32(1.9)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    mask = rng.random(n) < 0.4
    mask[64:160] = False  # whole tiles masked out
    t = 0.3
    den = model.density(torch.from_numpy(x).cuda(), t, lidar)
    with torch.no_grad():
        e_all = orc.color(torch.from_numpy(d), den["geo_feat"].float().cpu(), lidar).numpy()
    # (1) the view density() returned, no mask
    got = model.color(torch.from_numpy(x).cuda(), torch.from_numpy(d).cuda(), den["geo_feat"], None, lidar)
    assert got.shape == (n, 2 if lidar else 3) and got.dtype == torch.float32
    close(host(got), e_all, 1e-2, 1e-3, "color (geo16 view)")
    # (2) a contiguous fp32 [n,15] geo_feat + mask
    geo32 = den["geo_feat"].float().contiguous()
    got_m = model.color(None, torch.from_numpy(d).cuda(), geo32, torch.from_numpy(mask).cuda(), lidar)
    want = np.where(mask[:, None], e_all, 0.0)
    close(host(got_m), want, 1e-2, 1e-3, "color (masked)")
    assert not host(got_m)[~mask].any()
    np.testing.assert_allclose(host(got_m)[mask], host(got)[mask], rtol=1e-6, atol=1e-7)
    # (3) mask all false / empty input
    z = model.color(None, torch.from_numpy(d).cuda(), geo32, torch.zeros(n, dtype=torch.bool), lidar)
    assert not host(z).any()
    assert model.color(None, torch.zeros(0, 3), torch.zeros(0, 15), None, lidar).shape == (0, 2 if lidar else 3)


def test_color_matches_uniform_renderer(model):
    """The standalone heads and the heads fused into the uniform renderer agree: composite the
    standalone colours with the renderer's own weights."""
    o, d = S.lidar_rays(64, seed=2)
    to, td = torch.from_numpy(o).cuda()[None], torch.from_numpy(d).cuda()[None]
    Sn = 96
    r = model.render(to, td, 0.5, cal_lidar_color=True, num_steps=Sn)
    w, z = r["weights"], r["z_vals"]
    xyz = (to[0][:, None, :] + td[0][:, None, :] * z[..., None]).clamp(-S.BOUND, S.BOUND).reshape(-1, 3)
    den = model.density(xyz, 0.5, True)
    dirs = td[0][:, None, :].expand(-1, Sn, -1).reshape(-1, 3)
    rgb = model.color(xyz, dirs, den["geo_feat"], (w > 1e-4).reshape(-1), True).view(64, Sn, 2)
    img = (w[..., None] * rgb).sum(1)
    close(host(img), host(r["image_lidar"])[0], 1e-2, 1e-3, "image from standalone heads")


def test_color_cabi_errors(pkg, model):
    L = pkg._lib.lib()
    model.prepare(0.0, True)
    ws = model._ws[True]
    d = torch.zeros(8, 3, device="cuda"); g = torch.zeros(8, 16, dtype=torch.float16, device="cuda")
    out = torch.zeros(8, 4, device="cuda")
    cfg = ctypes.byref(model._cfg)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    assert L.nvsf_field_color(cfg, P(ws), 1, P(d), P(g), 16, 1, None, 8, P(out), 1, None) == -1   # out_ld < 2
    assert L.nvsf_field_color(cfg, P(ws), 1, P(d), P(g), 12, 1, None, 8, P(out), 2, None) == -1   # geo too narrow
    assert L.nvsf_field_color(cfg, P(ws), 1, None, P(g), 16, 1, None, 8, P(out), 2, None) == -1
    assert L.nvsf_field_color(cfg, P(ws), 1, None, None, 16, 1, None, 0, None, 2, None) == 0     # n == 0


# ------------------------------------------------------------------------------ occupancy grid
def test_grid_cell_points_bit_exact(pkg, SO):
    L = pkg._lib.lib()
    for C, H, bound, with_noise in ((2, 128, 2.0, True), (1, 64, 1.0, False), (3, 32, 3.0, True)):
        n = C * H ** 3
        noise = np.random.default_rng(C).random((n, 3), dtype=np.float32) if with_noise else None
        xyz = torch.empty(n, 3, device="cuda")
        nz = torch.from_numpy(noise).cuda() if with_noise else None
        assert L.nvsf_grid_cell_points(C, H, bound, nz.data_ptr() if with_noise else None, xyz.data_ptr(),
                                       None) == 0
        assert_bits_equal(host(xyz), SO.grid_cell_points(C, H, bound, noise), f"cell points C={C} H={H}")
        # a slice of the cells (multi-GPU update: one slice per rank) equals the same rows of the whole grid
        first, count = n // 3 + 5, n // 5 + 3
        part = torch.empty(count, 3, device="cuda")
        nzp = nz[first:first + count].contiguous() if with_noise else None
        assert L.nvsf_grid_cell_points_range(C, H, bound, nzp.data_ptr() if with_noise else None, first, count,
                                             part.data_ptr(), None) == 0
        assert torch.equal(part, xyz[first:first + count])
    x = torch.empty(8, 3, device="cuda")
    assert L.nvsf_grid_cell_points_range(1, 16, 1.0, None, 16 ** 3 + 1, 0, x.data_ptr(), None) == -1   # first > n
    assert L.nvsf_grid_cell_points_range(1, 16, 1.0, None, 16 ** 3 - 4, 8, x.data_ptr(), None) == -1  # runs past the end
    assert L.nvsf_grid_cell_points_range(1, 16, 1.0, None, 16 ** 3, 0, x.data_ptr(), None) == 0       # empty slice


def test_grid_update_vs_oracle(pkg, SO):
    L = pkg._lib.lib()
    rng = np.random.default_rng(1)
    n = 2 * 64 ** 3
    grid = rng.random(n, dtype=np.float32) * 0.02
    grid[rng.random(n) < 0.1] = -1.0   # untrained cells stay untouched
    grid[rng.random(n) < 0.3] = 0.0
    sig_a = np.exp(rng.normal(-5, 2, n)).astype(np.float32)
    sig_b = np.exp(rng.normal(-5, 2, n)).astype(np.float32)
    tmp = torch.empty(n, device="cuda")
    assert L.nvsf_grid_accumulate(tmp.data_ptr(), torch.from_numpy(sig_a).cuda().data_ptr(), n, 1.5, 1, None) == 0
    assert L.nvsf_grid_accumulate(tmp.data_ptr(), torch.from_numpy(sig_b).cuda().data_ptr(), n, 1.5, 0, None) == 0
    want_tmp = np.maximum(sig_a * np.float32(1.5), sig_b * np.float32(1.5))
    assert_bits_equal(host(tmp), want_tmp, "tmp grid")
    g = torch.from_numpy(grid).cuda()
    bits = torch.zeros(n // 8, dtype=torch.uint8, device="cuda")
    stats = torch.zeros(2, device="cuda")
    wb = L.nvsf_grid_update_workspace_bytes(n)
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
    for thresh in (0.01, 1e-6):
        g.copy_(torch.from_numpy(grid))
        assert L.nvsf_grid_update(g.data_ptr(), tmp.data_ptr(), n, 0.95, thresh, bits.data_ptr(), stats.data_ptr(),
                                  ws.data_ptr(), wb, None) == 0
        eg, mean, th, ebits = SO.grid_update(grid, want_tmp, 0.95, thresh)
        assert_bits_equal(host(g), eg, "density grid")
        st = host(stats)
        assert abs(st[0] - mean) <= 1e-6 * mean and st[1] == min(st[0], np.float32(thresh))
        from oracle import raymarching_oracle as RO
        np.testing.assert_array_equal(bits.cpu().numpy(), RO.packbits(eg, st[1]))
        if st[1] == th:
            np.testing.assert_array_equal(bits.cpu().numpy(), ebits)
    assert L.nvsf_grid_update(g.data_ptr(), tmp.data_ptr(), n, 0.95, 0.01, bits.data_ptr(), stats.data_ptr(),
                              ws.data_ptr(), 8, None) == -2


def test_update_extra_state(model, orc, SO):
    """End to end on the real field: sigma at the jittered cell points vs the oracle on a sample
    of cells (1e-2), decay on the second update, union over times, bitfield == packbits(grid)."""
    from oracle import raymarching_oracle as RO
    C, H = model.cascade, model.grid_size
    n = C * H ** 3
    noise = torch.rand(n, 3, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    model._grid = {}
    bits = model.update_extra_state(0.5, cal_lidar_color=True, noise=noise)
    grid1 = host(model.density_grid(True)).reshape(-1)
    x = SO.grid_cell_points(C, H, S.BOUND, host(noise))
    idx = np.random.default_rng(0).choice(n, 2000, replace=False)
    with torch.no_grad():
        e = orc.density(torch.from_numpy(x[idx]), 0.5, True)["sigma"].numpy()
    close(grid1[idx], e, 1e-2, 0, "grid after first update")   # grid0 = 0 -> max(0, sigma)
    mean = float(model.mean_density(True))
    assert abs(mean - grid1.clip(0).astype(np.float64).mean()) <= 1e-6 * mean
    th = min(np.float32(mean), np.float32(model.density_thresh))
    np.testing.assert_array_equal(bits.cpu().numpy(), RO.packbits(grid1, th))
    assert 0 < np.unpackbits(bits.cpu().numpy()).mean() <= 1
    # second update at two other times with a strong decay: max(grid*decay, max_t sigma_t)
    model.update_extra_state([0.0, 1.0], cal_lidar_color=True, decay=0.5, noise=noise)
    grid2 = host(model.density_grid(True)).reshape(-1)
    with torch.no_grad():
        e0 = orc.density(torch.from_numpy(x[idx]), 0.0, True)["sigma"].numpy()
        e1 = orc.density(torch.from_numpy(x[idx]), 1.0, True)["sigma"].numpy()
    close(grid2[idx], np.maximum(grid1[idx] * np.float32(0.5), np.maximum(e0, e1)), 1e-2, 0, "grid after decay")
    # the camera grid is separate state
    assert not host(model.density_grid(False)).any()


def test_compact_alive(pkg):
    L = pkg._lib.lib()
    rng = np.random.default_rng(2)
    for n in (1, 31, 1024, 1025, 67980, 529408):
        a = rng.integers(0, n, n).astype(np.int32)
        a[rng.random(n) < 0.6] = -1
        if n == 1024:
            a[:] = -1
        ta = torch.from_numpy(a).cuda()
        out = torch.full((n,), -7, dtype=torch.int32, device="cuda")
        cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
        wb = L.nvsf_compact_alive_workspace_bytes(n)
        ws = torch.empty(max(wb, 4), dtype=torch.uint8, device="cuda")
        assert L.nvsf_compact_alive(ta.data_ptr(), n, out.data_ptr(), cnt.data_ptr(), ws.data_ptr(), wb, None) == 0
        want = a[a >= 0]
        assert int(cnt) == want.size
        np.testing.assert_array_equal(out.cpu().numpy()[:want.size], want)
    assert L.nvsf_compact_alive(None, 0, None, cnt.data_ptr(), None, 0, None) == 0 and int(cnt) == 0


# ------------------------------------------------------------------------------ run_cuda
def _bitfield(fill):
    return S.packbits_np(S.density_grid(fill), 0.01)


@pytest.mark.parametrize("lidar", [True, False])
@pytest.mark.parametrize("one_shot", [True, False])
def test_run_cuda_vs_oracle(model, orc, SO, lidar, one_shot):
    from oracle import raymarching_oracle as RO
    N = 192
    o, d = (S.lidar_rays if lidar else S.camera_rays)(N, seed=3)
    bf = _bitfield("shell")
    noises = np.random.default_rng(9).random(N, dtype=np.float32)
    if lidar:
        nears = np.full(N, S.MIN_NEAR_LIDAR, np.float32); fars = np.full(N, S.LIDAR_MAX_DEPTH, np.float32)
    else:
        nears, fars = RO.near_far_from_aabb(o, d, S.AABB, S.MIN_NEAR)
    t = 0.5
    kw = dict(dt_gamma=S.DT_GAMMA, max_steps=1024, T_thresh=1e-2, one_shot=one_shot)
    e = SO.run_cuda(orc, o, d, t, lidar, bf, S.CASCADE, S.GRID_SIZE, S.BOUND, nears, fars, noises=noises,
                    n_step_fn=lambda n, a: max(min(n // a, 8), 1) * 16, **kw)
    r = model.run_cuda(torch.from_numpy(o).cuda()[None], torch.from_numpy(d).cuda()[None], t, cal_lidar_color=lidar,
                       noises=torch.from_numpy(noises).cuda(), density_bitfield=torch.from_numpy(bf).cuda(),
                       perturb=True, **kw)
    sfx = "_lidar" if lidar else ""
    assert r["image" + sfx].shape == (1, N, 2 if lidar else 3) and r["depth" + sfx].shape == (1, N)
    assert model.last_run_cuda_samples == e["n_samples"]   # same sample counts: the marcher is bit-exact
    close(host(r["weights_sum" + sfx]), e["weights_sum"], 1e-2, 1e-5, "weights_sum")
    close(host(r["depth" + sfx])[0], e["depth"], 1e-2, 1e-5, "depth")
    close(host(r["image" + sfx])[0], e["image"], 1e-2, 1e-4, "image")
    assert e["weights_sum"].max() > 0.05


def test_run_cuda_loop_independent_of_step_size(model):
    """The alive-ray loop composites the same samples in the same order whatever n_step is, and
    equals the one-shot path with the same T_thresh — up to fp32 rounding of the restart point:
    composite_rays stores t = sum(deltas[:,1]) and march_rays resumes from it (raymarching.cu:
    846,1046), which differs in the last bits from the marcher's own running t."""
    N = 4096
    o, d = S.camera_rays(N, seed=1)
    to, td = torch.from_numpy(o).cuda()[None], torch.from_numpy(d).cuda()[None]
    bf = torch.from_numpy(_bitfield("shell")).cuda()
    kw = dict(cal_lidar_color=False, dt_gamma=S.DT_GAMMA, T_thresh=1e-2, density_bitfield=bf)
    a = model.run_cuda(to, td, 0.25, one_shot=False, step_scale=16, **kw)
    b = model.run_cuda(to, td, 0.25, one_shot=False, step_scale=1, **kw)
    c = model.run_cuda(to, td, 0.25, one_shot=True, **kw)
    for k in ("depth", "image", "weights_sum"):
        np.testing.assert_allclose(host(a[k]), host(b[k]), rtol=5e-5, atol=1e-6)
        np.testing.assert_allclose(host(a[k]), host(c[k]), rtol=5e-5, atol=1e-6)
    assert float(a["weights_sum"].max()) > 0.05


def test_run_cuda_with_updated_grid(model):
    """update_extra_state -> run_cuda: with the field's own grid the occupancy-skipping render
    approaches the dense uniform render of the same rays (same field, different quadrature)."""
    model._grid = {}
    for _ in range(2):
        model.update_extra_state(0.5, cal_lidar_color=True, perturb=True)
    o, d = S.lidar_rays(512, seed=6)
    to, td = torch.from_numpy(o).cuda()[None], torch.from_numpy(d).cuda()[None]
    r = model.run_cuda(to, td, 0.5, cal_lidar_color=True, dt_gamma=0.0, one_shot=True)
    u = model.render(to, td, 0.5, cal_lidar_color=True, num_steps=768)
    ws_m, ws_u = host(r["weights_sum_lidar"]), host(u["weights_sum_lidar"])
    assert np.isfinite(ws_m).all() and ws_m.max() <= 1 + 1e-5
    assert abs(ws_m.mean() - ws_u.mean()) < 0.25 * max(ws_u.mean(), 1e-3)


def test_color_net_tcgen05_matches_mma_sync(pkg, model):
    """color_net on tcgen05.mma / TMEM (csrc/color.cu k_color_tc, option heads_tc, camera) against the
    mma.sync kernel k_field_color: same fp16 operands, fp32 accumulation in a different order; ragged
    last tile, whole 128-sample tiles masked out, both geo layouts."""
    L = pkg._lib.lib()
    n = 100001
    rng = np.random.default_rng(8)
    x = ((rng.random((n, 3), dtype=np.float32) * 2 - 1) * np.float32(1.9)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    mask = rng.random(n) < 0.5
    mask[1024:2048] = False
    den = model.density(torch.from_numpy(x).cuda(), 0.3, False)
    geo32 = den["geo_feat"].float().contiguous()
    dd, mm = torch.from_numpy(d).cuda(), torch.from_numpy(mask).cuda()
    out = {}
    try:
        for tc in (0, 1):
            assert L.nvsf_set_option(b"heads_tc", tc) == 0
            out[tc] = (host(model.color(None, dd, den["geo_feat"], None, False)),
                       host(model.color(None, dd, geo32, mm, False)))
    finally:
        L.nvsf_set_option(b"heads_tc", 6)
    assert np.abs(out[0][0]).max() > 0.1
    close(out[1][0], out[0][0], 2e-3, 2e-3, "color_net tcgen05 vs mma.sync (geo16 view)")
    close(out[1][1], out[0][1], 2e-3, 2e-3, "color_net tcgen05 vs mma.sync (fp32 geo, mask)")
    assert not out[1][1][~mask].any()
