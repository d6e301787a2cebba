"""Error-map guided ray sampling (torch-ngp's convention, DESIGN.md §3.5, parity unpinned): the numpy oracle
against the exact successive-sampling probabilities and torch, and on the GPU the sampler / update kernels
against the oracle and torch bit for bit, with no host sync and under CUDA-graph capture."""
import ctypes
import importlib
import itertools
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import error_map_oracle as SO

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

LIDAR_HW, CAMERA_HW = (66, 1030), (376, 1408)


def _pkg():
    p = importlib.import_module("selfsupervised-nvsf_b200")
    importlib.import_module("selfsupervised-nvsf_b200.build").build()
    return p


def inclusion_probabilities(w, N):
    """P(cell i is among N draws without replacement, each draw proportional to the remaining weight),
    enumerated over every ordered draw.  Zero-weight cells are never drawn (N <= #positive)."""
    w = np.asarray(w, np.float64)
    p = np.zeros(len(w))
    for seq in itertools.permutations(np.flatnonzero(w > 0), N):
        pr, left = 1.0, w.sum()
        for c in seq:
            pr *= w[c] / left
            left -= w[c]
        p[list(seq)] += pr
    return p


def assert_within_5_sigma(freq, p, trials, what):
    sigma = np.sqrt(p * (1 - p) / trials)
    bad = np.abs(freq - p) > 5 * sigma + 1e-12
    assert not bad.any(), f"{what}: frequencies {freq[bad]} vs probabilities {p[bad]} (5 sigma {5 * sigma[bad]})"


def torch_ngp_inds(inds_coarse, jitter, res, H, W):
    """torch-ngp's coarse -> fine expression, evaluated by torch (rand(N, 2) holds both jitters)."""
    ix, iy = inds_coarse // res, inds_coarse % res
    sx, sy = H / res, W / res
    ix = (ix * sx + jitter[..., 0] * sx).long().clamp(max=H - 1)
    iy = (iy * sy + jitter[..., 1] * sy).long().clamp(max=W - 1)
    return ix * W + iy


# ------------------------------------------------------------------------------------------------------ CPU
W9 = np.array([5.0, 1.0, 0.0, 3.0, 0.5, 2.0, 8.0, 1.0, 0.25], np.float32)


def test_oracle_matches_exact_inclusion_probabilities():
    p = inclusion_probabilities(W9, 3)
    assert p.sum() == pytest.approx(3.0)
    trials = 100_000
    rng = np.random.default_rng(0)
    E = rng.exponential(size=(trials, 9)).astype(np.float32)
    jit = np.zeros((3, 2), np.float32)
    counts = np.zeros(9)
    for t in range(trials):
        cells, _ = SO.error_map_sample(W9, E[t], jit, 3, 3, 3, 3)
        counts[cells] += 1
    assert counts[2] == 0
    assert_within_5_sigma(counts / trials, p, trials, "oracle")


def test_torch_multinomial_cpu_matches_the_same_probabilities():
    p = inclusion_probabilities(W9, 3)
    trials = 100_000
    g = torch.Generator().manual_seed(0)
    draws = torch.multinomial(torch.from_numpy(W9).expand(trials, 9), 3, replacement=False, generator=g)
    freq = np.bincount(draws.reshape(-1).numpy(), minlength=9) / trials
    assert_within_5_sigma(freq, p, trials, "torch.multinomial")


def test_zero_weight_cells_fill_by_smallest_expo():
    # positive cells: 1 and 4 only (0, -1, nan, inf have zero weight); N = 4 takes both, then the two smallest E
    # among the others, the tie at E = 0.3 going to the lower cell
    w = np.array([0, 2, 0, -1, 1, np.nan, np.inf, 0, 0], np.float32)
    E = np.array([0.9, 5.0, 0.3, 0.7, 9.0, 0.1, 0.3, 0.3, 2.0], np.float32)
    cells, _ = SO.error_map_sample(w, E, np.zeros((4, 2), np.float32), 3, 4, 3, 3)
    assert cells.tolist() == [1, 2, 4, 5]
    cells, _ = SO.error_map_sample(w, E, np.zeros((2, 2), np.float32), 3, 2, 3, 3)
    assert cells.tolist() == [1, 4]                     # N <= #positive: the fill tier is never used
    cells, _ = SO.error_map_sample(w, E, np.zeros((9, 2), np.float32), 3, 9, 3, 3)
    assert cells.tolist() == list(range(9))


def test_key_ties_go_to_the_lower_cell():
    w = np.ones(9, np.float32)
    E = np.array([0.5, 0.1, 0.5, 0.5, 0.2, 0.5, 0.5, 0.5, 0.5], np.float32)
    cells, _ = SO.error_map_sample(w, E, np.zeros((3, 2), np.float32), 3, 3, 3, 3)
    assert cells.tolist() == [0, 1, 4]
    w = np.array([1, 2, 1, 4, 1, 1, 1, 1, 1], np.float32)  # keys 1/2 and 2/4 tie exactly
    E = np.array([3, 1, 3, 2, 3, 3, 3, 3, 3], np.float32)
    cells, _ = SO.error_map_sample(w, E, np.zeros((1, 2), np.float32), 3, 1, 3, 3)
    assert cells.tolist() == [1]


@pytest.mark.parametrize("res,H,W", [(128, *LIDAR_HW), (128, *CAMERA_HW), (127, *LIDAR_HW), (5, 7, 9)])
def test_oracle_mapping_equals_torch_ngp_expression_on_cpu(res, H, W):
    rng = np.random.default_rng(res)
    R, N = res * res, min(res * res, 2048)
    w = rng.random(R).astype(np.float32)
    E = rng.exponential(size=R).astype(np.float32)
    jit = rng.random((N, 2), dtype=np.float32)
    jit[:4] = np.float32(1) - np.finfo(np.float32).epsneg    # the largest jitter: the clamp at the frame's edge
    cells, inds = SO.error_map_sample(w, E, jit, res, N, H, W)
    want = torch_ngp_inds(torch.from_numpy(cells), torch.from_numpy(jit), res, H, W)
    assert np.array_equal(inds, want.numpy())


def test_oracle_update_equals_torch_gather_scatter():
    rng = np.random.default_rng(1)
    m = rng.random(16384).astype(np.float32) * 3
    ic = np.sort(rng.choice(16384, 4096, replace=False))
    e = rng.random(4096).astype(np.float32)
    t = torch.from_numpy(m.copy())
    ict = torch.from_numpy(ic)
    t.scatter_(0, ict, 0.1 * t.gather(0, ict) + 0.9 * torch.from_numpy(e))
    got = SO.error_map_update(m, ic, e)
    assert np.array_equal(got.view(np.uint32), t.numpy().view(np.uint32))


def test_c_abi_rejects_invalid_arguments():
    """Every argument check fires before anything is launched, so it runs without a device; the pointers are
    never dereferenced."""
    L = _pkg()._lib.lib()
    p = ctypes.c_void_p(256)
    ok = dict(map=p, expo=p, jit=p, res=128, N=2048, H=66, W=1030, ic=p, inds=p)

    def sample(**kw):
        a = {**ok, **kw}
        return L.nvsf_error_map_sample(a["map"], a["expo"], a["jit"], a["res"], a["N"], a["H"], a["W"], a["ic"],
                                       a["inds"], None)

    for bad in (dict(N=0), dict(N=128 * 128 + 1), dict(res=0), dict(res=225, N=1), dict(H=0), dict(W=0),
                dict(map=None), dict(expo=None), dict(jit=None), dict(ic=None), dict(inds=None)):
        assert sample(**bad) == -1, bad
    assert L.nvsf_error_map_update(None, 16, p, 4, p, None) == -1
    assert L.nvsf_error_map_update(p, 0, p, 4, p, None) == -1
    assert L.nvsf_error_map_update(p, 16, None, 4, p, None) == -1
    assert L.nvsf_error_map_update(p, 16, p, 4, None, None) == -1
    assert L.nvsf_error_map_update(None, 0, None, 0, None, None) == 0     # nothing to do


# ------------------------------------------------------------------------------------------------------ GPU
def _map(kind, R, N, g):
    if kind == "ones":
        return torch.ones(R)
    if kind == "uniform":
        return torch.rand(R, generator=g)
    if kind == "heavy":                       # Pareto-like: a few cells hold most of the weight
        return torch.rand(R, generator=g).clamp_min(1e-6) ** -3.0
    if kind == "few_positive":                # fewer positive cells than N: the fill tier is used
        w = torch.zeros(R)
        w[torch.randperm(R, generator=g)[: N // 2]] = torch.rand(N // 2, generator=g) + 0.1
        return w
    w = torch.rand(R, generator=g)            # "nonfinite": NaN, inf, negative and zero entries
    idx = torch.randperm(R, generator=g)
    q = R // 8
    w[idx[:q]] = float("nan")
    w[idx[q:2 * q]] = -1.0
    w[idx[2 * q:3 * q]] = 0.0
    w[idx[3 * q:3 * q + 3]] = float("inf")
    return w


def _sample_dev(L, w, E, jit, res, N, H, W):
    ic = torch.full((N,), -7, dtype=torch.int64, device="cuda")     # dirty outputs: every entry must be written
    inds = torch.full((N,), -7, dtype=torch.int64, device="cuda")
    st = L.nvsf_error_map_sample(w.data_ptr(), E.data_ptr(), jit.data_ptr(), res, N, H, W, ic.data_ptr(),
                                 inds.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert st == 0
    return ic, inds


CASES = [(res, N) for res in (128, 127, 5) for N in (1, 2048, 4096, res * res) if N <= res * res]


@gpu
@pytest.mark.parametrize("res,N", CASES)
@pytest.mark.parametrize("hw", [LIDAR_HW, CAMERA_HW], ids=["lidar", "camera"])
def test_sampler_bit_exact_against_oracle(res, N, hw):
    L = _pkg()._lib.lib()
    H, W = hw
    R = res * res
    g = torch.Generator().manual_seed(res * 7919 + N)
    for kind in ("ones", "uniform", "heavy", "few_positive", "nonfinite"):
        w = _map(kind, R, N, g).float()
        E = torch.empty(R).exponential_(generator=g)
        jit = torch.rand(N, 2, generator=g)
        ic, inds = _sample_dev(L, w.cuda(), E.cuda(), jit.cuda(), res, N, H, W)
        want_c, want_i = SO.error_map_sample(w.numpy(), E.numpy(), jit.numpy(), res, N, H, W)
        got_c, got_i = ic.cpu().numpy(), inds.cpu().numpy()
        assert np.array_equal(got_c, want_c), kind
        assert np.array_equal(got_i, want_i), kind
        # torch-ngp's expression on the GPU, from the returned cells and the same jitter
        assert torch.equal(inds, torch_ngp_inds(ic, jit.cuda(), res, H, W)), kind
        # distinct, ascending, and every pixel inside (the closure of) its cell's footprint
        assert (np.diff(got_c) > 0).all() and got_c[0] >= 0 and got_c[-1] < R
        row, col, cr, cc = got_i // W, got_i % W, got_c // res, got_c % res
        assert ((row >= cr * H // res) & (row <= np.minimum(-(-(cr + 1) * H // res), H - 1))).all(), kind
        assert ((col >= cc * W // res) & (col <= np.minimum(-(-(cc + 1) * W // res), W - 1))).all(), kind


@gpu
def test_gpu_inclusion_frequencies_match_probabilities():
    """A 16-cell map, 4000 draws of N = 3 through get_lidar_rays (one map per pose), seeded."""
    pkg = _pkg()
    w = torch.tensor([4, 1, 0, 2, 0.5, 3, 1, 6, 0.25, 2, 1, 0, 5, 1.5, 1, 0.75])
    p = inclusion_probabilities(w.numpy(), 3)
    trials = 4000
    torch.manual_seed(11)
    poses = torch.eye(4, device="cuda").expand(trials, 4, 4)
    r = pkg.rays.get_lidar_rays(poses, [2.0, 26.9], [180.0, 360.0], 8, 8, 3,
                                error_map=w.cuda().expand(trials, 16), use_error_map=True)
    ic = r["inds_coarse"].cpu()
    assert (ic[:, 1:] > ic[:, :-1]).all()
    freq = np.bincount(ic.reshape(-1).numpy(), minlength=16) / trials
    assert freq[2] == 0 and freq[11] == 0
    assert_within_5_sigma(freq, p, trials, "GPU sampler")


def _torch_update(maps, index, ic, loss):
    m = maps.clone()
    for b, f in enumerate(index):
        row = m[f]
        row.scatter_(0, ic[b], 0.1 * row.gather(0, ic[b]) + 0.9 * loss[b])
    return m


@gpu
def test_update_bit_exact_and_touches_nothing_else():
    pkg = _pkg()
    torch.manual_seed(2)
    F, R, N = 6, 128 * 128, 4096
    maps = torch.rand(F, R, device="cuda") * 4
    index = [4, 1, 2]
    r = pkg.rays.get_lidar_rays(torch.eye(4, device="cuda").expand(3, 4, 4), [2.0, 26.9], [180.0, 360.0], *LIDAR_HW,
                                N, error_map=maps[index], use_error_map=True)
    loss = torch.rand(3, N, device="cuda") * 2
    want = _torch_update(maps, index, r["inds_coarse"], loss)
    before = maps.clone()
    pkg.rays.update_error_map(maps, index, r["inds_coarse"], loss)
    assert torch.equal(maps.view(torch.int32), want.view(torch.int32))
    for b, f in enumerate(index):
        got = SO.error_map_update(before[f].cpu().numpy(), r["inds_coarse"][b].cpu().numpy(), loss[b].cpu().numpy())
        assert np.array_equal(maps[f].cpu().numpy().view(np.uint32), got.view(np.uint32))
    untouched = torch.ones(F, R, dtype=torch.bool, device="cuda")
    for b, f in enumerate(index):
        untouched[f, r["inds_coarse"][b]] = False
    assert torch.equal(maps[untouched].view(torch.int32), before[untouched].view(torch.int32))
    assert (~untouched).sum().item() == 3 * N


@gpu
@pytest.mark.parametrize("kind", ["lidar", "camera"])
def test_rays_equal_existing_kernels_on_returned_inds(kind):
    pkg = _pkg()
    g = np.load(os.path.join(GOLDEN, "rays_ref.npz"))
    poses = torch.from_numpy(np.stack([g["pose_a"], g["pose_b"]])).cuda()
    maps = torch.rand(2, 128 * 128, device="cuda")
    if kind == "lidar":
        H, W = LIDAR_HW
        gen = lambda **kw: pkg.rays.get_lidar_rays(poses, g["lidar_K"], g["lidar_K_hoz"], H, W, **kw)
    else:
        H, W = CAMERA_HW
        gen = lambda **kw: pkg.rays.get_rays(poses, g["cam_K"], H, W, **kw)
    torch.manual_seed(5)
    r = gen(N=2048, error_map=maps, use_error_map=True)
    torch.manual_seed(5)
    r2 = gen(N=2048, error_map=maps.cpu(), use_error_map=True)       # a host map is moved to the device
    assert torch.equal(r["inds"], r2["inds"]) and torch.equal(r["inds_coarse"], r2["inds_coarse"])
    assert r["inds"].shape == (2, 2048) and r["inds_coarse"].shape == (2, 2048)
    assert not torch.equal(r["inds"][0], r["inds"][1])                # one draw per pose
    full = gen(N=-1, error_map=maps, use_error_map=True)              # N <= 0: the full frame, the map ignored
    assert "inds_coarse" not in full and full["inds"].shape == (2, H * W)
    for b in range(2):
        assert torch.equal(r["rays_o"][b], full["rays_o"][b][r["inds"][b]])
        assert torch.equal(r["rays_d"][b].view(torch.int32), full["rays_d"][b][r["inds"][b]].view(torch.int32))
    # the draws are exponential_ [B, R] and then rand [B, N, 2] from the current generator
    torch.manual_seed(5)
    E = torch.empty(2, 128 * 128, device="cuda").exponential_()
    jit = torch.rand(2, 2048, 2, device="cuda")
    for b in range(2):
        c, i = SO.error_map_sample(maps[b].cpu().numpy(), E[b].cpu().numpy(), jit[b].cpu().numpy(), 128, 2048, H, W)
        assert np.array_equal(r["inds_coarse"][b].cpu().numpy(), c) and np.array_equal(r["inds"][b].cpu().numpy(), i)
    # use_error_map=False ignores the map and draws exactly what it drew before
    torch.manual_seed(5)
    r3 = gen(N=2048, error_map=maps, use_error_map=False)
    torch.manual_seed(5)
    assert torch.equal(r3["inds"][0], torch.randint(0, H * W, size=[2048], device="cuda"))
    assert "inds_coarse" not in r3


@gpu
def test_sample_loss_update_without_host_sync():
    pkg = _pkg()
    maps = torch.rand(4, 128 * 128, device="cuda")
    poses = torch.eye(4, device="cuda")[None].expand(2, 4, 4)
    pred_d = torch.rand(2, 2048, device="cuda")
    pred_i = torch.rand(2, 2048, 2, device="cuda")
    gt = torch.rand(2, 2048, 3, device="cuda")
    index = [3, 0]
    em = maps[index]
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        r = pkg.rays.get_lidar_rays(poses, [2.0, 26.9], [180.0, 360.0], *LIDAR_HW, 2048, error_map=em,
                                    use_error_map=True)
        loss = pkg.losses.lidar_loss(pred_d, pred_i, gt)
        pkg.rays.update_error_map(maps, index, r["inds_coarse"], loss)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.isfinite(maps).all()


@gpu
def test_cuda_graph_capture_of_sample_and_update():
    pkg = _pkg()
    F, R, N = 3, 128 * 128, 2048
    maps = torch.rand(F, R, device="cuda")
    poses = torch.eye(4, device="cuda")[None].expand(2, 4, 4).contiguous()
    em = torch.rand(2, R, device="cuda")
    loss = torch.rand(2, N, device="cuda")
    index = [2, 0]
    run = lambda: pkg.rays.get_lidar_rays(poses, [2.0, 26.9], [180.0, 360.0], *LIDAR_HW, N, error_map=em,
                                          use_error_map=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):              # warm-up outside the capture
        pkg.rays.update_error_map(maps, index, run()["inds_coarse"], loss)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run()
        pkg.rays.update_error_map(maps, index, out["inds_coarse"], loss)
    seen = []
    for _ in range(3):
        before = maps.clone()
        graph.replay()
        torch.cuda.synchronize()
        ic = out["inds_coarse"]
        assert (ic[:, 1:] > ic[:, :-1]).all() and ic.min() >= 0 and ic.max() < R
        row, cr = out["inds"] // LIDAR_HW[1], ic // 128
        assert ((row >= cr * LIDAR_HW[0] // 128) & (row <= (cr + 1) * LIDAR_HW[0] // 128)).all()
        assert torch.equal(maps.view(torch.int32), _torch_update(before, index, ic, loss).view(torch.int32))
        seen.append(ic.clone())
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])   # fresh draws per replay


@gpu
def test_training_step_end_to_end():
    """Sample -> render(staged=False) -> lidar_loss -> backward -> update_error_map with the synthetic model."""
    import field_cases as FC
    pkg = _pkg()
    S = FC.S
    torch.manual_seed(0)
    model = pkg.NeRFNetwork(log2_hashmap_size=12, hash_size_dynamic=(10, 9, 9), flow_log2_hashmap_size=11,
                            time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND,
                            min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR,
                            lidar_max_depth=S.LIDAR_MAX_DEPTH).train()
    g = np.load(os.path.join(GOLDEN, "rays_ref.npz"))
    pose = torch.from_numpy(g["pose_a"]).clone()
    pose[:3, 3] *= 0.2
    F, R, N = 4, 128 * 128, 1024
    maps = torch.ones(F, R, device="cuda")
    index = [2]
    r = pkg.rays.get_lidar_rays(pose[None].cuda(), g["lidar_K"], g["lidar_K_hoz"], *LIDAR_HW, N,
                                error_map=maps[index], use_error_map=True)
    t = torch.tensor([[0.3]], device="cuda")
    out = model.render(r["rays_o"], r["rays_d"], t, cal_lidar_color=True, staged=False, num_steps=64, perturb=True)
    gt = torch.rand(1, N, 3, device="cuda")
    gt[..., 0] = (gt[..., 0] > 0.3).float()
    loss = pkg.losses.lidar_loss(out["depth_lidar"], out["image_lidar"], gt)
    assert loss.shape == (1, N)
    loss.mean().backward()
    grads = [p.grad for p in model.parameters() if p.grad is not None]
    assert grads and all(torch.isfinite(x).all() for x in grads)
    before = maps.clone()
    pkg.rays.update_error_map(maps, index, r["inds_coarse"], loss)
    assert torch.equal(maps.view(torch.int32), _torch_update(before, index, r["inds_coarse"], loss.detach())
                       .view(torch.int32))
    assert torch.equal(maps[[0, 1, 3]], before[[0, 1, 3]])


@gpu
def test_python_argument_checks():
    pkg = _pkg()
    Err = pkg._lib.NvsfError
    P = torch.eye(4, device="cuda")[None]
    lid = lambda **kw: pkg.rays.get_lidar_rays(P, [2.0, 26.9], [180.0, 360.0], *LIDAR_HW, **kw)
    with pytest.raises(Err):
        lid(N=16, error_map=torch.ones(1, 15, device="cuda"), use_error_map=True)        # not a square
    with pytest.raises(Err):
        lid(N=26, error_map=torch.ones(1, 25, device="cuda"), use_error_map=True)        # N > R
    with pytest.raises(Err):
        lid(N=16, error_map=torch.ones(2, 25, device="cuda"), use_error_map=True)        # B disagrees
    with pytest.raises(NotImplementedError):
        lid(N=16, use_error_map=True)                                                    # no map
    with pytest.raises(NotImplementedError):
        lid(N=16, error_map=torch.ones(1, 25, device="cuda"), use_error_map=True, patch_size=2)
    maps = torch.ones(3, 25, device="cuda")
    ic = torch.arange(4, device="cuda")[None]
    e = torch.ones(1, 4, device="cuda")
    for index in ([3], [-1], [0, 0]):
        with pytest.raises(Err):
            pkg.rays.update_error_map(maps, index, ic.expand(len(index), 4), e.expand(len(index), 4))
    with pytest.raises(Err):
        pkg.rays.update_error_map(maps.cpu(), [0], ic, e)
    with pytest.raises(Err):
        pkg.rays.update_error_map(maps, [0], ic, torch.ones(1, 5, device="cuda"))
    with pytest.raises(Err):
        pkg.rays.update_error_map(maps, torch.tensor([0], device="cuda"), ic, e)
    L = pkg._lib.lib()
    x = torch.zeros(16384, device="cuda")
    i64 = torch.zeros(16, dtype=torch.int64, device="cuda")
    st = lambda res, N, H=8, W=8: L.nvsf_error_map_sample(x.data_ptr(), x.data_ptr(), x.data_ptr(), res, N, H, W,
                                                          i64.data_ptr(), i64.data_ptr(), None)
    assert st(4, 0) == -1 and st(4, 17) == -1 and st(225, 1) == -1 and st(4, 4, H=0) == -1 and st(4, 4, W=0) == -1
    assert st(4, 16) == 0
    torch.cuda.synchronize()
