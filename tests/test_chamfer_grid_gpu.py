"""GPU: the uniform-grid path of the Chamfer forward (csrc/chamfer.cu k_grid_*) against the brute-force scan.

Every test runs the same inputs with option "chamfer_grid" forced on (1) and off (0) and asserts dist and idx
bit-identical: golden cases, sizes and batches, points on cell faces, ties at zero and positive distances,
degenerate / non-finite / extreme clouds, LiDAR-like scans and a 1 M-point accumulated cloud, the counted form
with garbage padding, determinism, gradients, flow_loss, the automatic selection, LidarMeter and PointsMeter."""
import math
import os

import numpy as np
import pytest

import chamfer_cases as CC
from conftest import GOLDEN

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
from oracle import chamfer_oracle as CO
from oracle import metrics_oracle as MO

LIDAR_K, LIDAR_K_HOZ = (2.0, 26.9), (180.0, 360.0)
H_FULL, W_FULL = 66, 1030


def _forward(pkg, a, b, grid):
    with pkg._lib.option_scope({"chamfer_grid": grid}):
        return [t.clone() for t in pkg.chamfer.chamfer_3DDist()(a, b)]


def _same(x, y, what=""):
    for u, v in zip(x, y):
        if u.dtype == torch.float32:
            u, v = u.view(torch.int32), v.view(torch.int32)
        assert torch.equal(u, v), what


def both(pkg, a, b, what=""):
    """grid and brute-force results of the [B,n,3] / [B,m,3] clouds a, b: bit-identical; returns them"""
    a = torch.as_tensor(a).cuda().float()
    b = torch.as_tensor(b).cuda().float()
    if a.dim() == 2:
        a, b = a[None], b[None]
    g = _forward(pkg, a, b, 1)
    f = _forward(pkg, a, b, 0)
    _same(g, f, what)
    return g


def _uniform(n, seed, lo=-1.0, hi=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return lo + (hi - lo) * torch.rand(n, 3, device="cuda", generator=g)


def _scan_depth(seed, H=H_FULL, W=W_FULL, pkg=None):
    """A street-like range image: ground plane 1.7 m below the sensor, walls of a 40 x 24 m box, a few boxes
    (cars), clipped to 80 m, 2 cm of range noise, every 9th ray dropped."""
    dirs = pkg.rays.get_lidar_rays(torch.eye(4, device="cuda")[None], LIDAR_K, LIDAR_K_HOZ, H, W, -1)["rays_d"][0]
    dx, dy, dz = dirs[:, 0], dirs[:, 1], dirs[:, 2]
    inf = torch.full_like(dx, math.inf)
    t = torch.where(dz < -1e-6, -1.7 / dz, inf)
    for d, half in ((dx, 20.0), (dy, 12.0)):
        t = torch.minimum(t, torch.where(d.abs() > 1e-6, half / d.abs(), inf))
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(6):      # boxes on the ground
        c = (torch.rand(2, device="cuda", generator=g) * 2 - 1) * torch.tensor([15.0, 9.0], device="cuda")
        tx0, tx1 = (c[0] - 2.0) / dx, (c[0] + 2.0) / dx
        ty0, ty1 = (c[1] - 1.0) / dy, (c[1] + 1.0) / dy
        tn = torch.maximum(torch.minimum(tx0, tx1), torch.minimum(ty0, ty1))
        tf = torch.minimum(torch.maximum(tx0, tx1), torch.maximum(ty0, ty1))
        hit = (tn < tf) & (tn > 0) & (dz * tn > -1.7) & (dz * tn < -0.2)
        t = torch.where(hit, torch.minimum(t, tn), t)
    t = t.clamp(max=80.0) + 0.02 * torch.randn(t.shape, device="cuda", generator=g)
    t[::9] = 0.0
    return t.reshape(H, W)


def _scan(pkg, seed):
    pts, cnt = pkg.metrics.lidar_points(_scan_depth(seed, pkg=pkg), LIDAR_K, LIDAR_K_HOZ)
    return pts[:int(cnt)]


# ------------------------------------------------------------------------------------------------ 1. golden
@pytest.mark.parametrize("name", list(CC.GOLDEN_CASES))
def test_golden_cases_through_the_grid(pkg, name):
    a, b, _, _ = CC.case(name)
    d1, d2, i1, i2 = [t.cpu().numpy() for t in both(pkg, a, b, name)]
    od1, od2, oi1, oi2 = CO.chamfer_forward(a, b)
    assert np.array_equal(i1, oi1) and np.array_equal(i2, oi2)
    assert np.array_equal(d1.view(np.uint32), od1.view(np.uint32)) and np.array_equal(d2.view(np.uint32),
                                                                                      od2.view(np.uint32))
    path = os.path.join(GOLDEN, "chamfer_ref_sm100a.npz")
    if os.path.exists(path):
        gold = np.load(path)
        assert np.array_equal(i1, gold[f"{name}_idx1"]) and np.array_equal(i2, gold[f"{name}_idx2"])
        assert np.array_equal(d1, gold[f"{name}_dist1"]) and np.array_equal(d2, gold[f"{name}_dist2"])


# ------------------------------------------------------------------------------------------ 2. sizes, batches
@pytest.mark.parametrize("n,m", [(5000, 3001), (1, 4000), (4000, 1), (1, 1), (20000, 20000)])
def test_uniform_sizes(pkg, n, m):
    both(pkg, _uniform(n, n), _uniform(m, m + 1) * 1.1, f"{n}x{m}")


def test_batch_of_three_distributions(pkg):
    g = torch.Generator(device="cuda").manual_seed(5)
    n, m = 6000, 4500
    a = torch.empty(3, n, 3, device="cuda")
    b = torch.empty(3, m, 3, device="cuda")
    a[0], b[0] = torch.rand(n, 3, device="cuda", generator=g), torch.rand(m, 3, device="cuda", generator=g)
    a[1], b[1] = torch.randn(n, 3, device="cuda", generator=g) * 30, torch.randn(m, 3, device="cuda", generator=g) * 30
    a[2], b[2] = torch.rand(n, 3, device="cuda", generator=g) * 100, torch.rand(m, 3, device="cuda", generator=g) * 100
    a[2, :, 2] = 0.0                       # a flat cloud in the third element
    b[2, :, 2] *= 0.01
    both(pkg, a, b, "b=3")


# ------------------------------------------------------------------------------------ 3. boundaries and ties
def test_lattice_points_on_cell_faces_and_equal_distance_ties(pkg):
    """Lattices of exactly representable coordinates: targets on or next to cell faces, queries at lattice cell
    centres (8 targets at one distance) and on edge midpoints (2 at one distance); a random index order."""
    g = torch.Generator(device="cuda").manual_seed(9)
    for side, step in ((32, 1.0), (20, 0.25), (64, 0.5)):
        ax = torch.arange(side, device="cuda", dtype=torch.float32) * step
        lat = torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)
        lat = lat[torch.randperm(lat.shape[0], device="cuda", generator=g)]
        centres = lat[: lat.shape[0] // 3] + step * 0.5
        both(pkg, centres, lat, f"centres {side}")
        both(pkg, lat, lat[torch.randperm(lat.shape[0], device="cuda", generator=g)], f"permuted {side}")
        faces = lat[: 5000].clone()
        faces[:, 0] += step * 0.5          # on faces between two lattice points along x
        both(pkg, faces, lat, f"faces {side}")


def test_duplicates_and_permuted_copies(pkg):
    n = 30000
    a = _uniform(n, 11)
    g = torch.Generator(device="cuda").manual_seed(12)
    perm = torch.randperm(n, device="cuda", generator=g)
    d1, d2, i1, i2 = both(pkg, a, a[perm], "permuted")
    assert float(d1.max()) == 0.0 and float(d2.max()) == 0.0
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(n, device="cuda")
    assert torch.equal(i1[0].long(), inv) and torch.equal(i2[0].long(), perm)
    dup = torch.cat([a, a, a[:100]])       # every target two or three times: the first copy wins
    d1, _, i1, _ = both(pkg, a, dup, "duplicates")
    assert float(d1.max()) == 0.0 and torch.equal(i1[0].long(), torch.arange(n, device="cuda"))


def test_tie_with_the_lower_index_in_a_farther_ring(pkg):
    """A query in an empty ball; two targets at the same computed distance, the lower index on the far side of the
    query's home cell (a farther ring than the first hit); several query offsets within a cell."""
    cloud = _uniform(40000, 13, 0.0, 64.0)
    for k, off in enumerate((0.125, 0.375, 0.5, 0.75, 0.9375, 1.375)):   # exact in fp32: 8 is exact too
        q = torch.tensor([32.0 + off, 32.0, 32.0], device="cuda")
        far = (cloud - q).norm(dim=1) > 9.0
        t = cloud[far]
        near = q[None] + torch.tensor([[8.0, 0.0, 0.0], [-8.0, 0.0, 0.0], [0.0, 8.0, 0.0]], device="cuda")
        # indices: -x copy first (lowest), +x copy last; +y in the middle
        t = torch.cat([near[1:2], t[: t.shape[0] // 2], near[2:3], t[t.shape[0] // 2:], near[0:1]])
        queries = torch.cat([q[None], _uniform(500, 14 + k, 0.0, 64.0)])
        d1, _, i1, _ = both(pkg, queries, t, f"offset {off}")
        assert float(d1[0, 0]) == 64.0 and int(i1[0, 0]) == 0


# -------------------------------------------------------------------------------------- 4. degenerate clouds
def test_degenerate_clouds(pkg):
    g = torch.Generator(device="cuda").manual_seed(15)
    n = 20000
    same = torch.full((n, 3), 0.25, device="cuda")
    line = torch.zeros(n, 3, device="cuda")
    line[:, 0] = torch.rand(n, device="cuda", generator=g) * 50
    plane = torch.rand(n, 3, device="cuda", generator=g) * 80 - 40
    plane[:, 2] = 0.0
    cluster = torch.randn(n, 3, device="cuda", generator=g) * 1e-3
    cluster[-1] = torch.tensor([1e4, -3e3, 50.0], device="cuda")
    queries = _uniform(n, 16, -2.0, 2.0)
    for name, t in (("identical", same), ("collinear", line), ("coplanar", plane), ("cluster+outlier", cluster)):
        both(pkg, queries, t, name)
        both(pkg, t, t.flip(0), name + " self")
    far = _uniform(3000, 17) + torch.tensor([500.0, -40.0, 3.0], device="cuda")
    far[:1000] *= 1e4
    both(pkg, far, _uniform(8000, 18), "queries far outside the box")
    both(pkg, far, plane, "far queries, flat targets")


# --------------------------------------------------------------------------------- 5. non-finite and extreme
def test_non_finite_and_extreme_coordinates(pkg):
    a, b = _uniform(6000, 19), _uniform(5000, 20)
    a[::7, 0] = math.nan
    a[3::11, 1] = math.inf
    a[5::13, 2] = -math.inf
    b[::5, 2] = math.nan
    b[2::9, 0] = -math.inf
    b[4::17, 1] = math.inf
    d1, _, i1, _ = both(pkg, a, b, "nan / inf")
    bad = ~torch.isfinite(a[:, :]).all(1)
    assert torch.isinf(d1[0, bad]).all() and (i1[0, bad] == 0).all()
    allbad = torch.full((300, 3), math.nan, device="cuda")
    d1, d2, i1, i2 = both(pkg, a, allbad, "every target NaN")
    assert torch.isinf(d1).all() and (i1 == 0).all() and torch.isinf(d2).all() and (i2 == 0).all()
    big = _uniform(4000, 21) * 3e19      # squares overflow: many distances are +inf
    big2 = _uniform(4000, 22) * 3e19
    big2[:50] = big[:50] * 1.0000001
    both(pkg, big, big2, "1e19")
    both(pkg, big, _uniform(4000, 23), "1e19 vs unit")
    both(pkg, _uniform(4000, 24) * 1e-30, _uniform(5000, 25) * 1e-30, "1e-30 extents")
    both(pkg, _uniform(4000, 26) * 1e-30 + 1.0, _uniform(5000, 27) * 1e-30 + 1.0, "1e-30 around 1")
    both(pkg, _uniform(4000, 28) * 1e-42, _uniform(5000, 29) * 1e-42, "subnormal extents")


# ---------------------------------------------------------------------------------- 6. LiDAR and large clouds
def test_lidar_frame_displaced_and_noisy(pkg):
    pc = _scan(pkg, 1)
    g = torch.Generator(device="cuda").manual_seed(30)
    assert pc.shape[0] > 50000
    both(pkg, pc, pc + torch.tensor([0.05, -0.02, 0.0], device="cuda"), "flow-loss case")
    both(pkg, pc, pc + 0.01 * torch.randn(pc.shape, device="cuda", generator=g), "evaluation case")
    both(pkg, pc, _scan(pkg, 2), "two scans")


def test_accumulated_million_point_cloud(pkg):
    """16 posed scans (about 1 M points) against a noisy copy: once, against the brute-force path."""
    scans = []
    for k in range(16):
        pc = _scan(pkg, 100 + k)
        th = 0.05 * k
        R = torch.tensor([[math.cos(th), -math.sin(th), 0.0], [math.sin(th), math.cos(th), 0.0], [0.0, 0.0, 1.0]],
                         device="cuda")
        scans.append(pc @ R.T + torch.tensor([1.5 * k, 0.2 * k, 0.0], device="cuda"))
    acc = torch.cat(scans)
    assert acc.shape[0] > 900000
    g = torch.Generator(device="cuda").manual_seed(31)
    both(pkg, acc, acc + 0.01 * torch.randn(acc.shape, device="cuda", generator=g), "accumulated")


# ------------------------------------------------------------------------------------------- 7. counted form
def _counted(pkg, a, b, n, m, grid):
    L, P = pkg._lib.lib(), pkg._lib.ptr
    cap_n, cap_m = a.shape[0], b.shape[0]
    cnt = torch.tensor([n, m], dtype=torch.int32, device="cuda")
    out = [torch.full((cap_n,), 7.0, device="cuda"), torch.full((cap_m,), 7.0, device="cuda"),
           torch.full((cap_n,), 7, dtype=torch.int32, device="cuda"), torch.full((cap_m,), 7, dtype=torch.int32,
                                                                                device="cuda")]
    wb = L.nvsf_chamfer_workspace_bytes(1, cap_n, cap_m)
    ws = torch.full((wb,), 0x5A, dtype=torch.uint8, device="cuda")
    with pkg._lib.option_scope({"chamfer_grid": grid}):
        assert L.nvsf_chamfer_forward_counted(P(a), P(b), cap_n, cap_m, P(cnt), P(cnt[1:]), P(out[0]), P(out[1]),
                                              P(out[2]), P(out[3]), P(ws), wb, None) == 0
    return out


@pytest.mark.parametrize("n,m,cap_n,cap_m", [(3000, 2500, 4096, 5000), (1, 700, 1, 1024), (0, 300, 64, 512),
                                             (40, 0, 40, 8), (0, 0, 16, 16), (20000, 18000, 20000, 30000),
                                             (-5, 70000, 100, 65000)])
def test_counted_form_with_garbage_padding(pkg, n, m, cap_n, cap_m):
    a = _uniform(cap_n, cap_n + 1)
    b = _uniform(cap_m, cap_m + 2) * 1.2
    a[max(n, 0):] = math.nan                 # garbage in the padding
    b[max(m, 0):] = -3e38
    g = _counted(pkg, a, b, n, m, 1)
    f = _counted(pkg, a, b, n, m, 0)
    _same(g, f, "counted")
    nn_, mm = min(max(n, 0), cap_n), min(max(m, 0), cap_m)
    if nn_ and mm:
        e = _forward(pkg, a[None, :nn_], b[None, :mm], 1)
        assert torch.equal(g[0][:nn_], e[0][0]) and torch.equal(g[2][:nn_], e[2][0])
        assert torch.equal(g[1][:mm], e[1][0]) and torch.equal(g[3][:mm], e[3][0])
    elif nn_ or mm:
        assert torch.isinf(g[0][:nn_]).all() and (g[2][:nn_] == -1).all()
        assert torch.isinf(g[1][:mm]).all() and (g[3][:mm] == -1).all()
    assert not g[0][nn_:].any() and (g[2][nn_:] == -1).all() and not g[1][mm:].any() and (g[3][mm:] == -1).all()


# --------------------------------------------------------------------------------- 8. determinism, autograd
def test_repeat_runs_are_bit_identical(pkg):
    pc = _scan(pkg, 3)
    other = pc + 0.03
    ref = _forward(pkg, pc[None], other[None], 1)
    for _ in range(3):
        _same(_forward(pkg, pc[None], other[None], 1), ref, "repeat")


def test_gradients_agree_between_paths(pkg):
    a0, b0 = _uniform(20000, 40), _uniform(15000, 41) * 1.3
    grads = []
    for grid in (1, 0):
        a = a0.clone()[None].requires_grad_(True)
        b = b0.clone()[None].requires_grad_(True)
        with pkg._lib.option_scope({"chamfer_grid": grid}):
            d1, d2, _, _ = pkg.chamfer.chamfer_3DDist()(a, b)
        ((d1 * 0.3).sum() + d2.sum()).backward()
        grads.append((a.grad.clone(), b.grad.clone()))
    for u, v in zip(*grads):
        torch.testing.assert_close(u, v, rtol=1e-5, atol=1e-6)


def test_flow_loss_is_identical(pkg):
    class Flow(torch.nn.Module):   # a stand-in flow field: the Chamfer terms are what differs between paths
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.tensor([[0.01, -0.02, 0.005]], device="cuda"))

        def flow(self, pc, time):
            return {"flow_forward": pc * 0.01 + self.w, "flow_backward": -pc * 0.02 - self.w}

    pc = _scan(pkg, 4) / 80.0
    g = torch.Generator(device="cuda").manual_seed(42)
    pcf = pc + 0.002 * torch.randn(pc.shape, device="cuda", generator=g)
    pcb = (pc - 0.001)[::2].contiguous()
    vals = []
    for grid in (1, 0):
        m = Flow()
        with pkg._lib.option_scope({"chamfer_grid": grid}):
            v = pkg.losses.flow_loss(m, pc, torch.tensor([[0.5]], device="cuda"), pcf, pcb)
        v.backward()
        vals.append((v.detach().clone(), m.w.grad.clone()))
    assert torch.equal(vals[0][0].view(torch.int32), vals[1][0].view(torch.int32))
    torch.testing.assert_close(vals[0][1], vals[1][1], rtol=1e-4, atol=1e-6)


# ----------------------------------------------------------------------------------------------- 9. selection
def test_automatic_selection_equals_both_paths_and_the_option_is_restored(pkg):
    L = pkg._lib.lib()
    before = L.nvsf_get_option(b"chamfer_grid")
    assert before == -1                                    # automatic by default
    for n in (4096, 16384):                                # 2^24 pairs: brute force; 2^28: grid
        a, b = _uniform(n, n + 3), _uniform(n, n + 4)
        auto = _forward(pkg, a[None], b[None], -1)
        _same(auto, both(pkg, a, b, f"auto {n}"), f"auto {n}")
    with pytest.raises(pkg._lib.NvsfError):
        with pkg._lib.option_scope({"chamfer_grid": 2}):
            pass
    assert L.nvsf_set_option(b"chamfer_grid", -2) == -1
    assert L.nvsf_get_option(b"chamfer_grid") == before


# ----------------------------------------------------------------------------------------------- 10. meters
def _frame(pkg, seed):
    """(depth, image, images_lidar) of a scan and a ground truth at a nearby range"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    d = _scan_depth(seed, pkg=pkg)
    prob = 0.5 + 0.5 * (d > 0).float() * torch.rand(d.shape, device="cuda", generator=g).clamp(min=0.02)
    inten = torch.rand(d.shape, device="cuda", generator=g)
    dt = (d + 0.03 * torch.randn(d.shape, device="cuda", generator=g)).clamp(min=0)
    mask = ((dt > 0) & (torch.rand(d.shape, device="cuda", generator=g) > 0.05)).float()
    gt = torch.stack([mask, inten, dt], -1)
    return d, torch.stack([prob, inten], -1), gt


def test_lidar_meter_row_is_identical(pkg):
    rows = []
    for grid in (1, 0):
        meter = pkg.metrics.LidarMeter(H_FULL, W_FULL, LIDAR_K, LIDAR_K_HOZ, 1.0)
        with pkg._lib.option_scope({"chamfer_grid": grid}):
            rows.append(meter.update(*_frame(pkg, 50)).clone())
    assert torch.equal(rows[0].view(torch.int32), rows[1].view(torch.int32))
    assert rows[0][-1] > 50000 and math.isfinite(float(rows[0][11]))


def test_points_meter_equals_lidar_meter_columns(pkg):
    M = pkg.metrics
    d, im, gt = _frame(pkg, 51)
    lm = M.LidarMeter(H_FULL, W_FULL, LIDAR_K, LIDAR_K_HOZ, 1.0)
    lrow = lm.update(d, im, gt)
    pp, pc = M.lidar_points(d, LIDAR_K, LIDAR_K_HOZ, raydrop=im[..., 0])
    gp, gc = M.lidar_points(gt[..., 2], LIDAR_K, LIDAR_K_HOZ, raydrop=gt[..., 0])
    pm = M.PointsMeter()
    row = pm.update(pp, gp, pc, gc)
    cols = [M.LIDAR_METRICS.index(k) for k in M.POINTS_METRICS]
    assert torch.equal(row.view(torch.int32), lrow[cols].view(torch.int32))
    assert pm.frame_results().shape == (1, 4) and set(pm.summary()) == set(M.POINTS_METRICS)
    pm.reset()
    assert pm.frame_results().shape == (0, 4)


def test_points_meter_raw_cloud_vs_oracle(pkg):
    g = torch.Generator(device="cuda").manual_seed(52)
    pred = torch.cat([_scan(pkg, 60), _scan(pkg, 61) + 0.3, _scan(pkg, 62) - 0.2, _scan(pkg, 63) * 1.1])[:200000]
    gt = pred + 0.05 * torch.randn(pred.shape, device="cuda", generator=g)
    gt4 = torch.cat([gt, torch.rand(gt.shape[0], 1, device="cuda", generator=g)], 1)   # xyz + intensity
    row = pkg.metrics.PointsMeter().update(pred, gt4).cpu().numpy().astype(np.float64)
    ch, fs = MO.chamfer(pred.cpu().numpy(), gt.cpu().numpy(), 0.05)
    assert row[0] == pytest.approx(ch, rel=1e-5)
    assert abs(row[1] - fs) <= 2.0 / pred.shape[0]
    assert row[2] == pred.shape[0] == 200000 and row[3] == gt.shape[0]


def test_points_meter_empty_clouds_and_device_counts(pkg):
    M = pkg.metrics
    pm = M.PointsMeter(fscore_threshold=0.01)
    a, b = _uniform(3000, 70), _uniform(2000, 71)
    r = pm.update(a[:0], b).cpu().tolist()
    assert r == [math.inf, 0.0, 0.0, 2000.0]
    r = pm.update(a, b, gt_count=torch.zeros((), dtype=torch.int32, device="cuda")).cpu().tolist()
    assert r == [math.inf, 0.0, 3000.0, 0.0]
    n = torch.tensor(1234, dtype=torch.int32, device="cuda")
    m = torch.tensor([777], dtype=torch.int64, device="cuda")
    r1 = pm.update(a, b, n, m)
    r2 = pm.update(a[:1234].clone(), b[:777].clone())
    assert torch.equal(r1.view(torch.int32), r2.view(torch.int32)) and r1[2] == 1234 and r1[3] == 777
    with pytest.raises(pkg._lib.NvsfError):
        pm.update(a.cpu(), b)
    with pytest.raises(pkg._lib.NvsfError):
        pm.update(a[:, :2], b)
    with pytest.raises(pkg._lib.NvsfError):
        pm.update(a, b, 5)


def test_points_meter_update_in_a_cuda_graph(pkg):
    pm = pkg.metrics.PointsMeter()
    a, b = _scan(pkg, 80), _scan(pkg, 81)
    na = torch.tensor(a.shape[0] - 100, dtype=torch.int32, device="cuda")
    nb = torch.tensor(b.shape[0], dtype=torch.int32, device="cuda")
    eager = pm.update(a, b, na, nb).clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pm.update(a, b, na, nb)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        row = pm.update(a, b, na, nb)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(row.view(torch.int32), eager.view(torch.int32))
    na.fill_(5000)
    graph.replay()
    want = pm.update(a[:5000].clone(), b)
    torch.cuda.synchronize()
    assert torch.equal(row.view(torch.int32), want.view(torch.int32))
