"""Evaluation on the device (metrics.py, csrc/eval.cu, C ABI Part 6): range image -> point cloud, Chamfer with
device-side counts, and the LiDAR / camera meters, against the float64 oracle (oracle/metrics_oracle.py).

CPU: the oracle itself (SSIM against a per-window loop, hand cases, directions against the pinned ray oracle)
and the distributed summary over gloo.  GPU: points bit-exact against get_lidar_rays, counted Chamfer
bit-identical to chamfer_3DDist, every metric against the oracle (counts and medians exact, RMSE / PSNR /
Chamfer 1e-5 relative, SSIM 1e-4 absolute), ragged sizes, repeatability, end to end from render_frame, and
capture in a CUDA graph."""
import importlib
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import GOLDEN
from oracle import metrics_oracle as MO

gpu = pytest.mark.gpu
LIDAR_K, LIDAR_K_HOZ = (2.0, 26.9), (180.0, 360.0)   # tests/golden/rays_ref.npz lidar_K / lidar_K_hoz
H_FULL, W_FULL = 66, 1030


def _pkg():
    return importlib.import_module("selfsupervised-nvsf_b200")


# ---------------------------------------------------------------------------------------------- CPU: the oracle
def _ssim_windows(x, y, R):
    """SSIM as a direct float64 loop over the 7x7 windows that lie inside the image."""
    H, W = x.shape
    C1, C2 = (0.01 * R) ** 2, (0.03 * R) ** 2
    vals = []
    for a in range(H - 6):
        for b in range(W - 6):
            wx, wy = x[a:a + 7, b:b + 7].astype(np.float64), y[a:a + 7, b:b + 7].astype(np.float64)
            mx, my = wx.mean(), wy.mean()
            vx, vy = ((wx - mx) ** 2).sum() / 48, ((wy - my) ** 2).sum() / 48
            vxy = ((wx - mx) * (wy - my)).sum() / 48
            vals.append((2 * mx * my + C1) * (2 * vxy + C2) / ((mx * mx + my * my + C1) * (vx + vy + C2)))
    return float(np.mean(vals))


@pytest.mark.parametrize("shape,R", [((12, 15), 1.0), ((9, 20), 80.0), ((7, 7), 3.0)])
def test_oracle_ssim_is_the_window_loop(shape, R):
    rng = np.random.default_rng(shape[0])
    x = rng.random(shape) * R
    y = x + rng.normal(0, 0.1 * R, shape)
    assert MO.ssim(x, y, R) == pytest.approx(_ssim_windows(x, y, R), rel=1e-9, abs=1e-12)
    assert MO.ssim(x, x, R) == pytest.approx(1.0, abs=1e-12)
    assert math.isnan(MO.ssim(x[:6], y[:6], R))


def _frame(gt_depth, pred_depth, pred_raydrop=None, gt_mask=None):
    W = len(gt_depth)
    gt = np.zeros((1, W, 3), np.float32)
    gt[0, :, 0] = 1.0 if gt_mask is None else gt_mask
    gt[0, :, 1] = 0.5
    gt[0, :, 2] = gt_depth
    im = np.zeros((1, W, 2), np.float32)
    im[0, :, 0] = 1.0 if pred_raydrop is None else pred_raydrop
    im[0, :, 1] = 0.5
    return np.asarray(pred_depth, np.float32).reshape(1, W), im, gt


def test_oracle_hand_cases():
    # |G - P| = 0, 1, 2 (odd count) and 0, 1, 2, 3 (even count)
    r3 = MO.lidar_metrics(*_frame([1, 2, 3], [1, 1, 1]), LIDAR_K, LIDAR_K_HOZ, 1.0)
    assert r3["depth_medae"] == 1.0 and r3["depth_rmse"] == pytest.approx(math.sqrt(5 / 3))
    r4 = MO.lidar_metrics(*_frame([1, 2, 3, 4], [1, 1, 1, 1]), LIDAR_K, LIDAR_K_HOZ, 1.0)
    assert r4["depth_medae"] == 1.5 and r4["depth_rmse"] == pytest.approx(math.sqrt(3.5))
    assert r4["depth_psnr"] == pytest.approx(10 * math.log10(80.0 ** 2 / 3.5))
    assert r4["intensity_rmse"] == 0.0 and r4["intensity_psnr"] == math.inf and r4["intensity_medae"] == 0.0
    assert r4["raydrop_acc"] == 1.0 and r4["raydrop_f1"] == 1.0 and r4["raydrop_rmse"] == 0.0
    assert r4["points_pred"] == 4 and r4["points_gt"] == 4
    # nothing returns, nothing predicted: F1's precision + recall = 0 -> 0; both clouds empty
    r0 = MO.lidar_metrics(*_frame([5, 6], [5, 6], pred_raydrop=[0.2, 0.4], gt_mask=[0, 0]), LIDAR_K, LIDAR_K_HOZ, 1.0)
    assert r0["raydrop_f1"] == 0.0 and r0["raydrop_acc"] == 1.0
    assert r0["chamfer"] == math.inf and r0["fscore"] == 0.0 and r0["points_pred"] == 0 and r0["points_gt"] == 0
    # one empty cloud
    pts = np.ones((3, 3))
    assert MO.chamfer(pts[:0], pts) == (math.inf, 0.0) and MO.chamfer(pts, pts[:0]) == (math.inf, 0.0)
    assert MO.fscore(0.0, 0.0) == 0.0 and MO.fscore(1.0, 0.5) == pytest.approx(2 / 3)
    assert MO.psnr(0.0, 80.0) == math.inf and MO.psnr(1.0, 1.0) == 0.0
    # identical clouds: chamfer 0, fscore 1
    assert MO.chamfer(pts + np.arange(3)[:, None], pts + np.arange(3)[:, None]) == (0.0, 1.0)


def test_oracle_directions_are_the_ray_oracle_at_identity():
    from oracle import scene_oracle
    g = np.load(os.path.join(GOLDEN, "rays_ref.npz"))
    _, d = scene_oracle.get_lidar_rays(np.eye(4, dtype=np.float32), g["lidar_K"], g["lidar_K_hoz"], H_FULL, W_FULL)
    np.testing.assert_allclose(MO.lidar_dirs(H_FULL, W_FULL, g["lidar_K"], g["lidar_K_hoz"]), d, rtol=0, atol=1e-6)


# ---------------------------------------------------------------------------------------------- CPU: gloo world 2
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rows():
    rows = torch.from_numpy(np.random.default_rng(5).random((7, len(_pkg().metrics.LIDAR_METRICS)), np.float32))
    rows[3, 2] = float("inf")      # a frame with a perfect depth: PSNR +inf
    return rows


def _worker_summary(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    M = _pkg().metrics
    res = M.summarize(_rows()[rank::world], M.LIDAR_METRICS)
    np.save(os.path.join(out_dir, f"sum{rank}.npy"), np.array([res], dtype=object), allow_pickle=True)
    dist.destroy_process_group()


def test_summary_all_reduces_over_ranks_gloo_world2(tmp_path):
    M = _pkg().metrics
    rows = _rows()
    one = M.summarize(rows, M.LIDAR_METRICS)
    want = rows.double().mean(0).tolist()
    assert [one[k] for k in M.LIDAR_METRICS] == pytest.approx(want, rel=1e-12)
    assert one["depth_psnr"] == math.inf
    mp.spawn(_worker_summary, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        got = np.load(tmp_path / f"sum{r}.npy", allow_pickle=True)[0]
        assert list(got) == list(M.LIDAR_METRICS)
        assert [got[k] for k in M.LIDAR_METRICS] == pytest.approx([one[k] for k in M.LIDAR_METRICS], rel=1e-12)
    empty = M.summarize(rows[:0], M.LIDAR_METRICS)
    assert all(math.isnan(v) for v in empty.values())


# ---------------------------------------------------------------------------------------------- GPU
def _synthetic_frame(H, W, seed, scale=1.0, drop_all=False):
    """(depth_lidar [H,W], image_lidar [H,W,2], images_lidar [H,W,3]) on the device: a ground-truth range image
    with ~15 % dropped rays and a prediction that is near it, with its own ray-drop errors."""
    g = torch.Generator().manual_seed(seed)
    depth_m = 2.0 + 70.0 * torch.rand(H, W, generator=g)
    mask = (torch.rand(H, W, generator=g) > 0.15).float()
    inten = torch.rand(H, W, generator=g)
    gt = torch.stack([mask, inten, depth_m * scale], -1)
    pred_depth = (depth_m + 0.3 * torch.randn(H, W, generator=g)).clamp_min(0.0) * scale
    prob = (0.75 * mask + 0.5 * torch.rand(H, W, generator=g)).clamp(0, 1)
    if drop_all:
        prob.zero_()
        gt[..., 0] = 0.0
    pred_int = (inten + 0.05 * torch.randn(H, W, generator=g)).clamp(0, 1)
    image = torch.stack([prob, pred_int], -1)
    return pred_depth.cuda(), image.cuda(), gt.cuda()


def _check_row(row, want, names, skip=()):
    got = dict(zip(names, row.cpu().numpy().astype(np.float64).tolist()))
    exact = ("depth_medae", "intensity_medae", "points_pred", "points_gt")
    rel5 = ("depth_rmse", "depth_psnr", "intensity_rmse", "intensity_psnr", "raydrop_rmse", "chamfer", "psnr")
    for k in names:
        if k in skip:
            continue
        a, b = got[k], want[k]
        if math.isnan(b) or math.isinf(b):
            assert (math.isnan(a) and math.isnan(b)) or a == b, (k, a, b)
        elif k in exact:
            assert a == np.float32(b), (k, a, b)
        elif k in rel5:
            assert a == pytest.approx(b, rel=1e-5), (k, a, b)
        elif k.endswith("ssim"):
            assert abs(a - b) <= 1e-4, (k, a, b)
        elif k == "fscore":       # a squared distance within rounding of the threshold may flip one point
            assert abs(a - b) <= 2.0 / max(got["points_pred"], got["points_gt"], 1), (k, a, b)
        else:                     # ratios of exact counts, stored as fp32
            assert a == pytest.approx(b, rel=1e-6), (k, a, b)
    return got


def _dirty(nfloats):
    """Leave a NaN-filled block of `nfloats` floats in the caching allocator, so that the next allocation of that
    size (the points tensor) starts dirty and rows past the count must be written to read as zero."""
    torch.full((nfloats,), float("nan"), device="cuda")


@gpu
@pytest.mark.parametrize("H,W", [(H_FULL, W_FULL), (13, 37), (1, 1), (7, 1031)])
def test_lidar_points_bit_exact_vs_rays(H, W):
    pkg = _pkg()
    g = torch.Generator(device="cuda").manual_seed(H * W)
    depth = 80.0 * torch.rand(H, W, device="cuda", generator=g)
    depth[:, ::7] = 0.0
    raydrop = torch.rand(H, W, device="cuda", generator=g)
    inten = torch.rand(H, W, device="cuda", generator=g)
    scale = 0.37
    rays = pkg.rays.get_lidar_rays(torch.eye(4, device="cuda")[None], LIDAR_K, LIDAR_K_HOZ, H, W, -1)["rays_d"][0]
    for rd, it in ((None, None), (raydrop, inten), (raydrop, None)):
        _dirty(H * W * (3 if it is None else 4))
        pts, count = pkg.metrics.lidar_points(depth, LIDAR_K, LIDAR_K_HOZ, scale, raydrop=rd, intensity=it)
        masked = (depth * (rd > 0.5).float() if rd is not None else depth).reshape(-1)
        keep = torch.nonzero(masked != 0).reshape(-1)
        r = masked / torch.full_like(masked, scale)
        want = rays[keep] * r[keep, None]
        assert count.dtype == torch.int32 and count.device.type == "cuda" and int(count) == keep.numel()
        assert pts.shape == (H * W, 3 if it is None else 4)
        assert torch.equal(pts[:keep.numel(), :3], want)
        if it is not None:
            assert torch.equal(pts[:keep.numel(), 3], it.reshape(-1)[keep])
        assert not pts[keep.numel():].any()
    # every pixel dropped
    _dirty(H * W * 3)
    pts, count = pkg.metrics.lidar_points(depth, LIDAR_K, LIDAR_K_HOZ, scale, raydrop=torch.zeros_like(depth))
    assert int(count) == 0 and not pts.any()


@gpu
def test_counted_chamfer_is_chamfer_on_trimmed_clouds():
    pkg = _pkg()
    L = pkg._lib.lib()
    P = pkg._lib.ptr
    g = torch.Generator(device="cuda").manual_seed(0)
    for n, m, cap_n, cap_m in ((3000, 2500, 4096, 5000), (1, 700, 1, 1024), (5000, 5000, 5000, 5000),
                               (0, 300, 64, 512), (40, 0, 40, 8)):
        a = torch.randn(cap_n, 3, device="cuda", generator=g)
        b = torch.randn(cap_m, 3, device="cuda", generator=g) * 1.1
        cnt = torch.tensor([n, m], dtype=torch.int32, device="cuda")
        d1 = torch.empty(cap_n, device="cuda"); d2 = torch.empty(cap_m, device="cuda")
        i1 = torch.empty(cap_n, dtype=torch.int32, device="cuda"); i2 = torch.empty(cap_m, dtype=torch.int32, device="cuda")
        wb = L.nvsf_chamfer_workspace_bytes(1, cap_n, cap_m)
        ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
        assert L.nvsf_chamfer_forward_counted(P(a), P(b), cap_n, cap_m, P(cnt), P(cnt[1:]), P(d1), P(d2), P(i1), P(i2),
                                              P(ws), wb, None) == 0
        if n and m:
            e1, e2, f1, f2 = pkg.chamfer.chamfer_3DDist()(a[None, :n], b[None, :m])
            assert torch.equal(d1[:n], e1[0]) and torch.equal(d2[:m], e2[0])
            assert torch.equal(i1[:n], f1[0]) and torch.equal(i2[:m], f2[0])
        else:   # the other cloud is empty: +inf / -1
            assert torch.isinf(d1[:n]).all() and torch.isinf(d2[:m]).all()
            assert (i1[:n] == -1).all() and (i2[:m] == -1).all()
        assert not d1[n:].any() and not d2[m:].any() and (i1[n:] == -1).all() and (i2[m:] == -1).all()
    # argument checks: non-zero status, nothing launched
    assert L.nvsf_chamfer_forward_counted(P(a), P(b), 0, cap_m, P(cnt), P(cnt), P(d1), P(d2), P(i1), P(i2), P(ws), wb,
                                          None) != 0
    assert L.nvsf_chamfer_forward_counted(P(a), None, cap_n, cap_m, P(cnt), P(cnt), P(d1), P(d2), P(i1), P(i2), P(ws),
                                          wb, None) != 0
    assert L.nvsf_chamfer_forward_counted(P(a), P(b), cap_n, cap_m, P(cnt), P(cnt), P(d1), P(d2), P(i1), P(i2), P(ws),
                                          wb - 1, None) == -2


@gpu
@pytest.mark.parametrize("H,W,drop_all", [(H_FULL, W_FULL, False), (13, 37, False), (1, 1, False),
                                          (9, 1031, True)])
def test_lidar_meter_vs_oracle(H, W, drop_all):
    pkg = _pkg()
    scale = 0.25
    d, im, gt = _synthetic_frame(H, W, seed=H + W, scale=scale, drop_all=drop_all)
    meter = pkg.metrics.LidarMeter(H, W, LIDAR_K, LIDAR_K_HOZ, scale)
    row = meter.update(d, im, gt)
    want = MO.lidar_metrics(d.cpu().numpy(), im.cpu().numpy(), gt.cpu().numpy(), LIDAR_K, LIDAR_K_HOZ, scale)
    # with every ray dropped both SSIM images are constant: data range 0, SSIM 0/0 (skimage's too)
    got = _check_row(row, want, pkg.metrics.LIDAR_METRICS, skip=("depth_ssim", "intensity_ssim") if drop_all else ())
    if drop_all:
        assert got["points_pred"] == 0 and got["points_gt"] == 0 and got["chamfer"] == math.inf
    if H < 7:
        assert math.isnan(got["depth_ssim"]) and math.isnan(got["intensity_ssim"])
    # the same inputs give the same row, bit for bit
    again = meter.update(d, im, gt)
    assert torch.equal(again.view(torch.int32), row.view(torch.int32))
    assert meter.frame_results().shape == (2, len(pkg.metrics.LIDAR_METRICS))


@gpu
def test_lidar_meter_summary_and_checks():
    pkg = _pkg()
    M = pkg.metrics
    meter = M.LidarMeter(H_FULL, W_FULL, LIDAR_K, LIDAR_K_HOZ, 1.0)
    wants = []
    for seed in (1, 2, 3):
        d, im, gt = _synthetic_frame(H_FULL, W_FULL, seed)
        meter.update(d, im, gt)
        wants.append(MO.lidar_metrics(d.cpu().numpy(), im.cpu().numpy(), gt.cpu().numpy(), LIDAR_K, LIDAR_K_HOZ, 1.0))
    s = meter.summary()
    for k in M.LIDAR_METRICS:
        assert s[k] == pytest.approx(np.mean([w[k] for w in wants]), rel=1e-4, abs=1e-4), k
    with pytest.raises(pkg._lib.NvsfError):
        meter.update(d[:10], im, gt)
    with pytest.raises(pkg._lib.NvsfError):
        meter.update(d.cpu(), im, gt)
    L = pkg._lib.lib()
    row = torch.empty(15, device="cuda")
    ws = torch.empty(L.nvsf_eval_lidar_workspace_bytes(H_FULL, W_FULL), dtype=torch.uint8, device="cuda")
    P = pkg._lib.ptr
    args = [P(d), P(im), P(gt), H_FULL, W_FULL, 2.0, 26.9, 360.0, 1.0, 80.0, 0.05, P(row), P(ws), ws.numel(), None]
    for i, bad in ((0, None), (3, 0), (8, 0.0), (9, 0.0), (12, None)):
        a = list(args)
        a[i] = bad
        assert L.nvsf_eval_lidar(*a) == -1
    a = list(args)
    a[13] = ws.numel() - 1
    assert L.nvsf_eval_lidar(*a) == -2
    assert L.nvsf_eval_lidar_workspace_bytes(0, 5) == 0 and L.nvsf_lidar_points_workspace_bytes(1 << 14, 1 << 13) == 0
    torch.cuda.synchronize()


@gpu
@pytest.mark.parametrize("H,W", [(120, 200), (7, 9), (5, 5)])
def test_camera_meter_vs_oracle(H, W):
    pkg = _pkg()
    g = torch.Generator(device="cuda").manual_seed(H)
    gt = torch.rand(H, W, 3, device="cuda", generator=g)
    pred = (gt + 0.05 * torch.randn(H, W, 3, device="cuda", generator=g)).clamp(0, 1)
    meter = pkg.metrics.CameraMeter(H, W)
    row = meter.update(pred, gt)
    want = MO.camera_metrics(pred.cpu().numpy(), gt.cpu().numpy())
    _check_row(row, want, pkg.metrics.CAMERA_METRICS)
    assert meter.update(gt, gt)[0].item() == math.inf
    if H >= 7:
        assert meter.frame_results()[1, 1].item() == pytest.approx(1.0, abs=1e-6)


@gpu
def test_end_to_end_render_frame_scored_by_lidar_meter():
    """Two full 66 x 1030 LiDAR frames of a synthetic model, at two poses and times: one is the prediction,
    the other supplies the ground truth; the meter's row equals the oracle on the same outputs copied back.
    The synthetic model's untrained ray-drop head renders probabilities of about 0.1-0.4 everywhere, which would
    drop every ray at the 0.5 threshold; the channel is shifted by +0.3 so that both clouds keep part of the
    frame.  Depth and intensity are scored as rendered."""
    import field_cases as FC
    pkg = _pkg()
    S = FC.S
    model = pkg.NeRFNetwork(time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND,
                            min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    model.load_flat_params(FC.oracle_params())
    model.eval()
    g = np.load(os.path.join(GOLDEN, "rays_ref.npz"))
    pose_a = torch.from_numpy(g["pose_a"]).clone()
    pose_a[:3, 3] *= 0.2
    pose_b = pose_a.clone()
    pose_b[:3, 3] += 0.01
    fa = model.render_frame(pose_a, g["lidar_K"], H_FULL, W_FULL, 0.3, cal_lidar_color=True,
                            intrinsics_hoz=g["lidar_K_hoz"])
    fb = model.render_frame(pose_b, g["lidar_K"], H_FULL, W_FULL, 0.5, cal_lidar_color=True,
                            intrinsics_hoz=g["lidar_K_hoz"])
    for f in (fa, fb):
        f["image_lidar"][..., 0] += 0.3
    gt = torch.stack([(fb["image_lidar"][..., 0] > 0.5).float(), fb["image_lidar"][..., 1], fb["depth_lidar"]], -1)
    meter = pkg.metrics.LidarMeter(H_FULL, W_FULL, g["lidar_K"], g["lidar_K_hoz"], S.SCALE)
    row = meter.update(fa["depth_lidar"], fa["image_lidar"], gt)
    want = MO.lidar_metrics(fa["depth_lidar"].cpu().numpy(), fa["image_lidar"].cpu().numpy(), gt.cpu().numpy(),
                            g["lidar_K"], g["lidar_K_hoz"], S.SCALE)
    got = _check_row(row, want, pkg.metrics.LIDAR_METRICS)
    assert 0 < got["points_pred"] < H_FULL * W_FULL and 0 < got["points_gt"] < H_FULL * W_FULL
    # the synthesized scan itself: lidar_points of the render composes with the meter's predicted cloud
    pts, count = pkg.metrics.lidar_points(fa["depth_lidar"], g["lidar_K"], g["lidar_K_hoz"], S.SCALE,
                                          raydrop=fa["image_lidar"][..., 0], intensity=fa["image_lidar"][..., 1])
    assert int(count) == got["points_pred"] and pts.shape == (H_FULL * W_FULL, 4)


@gpu
def test_lidar_meter_update_in_a_cuda_graph():
    """update() captured in a CUDA graph and replayed gives the eager row: it neither synchronises with the host
    nor allocates outside the graph's pool (capture fails on either)."""
    pkg = _pkg()
    meter = pkg.metrics.LidarMeter(H_FULL, W_FULL, LIDAR_K, LIDAR_K_HOZ, 1.0)
    f1, f2 = _synthetic_frame(H_FULL, W_FULL, 11), _synthetic_frame(H_FULL, W_FULL, 12)
    eager1 = meter.update(*f1).clone()
    eager2 = meter.update(*f2).clone()
    bufs = [t.clone() for t in f1]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        meter.update(*bufs)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        row = meter.update(*bufs)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(row.view(torch.int32), eager1.view(torch.int32))
    for b, t in zip(bufs, f2):
        b.copy_(t)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(row.view(torch.int32), eager2.view(torch.int32))
