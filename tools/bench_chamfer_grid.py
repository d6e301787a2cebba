"""Chamfer forward on the B200: brute-force scan vs the uniform-grid path (csrc/chamfer.cu), and what the grid path
changes for its callers.

Per workload (n query / m target points, both directions as nvsf_chamfer_forward computes them):
  - the whole C ABI call with "chamfer_grid" forced off (brute), forced on (grid, grid build included) and
    automatic: CUDA events, launches queued behind a spin kernel, median over the calls;
  - the kernels alone, from a torch.profiler run of its own: grid build (k_grid_bbox .. k_grid_scatter), grid
    search (k_grid_nn), the brute-force tiles (k_chamfer_nn, or the crowded-cloud k_chamfer_nn_crowded);
  - a check that the three paths give bit-identical dist / idx.
Workloads: uniform cubes at n = m from 4 K to 1 M points, a synthetic 66 x 1030 LiDAR scan against a displaced copy
(flow_loss) and a noisy copy (evaluation), 16 posed scans accumulated (~1 M points) against a noisy copy, and the
adversarial clouds (a tight cluster plus one far outlier; all points identical).  Then LidarMeter.update per frame
and flow_loss forward + backward at a full scan, brute force (before) against automatic (after).
Brute-force calls at 1 M points run once after one warm-up call.  Writes JSON lines to --out and prints them; the
first line names the card and its power limit.  Runs on the GPU only (no fallback)."""
import argparse
import importlib
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("selfsupervised-nvsf_b200")
L = pkg._lib.lib()
P = pkg._lib.ptr
LIDAR_K, LIDAR_K_HOZ = (2.0, 26.9), (180.0, 360.0)
MODES = {"brute": 0, "grid": 1, "auto": -1}


def gpu_time(fn, iters=10, warmup=3):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(iters):
        torch.cuda.synchronize()
        torch.cuda._sleep(400000)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def kernel_ms(fn, calls=3):
    """device time per call by kernel group, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    groups = {}
    for e in prof.key_averages():
        name = e.key
        if "k_grid_nn" in name:
            g = "search"
        elif "k_grid_" in name or name.startswith("Memset"):
            g = "build"
        elif "crowded" in name:
            g = "crowded_brute"
        elif "k_chamfer_nn" in name:
            g = "brute"
        elif "unpack" in name:
            g = "unpack"
        else:
            continue
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        groups[g] = groups.get(g, 0.0) + t / 1e3 / calls
    return {k: round(v, 4) for k, v in groups.items()}


def scan_depth(seed, H=66, W=1030):
    """the street-like range image of tests/test_chamfer_grid_gpu.py"""
    dirs = pkg.rays.get_lidar_rays(torch.eye(4, device="cuda")[None], LIDAR_K, LIDAR_K_HOZ, H, W, -1)["rays_d"][0]
    dx, dy, dz = dirs[:, 0], dirs[:, 1], dirs[:, 2]
    inf = torch.full_like(dx, math.inf)
    t = torch.where(dz < -1e-6, -1.7 / dz, inf)
    for d, half in ((dx, 20.0), (dy, 12.0)):
        t = torch.minimum(t, torch.where(d.abs() > 1e-6, half / d.abs(), inf))
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(6):
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


def scan(seed):
    pts, cnt = pkg.metrics.lidar_points(scan_depth(seed), LIDAR_K, LIDAR_K_HOZ)
    return pts[:int(cnt)].contiguous()


def workloads(big):
    g = torch.Generator(device="cuda").manual_seed(0)
    sizes = (4096, 8192, 16384, 32768, 65536, 262144, 1 << 20) if big else (4096, 16384, 65536)
    for n in sizes:
        yield f"uniform_{n}", torch.rand(n, 3, device="cuda", generator=g), torch.rand(n, 3, device="cuda", generator=g)
    pc = scan(1)
    yield "lidar_displaced", pc, pc + torch.tensor([0.05, -0.02, 0.0], device="cuda")
    yield "lidar_noisy", pc, pc + 0.02 * torch.randn(pc.shape, device="cuda", generator=g)
    if big:
        scans = []
        for k in range(16):
            th = 0.05 * k
            R = torch.tensor([[math.cos(th), -math.sin(th), 0.0], [math.sin(th), math.cos(th), 0.0], [0, 0, 1.0]],
                             device="cuda")
            scans.append(scan(100 + k) @ R.T + torch.tensor([1.5 * k, 0.2 * k, 0.0], device="cuda"))
        acc = torch.cat(scans).contiguous()
        yield "accumulated_16_scans", acc, acc + 0.02 * torch.randn(acc.shape, device="cuda", generator=g)
    n = 65536
    cl = torch.randn(n, 3, device="cuda", generator=g) * 1e-3
    cl[-1] = torch.tensor([1e4, -3e3, 50.0], device="cuda")
    yield "cluster_plus_outlier", cl, torch.randn(n, 3, device="cuda", generator=g) * 1e-3
    yield "all_identical", torch.full((n, 3), 0.25, device="cuda"), torch.rand(n, 3, device="cuda", generator=g)


def bench_workload(name, a, b):
    n, m = a.shape[0], b.shape[0]
    d1, d2 = torch.empty(n, device="cuda"), torch.empty(m, device="cuda")
    i1, i2 = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(m, dtype=torch.int32, device="cuda")
    wb = L.nvsf_chamfer_workspace_bytes(1, n, m)
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")

    def call():
        assert L.nvsf_chamfer_forward(P(a), P(b), 1, n, m, P(d1), P(d2), P(i1), P(i2), P(ws), wb,
                                      pkg._lib.stream_ptr()) == 0

    row = {"workload": name, "n": n, "m": m, "pairs": 2 * n * m}
    outs = {}
    for mode, v in MODES.items():
        slow = mode == "brute" and n * m >= (1 << 36)
        with pkg._lib.option_scope({"chamfer_grid": v}):
            row[f"{mode}_ms"] = round(gpu_time(call, iters=1 if slow else 10, warmup=1 if slow else 3), 4)
            if not slow:
                row[f"{mode}_kernels_ms"] = kernel_ms(call)
            call()
        torch.cuda.synchronize()
        outs[mode] = [t.clone() for t in (d1.view(torch.int32), d2.view(torch.int32), i1, i2)]
    row["identical"] = all(torch.equal(x, y) for mode in ("grid", "auto") for x, y in zip(outs[mode], outs["brute"]))
    row["grid_speedup"] = round(row["brute_ms"] / row["grid_ms"], 2)
    return row


def bench_meter():
    d = scan_depth(7)
    g = torch.Generator(device="cuda").manual_seed(8)
    prob = 0.5 + 0.5 * (d > 0).float() * torch.rand(d.shape, device="cuda", generator=g).clamp(min=0.02)
    inten = torch.rand(d.shape, device="cuda", generator=g)
    dt = (d + 0.03 * torch.randn(d.shape, device="cuda", generator=g)).clamp(min=0)
    gt = torch.stack([(dt > 0).float(), inten, dt], -1)
    im = torch.stack([prob, inten], -1)
    meter = pkg.metrics.LidarMeter(66, 1030, LIDAR_K, LIDAR_K_HOZ, 1.0)
    row = {"workload": "LidarMeter.update", "H": 66, "W": 1030}
    rows = {}
    for mode in ("brute", "auto"):
        with pkg._lib.option_scope({"chamfer_grid": MODES[mode]}):
            row[f"{mode}_ms"] = round(gpu_time(lambda: meter.update(d, im, gt), iters=20), 4)
            rows[mode] = meter.update(d, im, gt).clone()
        meter.reset()
    row["points"] = [int(rows["auto"][13]), int(rows["auto"][14])]
    row["identical"] = torch.equal(rows["brute"].view(torch.int32), rows["auto"].view(torch.int32))
    row["speedup"] = round(row["brute_ms"] / row["auto_ms"], 2)
    return row


def bench_flow_loss():
    from oracle import field_init
    from oracle.field_oracle import FieldConfig
    S = importlib.import_module("selfsupervised-nvsf_b200.synth")
    kw = dict(bound=S.BOUND, num_frames=S.NUM_FRAMES, time_resolution=S.TIME_RESOLUTION, min_near=S.MIN_NEAR,
              min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    model = pkg.NeRFNetwork(**kw).train()
    model.load_flat_params(field_init.make_params(FieldConfig(**kw), seed=0, style="trained"))
    pc = (scan(9) / 80.0).contiguous()                      # normalised coordinates, inside the bound
    g = torch.Generator(device="cuda").manual_seed(10)
    pcf = (pc + 0.002 * torch.randn(pc.shape, device="cuda", generator=g)).contiguous()
    pcb = (pc - 0.001 + 0.002 * torch.randn(pc.shape, device="cuda", generator=g)).contiguous()
    t = torch.tensor([[0.4]], device="cuda")

    def step():
        model.zero_grad(set_to_none=True)
        pkg.losses.flow_loss(model, pc, t, pcf, pcb).backward()

    row = {"workload": "flow_loss fwd+bwd", "points": pc.shape[0], "neighbours": 2}
    vals = {}
    for mode in ("brute", "auto"):
        # set without option_scope: the model's backward takes the option lock from the autograd thread
        assert L.nvsf_set_option(b"chamfer_grid", MODES[mode]) == 0
        try:
            row[f"{mode}_ms"] = round(gpu_time(step, iters=20), 4)
            vals[mode] = pkg.losses.flow_loss(model, pc, t, pcf, pcb).detach().clone()
        finally:
            L.nvsf_set_option(b"chamfer_grid", -1)
    row["identical_value"] = torch.equal(vals["brute"].view(torch.int32), vals["auto"].view(torch.int32))
    row["speedup"] = round(row["brute_ms"] / row["auto_ms"], 2)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON lines file (default: print only)")
    ap.add_argument("--small", action="store_true", help="skip the 256 K / 1 M-point workloads")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_chamfer_grid.py runs on the GPU"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    rows = [{"card": q[0] if q else torch.cuda.get_device_name(), "torch": torch.__version__,
             "grid_min_pairs_per_direction": "n*m >= 2^28 (automatic selection)"}]
    print(json.dumps(rows[0]), flush=True)
    for name, a, b in workloads(not args.small):
        rows.append(bench_workload(name, a.contiguous(), b.contiguous()))
        print(json.dumps(rows[-1]), flush=True)
    for fn in (bench_meter, bench_flow_loss):
        rows.append(fn())
        print(json.dumps(rows[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
