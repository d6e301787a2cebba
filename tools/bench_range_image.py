"""Cost of point cloud -> range image (metrics.range_image) at 66 x 1030, the KITTI-360 LiDAR frame:
  (a) one synthetic 120 K-point scan (4 channels, sensor frame);
  (b) 1024 such scans in one call (123 M points; 0.56 GB of keys, beyond the 126 MB L2);
  (c) a world-frame cloud of 16 scans taken at 16 poses, projected at one pose (1.9 M points, ~28 per pixel);
  (d) 16 M points on one pixel (the contention worst case of the same-address reduction);
and, for (a), the vectorised numpy oracle and the literal per-point loop on the host cores.
Per workload: the median of 30 calls, each timed with CUDA events after 5 warm-ups, points/s, and the byte floor
(channels x 4 B read per point + 8 B key cleared, 12 B image written per pixel) at the measured device-to-device
copy bandwidth.  Prints one JSON line with the card's name and power limit; GPU only (no fallback)."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("selfsupervised-nvsf_b200")
H, W, K, K_HOZ = 66, 1030, (2.0, 26.9), (180.0, 360.0)


def gpu_time(fn, iters=30, warmup=5):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, check=True).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except (OSError, subprocess.CalledProcessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def copy_bandwidth():
    """Read + write bytes per second of a 4 GiB device-to-device copy."""
    a = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    ms = gpu_time(lambda: b.copy_(a), iters=10, warmup=2)
    del a, b
    return 2 * (4 << 30) / (ms * 1e-3)


def scan(n, g, channels=4):
    """n points over the frame's frustum (and 1 deg around it), depths 1-90 m, on the device."""
    b = torch.deg2rad(torch.rand(n, device="cuda", generator=g) * 360 - 180)
    a = torch.deg2rad(torch.rand(n, device="cuda", generator=g) * 28.9 - 25.9)
    d = 1 + 89 * torch.rand(n, device="cuda", generator=g)
    cols = [d * a.cos() * b.cos(), d * a.cos() * b.sin(), d * a.sin(), torch.rand(n, device="cuda", generator=g)]
    return torch.stack(cols[:channels], 1).contiguous()


def rigid(g):
    q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g, dtype=torch.float64))
    if torch.det(q) < 0:
        q[:, 0] = -q[:, 0]
    p = torch.eye(4)
    p[:3, :3] = q.float()
    p[:3, 3] = torch.randn(3, generator=g) * 3
    return p.cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--no-host", action="store_true", help="skip the host oracle timings")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_range_image measures on the GPU"
    from oracle import range_image_oracle as RO
    name, power = card()
    bw = copy_bandwidth()
    g = torch.Generator(device="cuda").manual_seed(0)
    gh = torch.Generator().manual_seed(0)
    n1 = 120_000
    a = scan(n1, g)
    big = scan(1024 * n1, g)
    offs = [i * n1 for i in range(1025)]
    poses = [rigid(gh) for _ in range(16)]
    world = torch.cat([torch.cat([(p[:3, :3][None] * s[:, None, :3]).sum(-1) + p[:3, 3], s[:, 3:]], 1)
                       for p, s in zip(poses, (scan(n1, g) for _ in range(16)))])
    one = torch.zeros(16 << 20, 4, device="cuda")
    one[:, 0] = 1 + 49 * torch.rand(16 << 20, device="cuda", generator=g)
    M = pkg.metrics
    work = {
        "a_scan": (a, 1, lambda: M.range_image(a, H, W, K, K_HOZ)),
        "b_1024_scans": (big, 1024, lambda: M.range_image(big, H, W, K, K_HOZ, offsets=offs)),
        "c_world_cloud_at_pose": (world, 1, lambda: M.range_image(world, H, W, K, K_HOZ, poses=poses[0])),
        "d_one_pixel": (one, 1, lambda: M.range_image(one, H, W, K, K_HOZ)),
    }
    out = {"gpu": name, "power_limit": power, "frame": [H, W], "copy_bandwidth_GBps": round(bw / 1e9, 1)}
    for key, (pts, B, fn) in work.items():
        ms = gpu_time(fn)
        P = pts.shape[0]
        floor_bytes = P * pts.shape[1] * 4 + B * H * W * (8 + 12)
        floor_ms = floor_bytes / bw * 1e3
        hits = int((fn()[..., 0] > 0).sum())
        out[key] = {"points": P, "scans": B, "pixels_hit": hits, "ms": round(ms, 4),
                    "Gpoints_per_s": round(P / (ms * 1e-3) / 1e9, 2), "floor_ms": round(floor_ms, 4),
                    "time_over_floor": round(ms / floor_ms, 2)}
    # the device image of (a) equals the host oracle
    host = a.cpu().numpy()
    want, _ = RO.range_image(host, H, W, K, K_HOZ)
    out["a_matches_oracle"] = bool(np.array_equal(M.range_image(a, H, W, K, K_HOZ).cpu().numpy().view(np.uint32),
                                                  want.view(np.uint32)))
    if not args.no_host:
        t0 = time.perf_counter()
        RO.range_image(host, H, W, K, K_HOZ)
        out["a_host_numpy_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
        t0 = time.perf_counter()
        RO.range_image_loop(host, H, W, K, K_HOZ)
        out["a_host_loop_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
        out["host_cores"] = os.cpu_count()
    out["lib"] = os.path.basename(pkg._lib.LIB_PATH)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
