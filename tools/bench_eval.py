"""Cost of evaluating one full LiDAR frame (66 x 1030) on the device, against scoring it on the host:
  - LidarMeter.update alone (pixel pass, SSIM x 2, medians, two point clouds, counted Chamfer, finalize);
  - render_frame + LidarMeter.update (what an evaluation epoch does per frame);
  - the float64 oracle (oracle/metrics_oracle.py: numpy / scipy on the host cores, the way the reference scores
    frames) on the same frame, and the device-to-host copy that path needs first.
The frame is rendered by a synthetic model (oracle/field_init.py "trained" tables) at the LiDAR pose of
tests/golden/rays_ref.npz; the ground truth is a render of the same model at a nearby pose and time.  The model's
untrained ray-drop head renders probabilities below 0.5 everywhere, which would drop every ray; its channel is
raised by 0.5 in both frames so that every ray returns and the Chamfer distance runs on two full clouds of 67 980
points, the largest a frame gives.  Device times are CUDA events (median of 20, launches queued behind a spin
kernel); host times are a wall clock.  Prints one JSON line with the card's name and power limit; run on
the GPU (no fallback)."""
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


def gpu_time(fn, iters=20):
    for _ in range(3):
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


def wall_time(fn, iters=3):
    ts = []
    for _ in range(iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return sorted(ts)[len(ts) // 2]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, check=True).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except (OSError, subprocess.CalledProcessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def main():
    assert torch.cuda.is_available(), "bench_eval measures on the GPU"
    from oracle import field_init
    from oracle import metrics_oracle as MO
    from oracle.field_oracle import FieldConfig
    S = importlib.import_module("selfsupervised-nvsf_b200.synth")
    H, W = 66, 1030
    K, K_hoz = (2.0, 26.9), (180.0, 360.0)
    kw = dict(bound=S.BOUND, num_frames=S.NUM_FRAMES, time_resolution=S.TIME_RESOLUTION, min_near=S.MIN_NEAR,
              min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    model = pkg.NeRFNetwork(**kw).eval()
    model.load_flat_params(field_init.make_params(FieldConfig(**kw), seed=0, style="trained"))
    pose = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "rays_ref.npz"))["pose_a"]).clone()
    pose[:3, 3] *= 0.2
    pose_gt = pose.clone()
    pose_gt[0, 3] += 0.01

    def render(p, t):
        f = model.render_frame(p, K, H, W, t, cal_lidar_color=True, intrinsics_hoz=K_hoz)
        f["image_lidar"][..., 0] += 0.5
        return f

    fb = render(pose_gt, 0.5)
    gt = torch.stack([(fb["image_lidar"][..., 0] > 0.5).float(), fb["image_lidar"][..., 1], fb["depth_lidar"]], -1)
    fa = render(pose, 0.3)
    meter = pkg.metrics.LidarMeter(H, W, K, K_hoz, S.SCALE)
    row = meter.update(fa["depth_lidar"], fa["image_lidar"], gt)
    host = [fa["depth_lidar"].cpu().numpy(), fa["image_lidar"].cpu().numpy(), gt.cpu().numpy()]
    want = MO.lidar_metrics(*host, K, K_hoz, S.SCALE)
    got = dict(zip(pkg.metrics.LIDAR_METRICS, row.tolist()))

    def update():
        meter.update(fa["depth_lidar"], fa["image_lidar"], gt)
        if len(meter._rows) > 64:
            meter.reset()

    def render_update():
        f = render(pose, 0.3)
        meter.update(f["depth_lidar"], f["image_lidar"], gt)
        if len(meter._rows) > 64:
            meter.reset()

    t_update = gpu_time(update)
    t_render = gpu_time(lambda: render(pose, 0.3))
    t_both = gpu_time(render_update)
    t_copy = wall_time(lambda: [fa["depth_lidar"].cpu(), fa["image_lidar"].cpu(), gt.cpu()])
    t_oracle = wall_time(lambda: MO.lidar_metrics(*host, K, K_hoz, S.SCALE))
    name, power = card()
    n_p, n_g = int(got["points_pred"]), int(got["points_gt"])
    print(json.dumps({
        "gpu": name, "power_limit": power, "frame": [H, W], "points_pred": n_p, "points_gt": n_g,
        "chamfer_pairs": 2 * n_p * n_g,
        "row_matches_oracle": bool(got["points_pred"] == want["points_pred"] and got["depth_medae"] == np.float32(
            want["depth_medae"]) and abs(got["chamfer"] - want["chamfer"]) <= 1e-5 * abs(want["chamfer"])),
        "update_ms": round(t_update, 4), "render_frame_ms": round(t_render, 4),
        "render_frame_plus_update_ms": round(t_both, 4),
        "host_copy_ms": round(t_copy, 3), "host_oracle_ms": round(t_oracle, 2),
        "host_cores": os.cpu_count()}))


if __name__ == "__main__":
    main()
