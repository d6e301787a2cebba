"""Occupancy-grid maintenance on the trained-style synthetic model (oracle/field_init.py, style "trained", the model
tools/bench_mesh.py uses; camera grid, C = 2, H = 128: 4.19 M cells):
  mark_ms:        mark_untrained_grid against 64 LiDAR + 64 camera poses of a KITTI-like drive (straight through
                  the scene along x with a slow yaw, 1.2 scene units over 64 frames), including its one host read
                  (the trainable-cell count); coverage_ms: the two coverage launches alone;
  update_full_ms: update_extra_state over every cell (today's default);
  update_marked_ms: the same after the marks (only trainable cells are evaluated);
  update_partial_ms: torch-ngp's partial update (C * H^3 / 2 drawn cells);
  frame: a held-out camera frame (halfway between two training poses) through run_cuda, one-shot, with the grid
         after 3 full updates, without and with the marks: samples and ms.
Each time is the median of REPS runs after WARMUP runs (CUDA events).  Prints one JSON line with the card's name
and power limit; run on the GPU (no fallback)."""
import importlib
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_mesh import card, median_ms, model  # noqa: E402

pkg = importlib.import_module("selfsupervised-nvsf_b200")
S = importlib.import_module("selfsupervised-nvsf_b200.synth")

REPS, WARMUP, T_FRAME, FRAMES = 9, 2, 0.4, 64
K = np.array([[S.CAM_FX, 0, S.CAM_CX], [0, S.CAM_FY, S.CAM_CY], [0, 0, 1]])
CAM_AXES = np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])   # (right, down, forward) in the body


def drive_pose(s, camera):
    """Body pose at trajectory parameter s in [0, FRAMES - 1]: x from -0.6 to 0.6, yaw up to 0.2 rad."""
    u = s / (FRAMES - 1)
    yaw = 0.2 * math.sin(math.pi * u)
    c, si = math.cos(yaw), math.sin(yaw)
    R = np.array([[c, -si, 0.0], [si, c, 0.0], [0.0, 0.0, 1.0]])
    P = np.eye(4)
    P[:3, :3] = R @ CAM_AXES if camera else R
    P[:3, 3] = (-0.6 + 1.2 * u, 0.02 * math.sin(3 * u), 0.0)
    return P.astype(np.float32)


def main():
    assert torch.cuda.is_available(), "bench_occupancy measures on the GPU"
    L, ptr, sp = pkg._lib.lib(), pkg._lib.ptr, pkg._lib.stream_ptr
    m = model()
    C, H = m.cascade, m.grid_size
    n = C * H ** 3
    lid_p = torch.from_numpy(np.stack([drive_pose(k, False) for k in range(FRAMES)])).cuda()
    cam_p = torch.from_numpy(np.stack([drive_pose(k, True) for k in range(FRAMES)])).cuda()
    mark_kw = dict(camera_poses=cam_p, intrinsics=K, H=S.CAM_H, W=S.CAM_W, lidar_poses=lid_p,
                   intrinsics_lidar=(S.LIDAR_FOV_UP, S.LIDAR_FOV), intrinsics_hoz_lidar=(0.0, S.LIDAR_FOV_HOZ))
    res = {"reps": REPS, "warmup": WARMUP, "cells": n, "lidar_poses": FRAMES, "camera_poses": FRAMES}

    def fresh(updates):
        m._grid = {}
        for _ in range(updates):
            m.update_extra_state(T_FRAME, cal_lidar_color=False)

    fresh(3)
    res["update_full_ms"] = round(median_ms(lambda: m.update_extra_state(T_FRAME)), 3)
    fresh(3)
    res["mark_ms"] = round(median_ms(lambda: m.mark_untrained_grid(**mark_kw)), 3)
    cov = torch.zeros(n // 8, dtype=torch.uint8, device="cuda")

    def coverage():
        cov.zero_()
        L.nvsf_grid_coverage_camera(C, H, m.bound, ptr(cam_p), FRAMES, S.CAM_FX, S.CAM_FY, S.CAM_CX, S.CAM_CY,
                                    S.CAM_H, S.CAM_W, ptr(cov), sp())
        L.nvsf_grid_coverage_lidar(C, H, m.bound, ptr(lid_p), FRAMES, S.LIDAR_FOV_UP, S.LIDAR_FOV, S.LIDAR_FOV_HOZ,
                                   m.min_near_lidar, m.lidar_max_depth, ptr(cov), sp())
    res["coverage_ms"] = round(median_ms(coverage), 3)
    st = m._grid[False]
    res["trainable_cells"] = int(st["trainable"].shape[0]) if st["trainable"] is not None else n
    res["marked_cells"] = n - res["trainable_cells"]
    res["update_marked_ms"] = round(median_ms(lambda: m.update_extra_state(T_FRAME)), 3)
    res["update_partial_ms"] = round(median_ms(lambda: m.update_extra_state(T_FRAME, mode="partial")), 3)

    # held-out frame: the same grid (3 full updates), bitfield without and with the marks
    fresh(3)
    bits_plain = m.density_bitfield(False).clone()
    m.mark_untrained_grid(**mark_kw)
    bits_marked = m.density_bitfield(False).clone()
    r = pkg.rays.get_rays(torch.from_numpy(drive_pose(FRAMES / 2 - 0.5, True))[None].cuda(), K, S.CAM_H, S.CAM_W, -1)
    o, d = r["rays_o"], r["rays_d"]
    frame = {}
    outs = {}
    for name, bits in (("plain", bits_plain), ("marked", bits_marked)):
        run = lambda: m.run_cuda(o, d, T_FRAME, cal_lidar_color=False, dt_gamma=S.DT_GAMMA, density_bitfield=bits)
        ms = median_ms(run)
        outs[name] = run()
        frame[name] = {"ms": round(ms, 3), "samples": int(m.last_run_cuda_samples),
                       "occupied_cells": int(np.unpackbits(bits.cpu().numpy()).sum())}
    diff = (outs["plain"]["image"] - outs["marked"]["image"]).abs()
    frame["image_max_abs_diff"] = float(diff.max())
    frame["pixels_changed"] = int((diff.amax(-1) > 0).sum())
    res["frame"] = frame
    name, power = card()
    print(json.dumps({"gpu": name, "power_limit": power, **res}))


if __name__ == "__main__":
    main()
