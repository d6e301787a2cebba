"""Mesh extraction cost on the trained-style synthetic model (oracle/field_init.py, style "trained", LiDAR
tables, t = 0.4) at resolution 256, 512 and 1024:
  volume_ms:  sigma on the resolution^3 lattice (NeRFNetwork._density_volume, the first half of extract_geometry);
  mc_ms:      mesh.marching_cubes on that volume, including its one host read (the two counts);
  count_ms / write_ms: the two C ABI phases alone (CUDA events around the launches, no host read).
Each time is the median of REPS runs after WARMUP runs.  The threshold is torch-ngp's default 10 when the volume
has values on both sides of it, otherwise the volume's median (reported as `threshold`).

Bytes: the floor is the volume read once per phase plus the outputs, 8 N + 12 V + 24 T.  The algorithmic bytes
count what the kernels address: the volume twice (8 N); the 16-bit per-point code written by the count kernel and
read by both write kernels (6 N); the 16-bit vertex offsets written by the vertex kernel (2 N); the vertex kernel's
second edge endpoint (4 V); the triangle kernel's gathers of code and offset at each triangle corner's owner (12 T);
and the outputs (12 V + 24 T): 16 N + 16 V + 36 T.  The count kernel's neighbour reads and the gathers are mostly L2
hits, so this is an upper bound on DRAM traffic, and achieved/peak on it is not a DRAM utilisation.
The peak is the measured device-to-device copy bandwidth (read + write bytes of a 4 GiB copy_, median of REPS):
floor_ms = floor bytes / peak, kernels_frac_of_floor = floor_ms / (count_ms + write_ms), and algorithmic_gbs =
algorithmic bytes / (count_ms + write_ms).  The numpy oracle (oracle/mesh_oracle.py) is timed once at 256 for comparison.
Prints one JSON line with the card's name and power limit; run on the GPU (no fallback)."""
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

REPS, WARMUP, T_FRAME = 7, 2, 0.4


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, check=True).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except (OSError, subprocess.CalledProcessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def median_ms(fn, reps=REPS, warmup=WARMUP):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def copy_gbs():
    a = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    ms = median_ms(lambda: b.copy_(a))
    return 2 * a.numel() * 4 / (ms * 1e-3) / 1e9


def model():
    from oracle import field_init
    from oracle.field_oracle import FieldConfig
    S = importlib.import_module("selfsupervised-nvsf_b200.synth")
    kw = dict(bound=S.BOUND, num_frames=S.NUM_FRAMES, time_resolution=S.TIME_RESOLUTION, min_near=S.MIN_NEAR,
              min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    m = pkg.NeRFNetwork(**kw).eval()
    m.load_flat_params(field_init.make_params(FieldConfig(**kw), seed=0, style="trained"))
    return m


def main():
    assert torch.cuda.is_available(), "bench_mesh measures on the GPU"
    from oracle import mesh_oracle
    L, ptr, sp = pkg._lib.lib(), pkg._lib.ptr, pkg._lib.stream_ptr
    peak = copy_gbs()
    m = model()
    result = {"reps": REPS, "warmup": WARMUP, "time": T_FRAME, "copy_gbs": round(peak, 1)}
    for R in (256, 512, 1024):
        t_vol = median_ms(lambda: m._density_volume(T_FRAME, R, True))
        vol, _ = m._density_volume(T_FRAME, R, True)
        tau = 10.0 if bool((vol > 10.0).any() and (vol <= 10.0).any()) else float(vol.median())
        t_mc = median_ms(lambda: pkg.mesh.marching_cubes(vol, tau))
        v, f = pkg.mesh.marching_cubes(vol, tau)
        V, T, N = v.shape[0], f.shape[0], R ** 3
        wb = L.nvsf_marching_cubes_workspace_bytes(R, R, R)
        ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
        counts = torch.empty(2, dtype=torch.int64, device="cuda")
        t_count = median_ms(lambda: L.nvsf_marching_cubes_count(ptr(vol), R, R, R, tau, ptr(counts), ptr(ws), wb,
                                                                sp()))
        t_write = median_ms(lambda: L.nvsf_marching_cubes_write(ptr(vol), R, R, R, tau, ptr(v), V, ptr(f), T, ptr(ws),
                                                                wb, sp()))
        floor_b, alg_b = 8 * N + 12 * V + 24 * T, 16 * N + 16 * V + 36 * T
        k_ms = t_count + t_write
        e = {"threshold": tau, "V": V, "T": T, "volume_ms": round(t_vol, 3), "mc_ms": round(t_mc, 3),
             "count_ms": round(t_count, 3), "write_ms": round(t_write, 3),
             "floor_bytes": floor_b, "algorithmic_bytes": alg_b,
             "floor_ms": round(floor_b / (peak * 1e9) * 1e3, 3),
             "kernels_frac_of_floor": round(floor_b / (peak * 1e9) * 1e3 / k_ms, 3),
             "algorithmic_gbs": round(alg_b / (k_ms * 1e-3) / 1e9, 1)}
        if R == 256:
            u = vol.cpu().numpy()
            t0 = time.perf_counter()
            ov, of = mesh_oracle.marching_cubes(u, tau)
            e["numpy_oracle_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
            e["matches_oracle"] = bool(np.array_equal(of, f.cpu().numpy()) and
                                       np.array_equal(ov.view(np.uint32), v.cpu().numpy().view(np.uint32)))
        result[f"r{R}"] = e
        del vol, v, f, ws
        torch.cuda.empty_cache()
    name, power = card()
    print(json.dumps({"gpu": name, "power_limit": power, **result}))


if __name__ == "__main__":
    main()
