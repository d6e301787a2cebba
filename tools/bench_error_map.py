"""Per-step cost of error-map guided ray sampling (sample + rays + update, one pose, a 128 x 128 map) in three forms:
  (a) device:      rays.get_lidar_rays / get_rays(use_error_map=True) and rays.update_error_map (the kernels of
                   csrc/scene.cu, no host sync);
  (b) host_map:    the reference's sequence as torch-ngp runs it: the frame's map on the host, .to(device),
                   torch.multinomial(replacement=False), the jitter ops, the ray kernel on the chosen pixels, the
                   loss and the cells copied to the host, gather / scatter on the host map;
  (c) torch_dev:   the same torch ops with the maps kept on the device.
N = 2048 (the reference's num_rays_lidar) and 4096 (bench.py's train step), on the LiDAR 66 x 1030 and camera
376 x 1408 frames.  The per-ray loss is a fixed tensor: the loss head is not part of what is timed.  Each step is
bracketed by CUDA events and followed by a synchronise (path (b) synchronises inside anyway), so a time includes the
host's launch gaps; the median over 1000 steps after 50 warm-up steps is reported.  The sampler and update kernels
are also timed alone: the mean over 1000 back-to-back launches on one map.  The maps stay positive (ones
plus positive losses), a valid distribution for torch.multinomial.  Prints one JSON line with the card's name and
power limit; run on the GPU (no fallback)."""
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("selfsupervised-nvsf_b200")

RES, F, STEPS, WARMUP = 128, 8, 1000, 50
LIDAR_K, LIDAR_K_HOZ = (2.0, 26.9), (180.0, 360.0)
CAM_K = [[560.0, 0.0, 704.0], [0.0, 560.0, 188.0], [0.0, 0.0, 1.0]]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, check=True).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except (OSError, subprocess.CalledProcessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def step_time(fn):
    for _ in range(WARMUP):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(STEPS):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def kernel_us(fn, iters=STEPS):
    """Mean device time of one launch over `iters` back-to-back launches (the queue stays full)."""
    for _ in range(WARMUP):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def main():
    assert torch.cuda.is_available(), "bench_error_map measures on the GPU"
    Lib = pkg._lib.lib()
    ptr, stream_ptr = pkg._lib.ptr, pkg._lib.stream_ptr
    R = RES * RES
    pose = torch.eye(4, device="cuda")[None]
    result = {"res": RES, "steps": STEPS, "warmup": WARMUP}
    for frame, (H, W) in (("lidar", (66, 1030)), ("camera", (376, 1408))):
        if frame == "lidar":
            gen = lambda **kw: pkg.rays.get_lidar_rays(pose, LIDAR_K, LIDAR_K_HOZ, H, W, **kw)
            ray_fn = lambda inds, n, o, d: Lib.nvsf_get_lidar_rays(ptr(pose[0]), ptr(inds), n, H, W, *LIDAR_K,
                                                                   LIDAR_K_HOZ[1], ptr(o), ptr(d), stream_ptr())
        else:
            gen = lambda **kw: pkg.rays.get_rays(pose, CAM_K, H, W, **kw)
            ray_fn = lambda inds, n, o, d: Lib.nvsf_get_rays(ptr(pose[0]), ptr(inds), n, H, W, 560.0, 560.0, 704.0,
                                                             188.0, ptr(o), ptr(d), stream_ptr())
        for N in (2048, 4096):
            g = torch.Generator(device="cuda").manual_seed(N)
            loss = torch.rand(1, N, device="cuda", generator=g)
            maps_dev = torch.ones(F, R, device="cuda")
            maps_dev_t = torch.ones(F, R, device="cuda")
            maps_host = torch.ones(F, R)
            it = [0]

            def frame_index():
                it[0] += 1
                return [it[0] % F]

            def device_path():
                index = frame_index()
                r = gen(N=N, error_map=maps_dev[index], use_error_map=True)
                pkg.rays.update_error_map(maps_dev, index, r["inds_coarse"], loss)

            def torch_step(maps, host):
                index = frame_index()
                em = maps[index].to("cuda")
                inds_coarse = torch.multinomial(em, N, replacement=False)
                ix, iy = inds_coarse // RES, inds_coarse % RES
                sx, sy = H / RES, W / RES
                ix = (ix * sx + torch.rand(1, N, device="cuda") * sx).long().clamp(max=H - 1)
                iy = (iy * sy + torch.rand(1, N, device="cuda") * sy).long().clamp(max=W - 1)
                inds = (ix * W + iy).contiguous()
                o = torch.empty(1, N, 3, device="cuda")
                d = torch.empty(1, N, 3, device="cuda")
                pkg._lib.check(ray_fn(inds[0], N, o[0], d[0]), "rays")
                ic = inds_coarse.cpu() if host else inds_coarse
                e = loss.detach().cpu() if host else loss
                m = maps[index]
                m.scatter_(1, ic, 0.1 * m.gather(1, ic) + 0.9 * e)
                maps[index] = m

            t_dev = step_time(device_path)
            t_host = step_time(lambda: torch_step(maps_host, True))
            t_torch = step_time(lambda: torch_step(maps_dev_t, False))
            r = gen(N=N, error_map=maps_dev[:1], use_error_map=True)
            ic = r["inds_coarse"][0]
            valid = bool((ic[1:] > ic[:-1]).all() and ic[0] >= 0 and ic[-1] < R and torch.isfinite(maps_dev).all()
                         and maps_dev.ne(1.0).any())
            # the two kernels alone, on one map
            w, E = maps_dev[0], torch.empty(R, device="cuda").exponential_()
            jit, ic1 = torch.rand(N, 2, device="cuda"), r["inds_coarse"][0].clone()
            inds1 = torch.empty_like(ic1)
            t_sample = kernel_us(lambda: Lib.nvsf_error_map_sample(ptr(w), ptr(E), ptr(jit), RES, N, H, W, ptr(ic1),
                                                                   ptr(inds1), stream_ptr()))
            t_update = kernel_us(lambda: Lib.nvsf_error_map_update(ptr(maps_dev[1]), R, ptr(ic1), N, ptr(loss[0]),
                                                                   stream_ptr()))
            result[f"{frame}_N{N}"] = {"frame": [H, W], "device_ms": round(t_dev, 4), "host_map_ms": round(t_host, 4),
                                       "torch_device_ms": round(t_torch, 4), "sample_kernel_us": round(t_sample, 2),
                                       "update_kernel_us": round(t_update, 2), "draws_valid": valid}
    name, power = card()
    print(json.dumps({"gpu": name, "power_limit": power, **result}))


if __name__ == "__main__":
    main()
