#!/usr/bin/env python
"""bench.py — NVSF ray-rendering hot path on B200.

Workload (BASELINE.json configs[1]): full-frame LiDAR render of a KITTI-360-shaped range image,
66 x 1030 = 67 980 rays x 768 uniform samples (the reference's --num_steps default,
main_nvsf.py:72), random-init field (reference initialisers), synthetic rays, one frame time per
step.  One "step" = one frame: time-table collapse + field evaluation of 52.2 M samples +
compositing with the intensity / raydrop heads -> depth, intensity, raydrop per ray.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); every rank renders its own frame (rays are
independent: no data-path collective), value = all rays / max-over-ranks device time ("weak").

--dump-outputs DIR writes what the last timed step computed on rank 0 (per ray: depth.npy,
image.npy = intensity / raydrop, and on the CUDA path weights_sum.npy; float32) so that two builds
can be compared output for output: the field parameters, rays and frame times are seeded, so the
same arguments give the same inputs.
"""
import argparse
import ctypes
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "lidar_frame_render_rays_per_sec"
UNIT = "rays/s"
NUM_STEPS = 768
WORKLOAD = ("KITTI-360-shaped LiDAR range image 66x1030 full-frame render (depth/intensity/raydrop), "
            "768 uniform samples/ray, random-init NVSF field (BASELINE configs[1])")
# algorithmic bytes the density kernel must move per sample (DESIGN.md, "density kernel"):
#   static hash 8 lvl x 8 corners x 8 B                         =  512
#   collapsed dynamic hash 3 queries x 3 planes x 8 lvl x 4 x 4 B = 1152
#   collapsed flow grid 16 lvl x 8 corners x 8 B                = 1024
#   space planes 4 scales x 3 planes x 4 texels x 32 B          = 1536
#   collapsed time planes 3 queries x 4 scales x 3 x 2 x 32 B   = 2304
#   outputs sigma f32 + geo f16[16]                             =   36
DENSITY_BYTES_PER_SAMPLE = 512 + 1152 + 1024 + 1536 + 2304 + 36
GATHER_MISS_PEAK_GSECTORS = 290.2   # measured: random 4 / 8 / 16-byte gathers from a 32 MB (L2-resident) table, G sectors/s
GATHER_HIT_PEAK_GSECTORS = 861.1    # measured: the same from a 64 KB (L1-resident) table
SURVEY_BYTES_PER_SAMPLE = 13312 + 48  # SURVEY.md 8(d): the reference's un-collapsed gathers
HEADS_FLOP_PER_SAMPLE = 2 * 2 * (87 * 64 + 64 * 64 + 64 * 1)            # SURVEY.md 8(d), LiDAR heads
HEADS_EXECUTED_FLOP_PER_SAMPLE = 2 * 2 * (16 * 64 + 64 * 64 + 64 * 16)  # what k_composite_tc issues per sample
# Per-stage algorithmic bytes per sample of the staged density evaluation (DESIGN.md 3.2); the
# roofline object describes whichever stage took the largest share of the timed steps.
#   mode 1 (fp32 collapsed tables):  flow stage  = flow grid 16 x 8 x 8 B + 32 B flow out
#                                    encode stage = static hash 512 + collapsed dyn hash 1152 + space planes
#                                                   1536 + time planes 2304 + flow in 32 + feature row out 256
#                                    sigma stage  = feature row in 256 + sigma f32 + geo f16[16] out 36
#   mode 2 (fp16 mirrors, default):  flow stage  = 16 x 8 x 4 B + query positions out 36 (+ flow out 32 un-fused)
#                                    dyn stage   = 288 two-byte gathers from shared-memory tables (576) +
#                                                  query positions in 36 + 24 fp16 values out 48
#                                    encode stage (fused with the sigma MLP, tcgen05) = static hash 512 +
#                                                  fp16 space planes 768 + fp16 time planes 1152 + dyn in 48 +
#                                                  query positions in 36 + sigma / geo out 36
#                                    (un-fused: + feature row out 256 instead of the 36; sigma stage 256 + 36)
def stage_table(L):
    """(bytes per sample, kernel name) per stage for the options the library is running with."""
    opt = lambda k: int(L.nvsf_get_option(k))
    mode = opt(b"density_mode")
    if mode != 2:
        return mode, {"flow_stage": (1024 + 32, "k_flow_stage"), "dyn_stage": (0, "-"),
                      "encode_stage": (512 + 1152 + 1536 + 2304 + 32 + 256, "k_encode_stage"),
                      "sigma_stage": (256 + 36, "k_sigma_stage_tc" if opt(b"sigma_tc") else "k_sigma_stage")}
    fused = bool(opt(b"fuse_sigma"))
    return mode, {
        # the flow rows (32 B) are written only when somebody reads them: not on the fused tcgen05 path
        "flow_stage": (512 + 36 + (0 if fused and opt(b"flow_tc") else 32),
                       "k_flow_tc" if opt(b"flow_tc") else "k_flow_stage"),
        "dyn_stage": (576 + 36 + 48, "k_dyn_stage"),
        "encode_stage": (512 + 768 + 1152 + 48 + 36 + (36 if fused else 256),
                         "k_encode_sigma_tc" if fused else "k_encode_stage"),
        "sigma_stage": (0 if fused else 256 + 36, "-" if fused else
                        ("k_sigma_stage_tc" if opt(b"sigma_tc") else "k_sigma_stage"))}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return json.load(open(path)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled during the timed region: NVML every 20 ms, or nvidia-smi
    every 200 ms when pynvml is absent."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.nvml, self.stop_flag, self.samples = None, False, []

    def _nvml_loop(self):
        n = self.nvml
        h = n.nvmlDeviceGetHandleByIndex(self.index)
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                self.samples.append((n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM), mx, int(get_reasons(h))))
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        try:   # NVML directly: a sample every 20 ms (the timed region of the default run is ~0.3 s)
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            sm = sorted(x[0] for x in self.samples)
            bits = 0
            for x in self.samples:
                bits |= x[2]
            # nvml.h: SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
            reasons = [name for name, bit in (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40),
                                              ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20)) if bits & bit]
            return {"sm_mhz": float(sm[len(sm) // 2]) if sm else None,
                    "sm_max_mhz": float(self.samples[0][1]) if self.samples else None,
                    "reasons": sorted(reasons), "samples": len(sm), "source": "nvml, 20 ms"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one float32 DIR/<name>.npy per output tensor."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy().astype(np.float32))


def synth_frame(S, seed):
    o, d = S.lidar_rays(-1, seed=seed)
    return o, d


def make_oracle(cfg_kw, params):
    from oracle.field_oracle import FieldConfig, FieldOracle
    return FieldOracle(FieldConfig(**cfg_kw), params)


def cpu_render_sample(orc, o, d, t, n_rays):
    import torch
    idx = list(range(0, o.shape[0], max(o.shape[0] // n_rays, 1)))[:n_rays]
    t0 = time.perf_counter()
    with torch.no_grad():
        r = orc.render(torch.from_numpy(o[idx]), torch.from_numpy(d[idx]), t, True, NUM_STEPS)
    return time.perf_counter() - t0, idx, r


def cpu_baseline_and_parity(pkg, S, model, cfg_kw, dev, args):
    """The CPU leg of the bench line (BASELINE.md section 3), rank 0, outside every timed GPU region.

    cpu_baseline: BASELINE configs[0] — 4096 synthetic LiDAR rays x 128 samples, random-init field, the oracle PORT of
    the reference's PyTorch path (oracle/field_oracle.py: NeRFRenderer.run -> NeRFNetwork.density / color with the
    tinycudann stand-in) in fp32 on all host cores: (a) render under no_grad, (b) train step = forward + backward of an
    L1 depth + MSE intensity / raydrop loss; 2 warm-ups, median of 5 (3 for the train step when one run exceeds 8 s);
    plus the OpenMP C oracle of the ray-marching operators on the same 4096 rays (street-shell grid).
    parity: the GPU render of a strided ray sample of the LiDAR frame with TRAINED-style tables (tables U(-1,1), a
    flow that moves the warped queries: sigma is not ~1 everywhere as with the initialisers) against the oracle."""
    import numpy as np
    import torch
    from oracle import field_init
    from oracle import raymarching_oracle as RO
    from oracle.field_oracle import FieldConfig, FieldOracle
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = FieldConfig(**cfg_kw)
    params = field_init.make_params(cfg, seed=0, style="init")
    N0, S0 = 4096, 128
    o, d = S.lidar_rays(N0, seed=0)
    to, td = torch.from_numpy(o), torch.from_numpy(d)
    orc = FieldOracle(cfg, params)

    def render():
        with torch.no_grad():
            return orc.run(to, td, 0.5, True, S0)

    def timed(fn, warm, reps, budget_s):
        ts = []
        for i in range(warm + reps):
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            if i >= warm:
                ts.append(dt)
            if i >= warm + 2 and sum(ts) > budget_s:
                break
        return float(np.median(ts)), len(ts)

    r_s, r_n = timed(render, 2, 5, 60.0)
    leaf = {"lidar": {k: v.clone().requires_grad_(True) for k, v in params["lidar"].items()}}
    for k in ("flow_grid", "flow_mlp", "sigma_net", "intensity_net", "raydrop_net", "color_net"):
        leaf[k] = params[k].clone().requires_grad_(True)
    orc_t = FieldOracle(cfg, leaf)
    gt = torch.rand(N0, 3, generator=torch.Generator().manual_seed(1))

    def train_step():
        for grp in (leaf["lidar"], leaf):
            for v in grp.values():
                if torch.is_tensor(v):
                    v.grad = None
        out = orc_t.run(to, td, 0.5, True, S0)
        loss = ((out["depth"] - gt[:, 2]).abs().sum() + ((out["image"][:, 1] - gt[:, 1]) ** 2).sum()
                + ((out["image"][:, 0] - gt[:, 0]) ** 2).sum())
        loss.backward()

    t_s, t_n = timed(train_step, 1, 5, 24.0)
    # operators: OpenMP C restatement of raymarching.cu on the same rays
    grid = S.density_grid("shell")
    bf = S.packbits_np(grid, 0.01)
    nears = np.full(N0, S.MIN_NEAR_LIDAR, np.float32); fars = np.full(N0, S.LIDAR_MAX_DEPTH, np.float32)
    noises = np.zeros(N0, np.float32)
    cnt = int(RO.march_rays_train(o, d, S.BOUND, bf, S.CASCADE, S.GRID_SIZE, nears, fars, noises, dt_gamma=S.DT_GAMMA,
                                  M=1)[4][0])
    mr = lambda: RO.march_rays_train(o, d, S.BOUND, bf, S.CASCADE, S.GRID_SIZE, nears, fars, noises, dt_gamma=S.DT_GAMMA,
                                     M=max(cnt, 1))
    x_, d_, dl_, ry_, _ = mr()
    rng = np.random.default_rng(2)
    sg = np.exp(rng.normal(0, 2, size=max(cnt, 1))).astype(np.float32); cl = rng.random((max(cnt, 1), 3), dtype=np.float32)
    wsum, dep, img = RO.composite_rays_train_forward(sg, cl, dl_, ry_)
    ops = {}
    for name, fn in (("near_far_from_aabb", lambda: RO.near_far_from_aabb(o, d, S.AABB, S.MIN_NEAR)),
                     ("march_rays_train", mr),
                     ("composite_rays_train_forward", lambda: RO.composite_rays_train_forward(sg, cl, dl_, ry_)),
                     ("composite_rays_train_backward",
                      lambda: RO.composite_rays_train_backward(np.ones(N0, np.float32), np.ones((N0, 3), np.float32), sg, cl,
                                                               dl_, ry_, wsum, img)),
                     ("packbits", lambda: RO.packbits(grid, 0.01))):
        ops[name] = {"ms": timed(fn, 1, 5, 5.0)[0] * 1e3}
    ops["samples"] = cnt
    base = {"value": N0 / r_s, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"BASELINE configs[0]: {N0} LiDAR rays x {S0} samples, random-init field, fp32 torch on {cores} threads; "
                      f"render = median of {r_n} after 2 warm-ups ({r_s:.2f} s each), train step = median of {t_n} after 1",
            "render": {"rays_per_s": N0 / r_s, "samples_per_s": N0 * S0 / r_s, "s_per_run": r_s, "runs": r_n},
            "train_step": {"rays_per_s": N0 / t_s, "samples_per_s": N0 * S0 / t_s, "s_per_run": t_s, "runs": t_n,
                           "what": "forward + backward of L1 depth + MSE intensity / raydrop"},
            "operators_c_oracle_openmp": ops}
    # ---- parity on trained-style tables
    tparams = field_init.make_params(cfg, seed=0, style="trained")
    model.load_flat_params(tparams)
    fo, fd = S.lidar_rays(-1, seed=0)
    idx = np.arange(500, fo.shape[0], fo.shape[0] // args.parity_rays)[:args.parity_rays]
    with torch.no_grad():
        g = model.render(torch.from_numpy(fo).to(dev)[None], torch.from_numpy(fd).to(dev)[None], 31.0 / 63.0,
                         cal_lidar_color=True, staged=True, num_steps=NUM_STEPS)
        e = FieldOracle(cfg, tparams).run(torch.from_numpy(fo[idx]), torch.from_numpy(fd[idx]), 31.0 / 63.0, True, NUM_STEPS)
    gd, gi = g["depth_lidar"][0].cpu().numpy()[idx], g["image_lidar"][0].cpu().numpy()[idx]
    parity = {"what": f"{len(idx)} strided rays of the 66x1030x{NUM_STEPS} LiDAR frame, trained-style tables, GPU render vs CPU oracle",
              "max_rel_err": {"depth": float(np.max(np.abs(gd - e["depth"].numpy()) / (np.abs(e["depth"].numpy()) + 1e-6))),
                              "image": float(np.max(np.abs(gi - e["image"].numpy()) / (np.abs(e["image"].numpy()) + 1e-4)))},
              "tolerance": 1e-2,
              "oracle_weights_sum_mean": float(e["weights_sum"].mean()), "oracle_sigma_std": float(e["sigma"].std())}
    return base, parity


def run_reference(args):
    """--impl reference: the reference path on the host cores.  /root/reference and tinycudann do
    not exist on the GPU box, so this times the oracle PORT of that path (oracle/field_oracle.py,
    pinned to the reference modules by tests/test_field_oracle_golden.py) with all host threads,
    on a bounded sample of the same frame per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    S = importlib.import_module("selfsupervised-nvsf_b200.synth")
    from oracle import field_init
    torch.set_num_threads(os.cpu_count() or 1)
    cfg_kw = dict(bound=S.BOUND, num_frames=S.NUM_FRAMES, time_resolution=S.TIME_RESOLUTION, min_near=S.MIN_NEAR,
                  min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    from oracle.field_oracle import FieldConfig
    params = field_init.make_params(FieldConfig(**cfg_kw), seed=0, style="init")
    orc = make_oracle(cfg_kw, params)
    o, d = synth_frame(S, 0)
    n_rays = args.ref_rays
    for _ in range(args.warmup):
        cpu_render_sample(orc, o, d, 0.5, max(n_rays // 4, 1))
    t_total = 0.0
    for k in range(args.steps):
        dt, _, r = cpu_render_sample(orc, o, d, (k % 60 + 2) / 63.0, n_rays)
        t_total += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"depth": r["depth"], "image": r["image"]})
    value = n_rays * args.steps / t_total
    sample = f"{n_rays} of 67980 rays x {NUM_STEPS} samples per step (strided over the frame)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rays_per_gpu": 67980, "samples_per_ray": NUM_STEPS,
                   "parallelism": "host cores of rank 0"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def build_train_step(pkg, S, cfg_kw, dev, rank, world, rays, shard=False, comm_dtype=None):
    """The joint training step of bench_train as a closure (also used by tools/prof_train_timeline.py)."""
    import numpy as np
    import torch
    torch.manual_seed(0)   # same initial replica on every rank
    model = pkg.NeRFNetwork(device=dev, **cfg_kw).train()
    opt = pkg.optim.FlatAdam(model, lr=1e-2, shard=shard and world > 1, skip_nonfinite=True, comm_dtype=comm_dtype)
    lo, ld = S.lidar_rays(rays, seed=100 + rank)
    co, cd = S.camera_rays(rays, seed=200 + rank)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    lo_h, ld_h, co_h, cd_h = pin(lo), pin(ld), pin(co), pin(cd)
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    # images_lidar [1, N, 3] = (raydrop mask, intensity, depth) as the reference's train_step reads it
    gt_l = torch.rand(1, rays, 3, device=dev, generator=g)
    gt_l[..., 0] = (gt_l[..., 0] > 0.2).float()
    gt_l[..., 2] *= 0.8
    gt_c = torch.rand(1, rays, 3, device=dev, generator=g)
    loss_h = torch.zeros(1).pin_memory()
    t = torch.tensor([[0.4]], device=dev)
    cham = pkg.chamfer.chamfer_3DDist()
    gt_pts = (torch.from_numpy(np.ascontiguousarray(ld)).to(dev)[None] * (gt_l[..., 2] * gt_l[..., 0]).unsqueeze(-1)
              / S.SCALE).contiguous()

    def step():
        a, b = lo_h.to(dev, non_blocking=True), ld_h.to(dev, non_blocking=True)
        c, d = co_h.to(dev, non_blocking=True), cd_h.to(dev, non_blocking=True)
        opt.zero_grad()
        ol = model.render(a[None], b[None], t, cal_lidar_color=True, staged=False, num_steps=NUM_STEPS, perturb=True)
        # loss head of trainer.py:188-219 / 503-504 (csrc/loss.cu: loss and its derivative in one kernel)
        l1 = pkg.losses.lidar_loss(ol["depth_lidar"], ol["image_lidar"], gt_l).sum()
        # Chamfer term between predicted and ground-truth points (trainer.py:206, 229-233), csrc/chamfer.cu
        pred_depth = (ol["depth_lidar"] * gt_l[..., 0]).unsqueeze(-1)
        d1, d2, _, _ = cham(b[None] * pred_depth / S.SCALE, gt_pts)
        l1 = l1 + (d1 + d2).mean() * 0.5
        l1.backward()
        opt.sync.reduce_group("lidar")      # overlaps the camera render
        oc = model.render(c[None], d[None], t, cal_lidar_color=False, staged=False, num_steps=NUM_STEPS, perturb=True)
        l2 = pkg.losses.rgb_loss(oc["image"], gt_c).sum()
        l2.backward()
        opt.sync.reduce_group("camera")
        opt.sync.reduce_group("shared")
        opt.sync.wait()
        opt.step()      # found_inf check (4-byte MAX all-reduce at N > 1) + guarded Adam (+ parameter all-gather)
        loss_h.copy_((l1 + l2).detach().view(1), non_blocking=True)

    return step, model, opt, loss_h


def bench_train(pkg, S, cfg_kw, dev, rank, world, rays, steps, warmup, shard=False, comm_dtype=None):
    """Joint training step (BASELINE configs[2] at 4096+4096 rays, configs[4] at 32768+32768 rays per
    GPU): per step, pinned host rays -> device, LiDAR render + loss head + Chamfer term + backward, camera
    render + loss head + backward (NeRFNetwork.render with autograd, 768 samples/ray, perturb=True), gradient
    reduction over NCCL overlapped per group (dist.GradSync: all-reduce, or reduce-scatter with shard=True),
    non-finite check + Adam step (optim.FlatAdam; with shard=True on the rank's slice, then the parameter
    all-gather), loss read back to the host.  Returns whole-job rays/s from the max-over-ranks device time."""
    import torch
    import torch.distributed as dist
    step, model, opt, loss_h = build_train_step(pkg, S, cfg_kw, dev, rank, world, rays, shard, comm_dtype)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = max(e0.elapsed_time(e1), 0.0)
    wall_ms = (time.perf_counter() - t0) * 1e3
    tm = torch.tensor([max(ms, wall_ms)], device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_max = float(tm.item())
    grad_bytes = opt.sync.flat.numel() * 4
    del model, opt
    torch.cuda.empty_cache()
    return {"value": world * 2 * rays * steps / (ms_max * 1e-3), "unit": "rays/s", "ms_per_step": ms_max / steps,
            "rays_per_gpu": {"lidar": rays, "camera": rays}, "samples_per_ray": NUM_STEPS, "steps": steps,
            "final_loss": float(loss_h.item()), "allreduce_bytes_per_step": grad_bytes if world > 1 else 0,
            "gradient_reduction": ("none (1 rank)" if world == 1 else
                                   ("reduce-scatter + sharded Adam + parameter all-gather" if shard else "all-reduce + full Adam")
                                   + (", bf16 gradients on the wire" if comm_dtype is not None else ", fp32 wire")),
            "includes": "h2d rays, fwd + loss head (+ Chamfer term, LiDAR) + bwd of both modalities, gradient reduction (N>1), device-side non-finite check (4-byte MAX all-reduce at N>1), guarded Adam step, table re-pack, d2h loss"}


def op_rooflines(pkg, S, model, dev, o, d, bits, peak_gbs):
    """Per-kernel roofline entries of the ray-marching operators on this rank's camera rays (north_star:
    "achieved HBM GB/s against B200 peak for marching ... and compositing"): CUDA-event time of each operator
    (median of 5, working set > L2) against its ALGORITHMIC bytes (SURVEY 8d: marcher 48 B/ray + 32 B/sample,
    compositing forward 24 B/sample + 32 B/ray, backward 40 B/sample + 48 B/ray).  ncu --set full of the same
    kernels: profiles/r02_raymarching_ops_ncu_full.txt."""
    import numpy as np
    import torch
    rm = pkg.raymarching
    L = pkg._lib.lib()
    N = o.shape[0]
    aabb = torch.from_numpy(S.AABB).to(dev)
    nears, fars = rm.near_far_from_aabb(o, d, aabb, S.MIN_NEAR)

    def med(fn, reps=5):
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    xyzs, dirs, deltas, rays = rm.march_rays_train(o, d, S.BOUND, bits, S.CASCADE, S.GRID_SIZE, nears, fars, None, -1,
                                                   False, -1, True, S.DT_GAMMA, 1024)
    M = xyzs.shape[0]
    ws_bytes = L.nvsf_march_rays_train_workspace_bytes(N)
    ws = torch.empty(max(ws_bytes, 4), dtype=torch.uint8, device=dev)
    counter = torch.zeros(2, dtype=torch.int32, device=dev)
    noises = torch.zeros(N, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def march():
        counter.zero_()
        assert L.nvsf_march_rays_train(o.data_ptr(), d.data_ptr(), bits.data_ptr(), S.BOUND, S.DT_GAMMA, 1024, N, S.CASCADE,
                                       S.GRID_SIZE, M, nears.data_ptr(), fars.data_ptr(), xyzs.data_ptr(), dirs.data_ptr(),
                                       deltas.data_ptr(), rays.data_ptr(), counter.data_ptr(), noises.data_ptr(),
                                       ws.data_ptr(), ws_bytes, st) == 0

    with torch.no_grad():
        sig, rgb = model.forward(xyzs, dirs, 0.5, False, out_ld=3)       # the field's own sigmas / colours
    wsum = torch.empty(N, device=dev); dep = torch.empty(N, device=dev); img = torch.empty(N, 3, device=dev)
    gws = torch.ones(N, device=dev); gim = torch.ones(N, 3, device=dev)
    gs = torch.zeros(M, device=dev); gr = torch.zeros(M, 3, device=dev)

    def cfwd():
        assert L.nvsf_composite_rays_train_forward(sig.data_ptr(), rgb.data_ptr(), deltas.data_ptr(), rays.data_ptr(), M, N,
                                                   1e-4, wsum.data_ptr(), dep.data_ptr(), img.data_ptr(), st) == 0

    def cbwd():
        assert L.nvsf_composite_rays_train_backward(gws.data_ptr(), gim.data_ptr(), sig.data_ptr(), rgb.data_ptr(),
                                                    deltas.data_ptr(), rays.data_ptr(), wsum.data_ptr(), img.data_ptr(), M, N,
                                                    1e-4, gs.data_ptr(), gr.data_ptr(), st) == 0

    def nf():
        assert L.nvsf_near_far_from_aabb(o.data_ptr(), d.data_ptr(), aabb.data_ptr(), N, S.MIN_NEAR, nears.data_ptr(),
                                         fars.data_ptr(), st) == 0

    out = {}
    for name, fn, nbytes in (("near_far_from_aabb", nf, 32 * N), ("march_rays_train", march, 48 * N + 32 * M),
                             ("composite_rays_train_forward", cfwd, 24 * M + 32 * N),
                             ("composite_rays_train_backward", cbwd, 40 * M + 48 * N)):
        fn()
        ms = med(fn)
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[name] = {"bound": "hbm", "ms": ms, "algorithmic_bytes": int(nbytes), "achieved": gbs, "peak": peak_gbs,
                     "unit": "GB/s", "frac": gbs / peak_gbs}
    out["rays"], out["samples"] = N, M
    out["note"] = ("this rank's rays of the 376x1408 frame on the street-shell grid; sigmas / colours are the field's own "
                   "(early termination at T < 1e-4 as in training); launch latency included (CUDA events around the C-ABI call)")
    return out


def bench_camera_march(pkg, S, model, dev, rank, world, steps, warmup, peak_gbs):
    """BASELINE configs[3]: camera novel-view render 376x1408 RGB with occupancy-grid skipping, ONE
    frame whose rays are sharded across the ranks — image ROWS dealt round-robin (dist.shard_interleaved:
    a contiguous split is unbalanced, the upper rows miss the scene) — with no collective.  Per step through
    the public API: pinned host rays of this rank's shard -> device, NeRFNetwork.run_cuda (near_far ->
    march_rays_train -> density -> color heads -> composite_rays_train) against a synthetic street-shell
    occupancy bitfield, image -> host.  No host synchronisation inside a frame: the sample rows are
    provisioned from the count of the warm-up frame (`sample_capacity`, torch-ngp's mean_count protocol) and
    the device-side count is checked after the timed region.  value = frame rays / max-over-ranks time
    ("strong")."""
    import numpy as np
    import torch
    import torch.distributed as dist
    o, d = S.camera_rays(-1, seed=0)
    n_all = o.shape[0]
    idx = pkg.dist.shard_interleaved(n_all, rank, world, S.CAM_W).numpy()
    n_mine = idx.shape[0]
    o_pin = torch.from_numpy(np.ascontiguousarray(o[idx]))[None].pin_memory()
    d_pin = torch.from_numpy(np.ascontiguousarray(d[idx]))[None].pin_memory()
    img_h = torch.empty(1, n_mine, 3).pin_memory()
    bits = torch.from_numpy(S.packbits_np(S.density_grid("shell"), 0.01)).to(dev)
    t = torch.tensor([[0.5]], device=dev)
    # warm-up frame with the exact (synchronising) path learns the sample count of this shard
    model.run_cuda(o_pin.to(dev), d_pin.to(dev), t, cal_lidar_color=False, dt_gamma=S.DT_GAMMA, T_thresh=1e-2,
                   density_bitfield=bits, one_shot=True)
    my_samples = int(model.last_run_cuda_samples)
    capacity = (int(my_samples * 1.02) + 127) // 128 * 128
    counters = []

    def step():
        ro, rd = o_pin.to(dev, non_blocking=True), d_pin.to(dev, non_blocking=True)
        r = model.run_cuda(ro, rd, t, cal_lidar_color=False, dt_gamma=S.DT_GAMMA, T_thresh=1e-2,
                           density_bitfield=bits, one_shot=True, sample_capacity=capacity)
        counters.append(model.last_run_cuda_counter)
        img_h.copy_(r["image"], non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    seen = max(int(c[0].item()) for c in counters[-steps:])      # device-side counts, read after the timed region
    if seen > capacity:
        raise RuntimeError(f"camera frame: {seen} samples exceed the provisioned {capacity}")
    tm = torch.tensor([ms, float(my_samples)], device=dev)
    if world > 1:
        mx = tm.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(tm, op=dist.ReduceOp.SUM)
        ms, samples, smax = float(mx[0]), int(tm[1]), float(mx[1])
    else:
        samples, smax = int(tm[1]), float(tm[1])
    out = {"value": n_all * steps / (ms * 1e-3), "unit": "rays/s", "ms_per_frame": ms / steps, "rays": n_all,
           "samples": samples, "steps": steps, "scaling": "strong", "occupancy_grid": "synthetic street shell, 2x128^3",
           "sharding": f"image rows round-robin over {world} rank(s)",
           "samples_per_rank_max_over_mean": smax / (samples / world),
           "includes": "h2d rays of the shard, near_far, march (count+scan+write), density, colour heads, "
                       "compositing, d2h image; no host synchronisation inside a frame (sample rows provisioned "
                       "from the warm-up frame's count + 2 %, device-side count verified after the timed region)"}
    if rank == 0:
        out["operators"] = op_rooflines(pkg, S, model, dev, o_pin[0].to(dev), d_pin[0].to(dev), bits, peak_gbs)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-rays", type=int, default=512, help="rays per step of the CPU reference arm")
    ap.add_argument("--parity-rays", type=int, default=128, help="rays of the in-bench parity check against the oracle")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the train_step sub-benchmarks")
    ap.add_argument("--no-march", action="store_true", help="skip the camera occupancy-skipping render sub-benchmark")
    ap.add_argument("--train-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's per-ray outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    pkg = importlib.import_module("selfsupervised-nvsf_b200")
    S = importlib.import_module("selfsupervised-nvsf_b200.synth")
    F = pkg.field
    L = F._setup_lib()
    if "NVSF_DENSITY_MODE" in os.environ:  # development A/B switch; default = library default
        F.check(L.nvsf_set_option(b"density_mode", int(os.environ["NVSF_DENSITY_MODE"])), "set_option")

    # ---- model: random init exactly as the reference initialisers, same on every rank ----
    cfg_kw = dict(bound=S.BOUND, num_frames=S.NUM_FRAMES, time_resolution=S.TIME_RESOLUTION, min_near=S.MIN_NEAR,
                  min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    model = pkg.NeRFNetwork(device=dev, **cfg_kw).eval()
    params = None
    want_cpu = rank == 0 and not args.no_cpu_baseline
    if want_cpu:
        from oracle import field_init
        from oracle.field_oracle import FieldConfig
        params = field_init.make_params(FieldConfig(**cfg_kw), seed=0, style="init")
        model.load_flat_params(params)  # so that the CPU arm evaluates the very same field
    else:
        torch.manual_seed(0)

    # ---- this rank's frame (device resident for `value`) ----
    o_np, d_np = synth_frame(S, seed=rank)
    N, Sn = o_np.shape[0], NUM_STEPS
    rays_o, rays_d = torch.from_numpy(o_np).to(dev), torch.from_numpy(d_np).to(dev)
    nears = torch.full((N,), model.min_near_lidar, device=dev)
    fars = torch.full((N,), model.lidar_max_depth, device=dev)
    depth = torch.empty(N, device=dev); image = torch.empty(N, 2, device=dev); wsum = torch.empty(N, device=dev)
    sbytes = L.nvsf_render_uniform_scratch_bytes(N, Sn)
    scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
    cfg = ctypes.byref(model._cfg)
    stream = torch.cuda.current_stream().cuda_stream
    times = [(k % 60 + 2) / 63.0 for k in range(args.warmup + args.steps)]
    t_dev = [torch.tensor([t], dtype=torch.float32, device=dev) for t in times]
    ws = model.prepare(times[0], True)
    pc = model._params_c(True)
    launches_per_step = 9 + 1 + 1  # pack_time (1 setup + 3 dyn + 1 flow + 4 planes) + density + composite

    def step(k, ev=None):
        F.check(L.nvsf_field_pack_time(cfg, ctypes.byref(pc), t_dev[k].data_ptr(), ws.data_ptr(), ws.numel(), stream), "pack_time")
        if ev is not None:
            ev[0].record()
        F.check(L.nvsf_render_uniform_density(cfg, ws.data_ptr(), rays_o.data_ptr(), rays_d.data_ptr(), nears.data_ptr(),
                                              fars.data_ptr(), None, N, Sn, scratch.data_ptr(), sbytes, stream), "density")
        if ev is not None:
            ev[1].record()
        F.check(L.nvsf_render_uniform_composite(cfg, ws.data_ptr(), 1, rays_d.data_ptr(), nears.data_ptr(), fars.data_ptr(),
                                                None, N, Sn, 1.0, scratch.data_ptr(), sbytes, depth.data_ptr(),
                                                image.data_ptr(), wsum.data_ptr(), None, None, stream), "composite")
        if ev is not None:
            ev[2].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(args.warmup):
        step(k)
    torch.cuda.synchronize()
    F.check(L.nvsf_set_option(b"stage_timing", 1), "set_option")   # CUDA events around every stage launch
    sampler = ClockSampler(local) if rank == 0 else None
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.start()
    e0.record()
    for k in range(args.steps):
        step(args.warmup + k, evs[k])
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    stage_ms = (ctypes.c_float * 4)()
    stage_launches = ctypes.c_uint32(0)
    F.check(L.nvsf_stage_timing_read(stage_ms, ctypes.byref(stage_launches)), "stage_timing_read")
    F.check(L.nvsf_set_option(b"stage_timing", 0), "set_option")
    clocks = sampler.stop() if sampler else None
    t_max = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
    ms_total_max = float(t_max.item())
    dens_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in evs]))
    comp_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in evs]))
    value = world * N * args.steps / (ms_total_max * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"depth": depth, "image": image, "weights_sum": wsum})

    # ---- e2e: public API, pinned host rays -> device -> render -> host result, every step ----
    o_pin = torch.from_numpy(o_np)[None].pin_memory(); d_pin = torch.from_numpy(d_np)[None].pin_memory()
    depth_h = torch.empty(1, N).pin_memory(); image_h = torch.empty(1, N, 2).pin_memory()

    def e2e_step(k):
        ro, rd = o_pin.to(dev, non_blocking=True), d_pin.to(dev, non_blocking=True)
        r = model.render(ro, rd, t_dev[k].view(1, 1), cal_lidar_color=True, staged=True, num_steps=Sn)
        depth_h.copy_(r["depth_lidar"], non_blocking=True); image_h.copy_(r["image_lidar"], non_blocking=True)

    for k in range(args.warmup):
        e2e_step(k)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for k in range(args.steps):
        e2e_step(args.warmup + k)
    e1.record()
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    t_max = torch.tensor([e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
    e2e_value = world * N * args.steps / (float(t_max.item()) * 1e-3)

    # ---- the same frame from a sensor pose: rays generated on the device in the renderer's stream
    #      (NeRFNetwork.render_frame; the frame's host input is the 4x4 pose, 64 bytes) ----
    R_np, t_np = S.random_pose(rank)
    pose_np = np.eye(4, dtype=np.float32)
    pose_np[:3, :3], pose_np[:3, 3] = R_np.astype(np.float32), t_np.astype(np.float32)
    pose_pin = torch.from_numpy(pose_np).pin_memory()
    depth_f = torch.empty(S.LIDAR_H, S.LIDAR_W).pin_memory(); image_f = torch.empty(S.LIDAR_H, S.LIDAR_W, 2).pin_memory()

    def pose_step(k):
        r = model.render_frame(pose_pin, (S.LIDAR_FOV_UP, S.LIDAR_FOV), S.LIDAR_H, S.LIDAR_W, t_dev[k].view(1, 1),
                               cal_lidar_color=True, intrinsics_hoz=(S.LIDAR_FOV_UP, S.LIDAR_FOV_HOZ), num_steps=Sn)
        depth_f.copy_(r["depth_lidar"], non_blocking=True); image_f.copy_(r["image_lidar"], non_blocking=True)

    for k in range(args.warmup):
        pose_step(k)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for k in range(args.steps):
        pose_step(args.warmup + k)
    e1.record()
    barrier()
    pose_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    t_max = torch.tensor([pose_ms], device=dev)
    if world > 1:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
    pose_value = world * N * args.steps / (float(t_max.item()) * 1e-3)

    # ---- joint training step (configs[2]; configs[4] = 64 K rays per GPU when N > 1) ----
    train = {}
    del scratch
    torch.cuda.empty_cache()
    if not args.no_march:
        train["camera_march_render"] = bench_camera_march(pkg, S, model, dev, rank, world, args.train_steps, 3,
                                                          float(peaks()[0]["hbm_gbs"]))
    if not args.no_train:
        train["train_step"] = bench_train(pkg, S, cfg_kw, dev, rank, world, 4096, args.train_steps, 3)
        if world > 1:
            # the optimizer as the epilogue of the gradient reduction: reduce-scatter -> Adam on the rank's
            # slice -> parameter all-gather (fp32 wire, then bf16 gradients on the wire)
            train["train_step_sharded_adam"] = bench_train(pkg, S, cfg_kw, dev, rank, world, 4096,
                                                           args.train_steps, 3, shard=True)
            train["train_step_sharded_adam_bf16_wire"] = bench_train(pkg, S, cfg_kw, dev, rank, world, 4096,
                                                                     args.train_steps, 3, shard=True,
                                                                     comm_dtype=torch.bfloat16)
            train["train_step_64k_rays_per_gpu"] = bench_train(pkg, S, cfg_kw, dev, rank, world, 32768,
                                                               max(args.train_steps // 2, 2), 2, shard=True)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_kind = peaks()
    n_samples = N * Sn
    n_launch = max(int(stage_launches.value), 1)            # chunks of the staged evaluation, all timed steps
    flow_ms, dyn_ms, enc_ms, sig_ms = (float(stage_ms[i]) / args.steps for i in range(4))
    mode, table = stage_table(L)
    stage_step_ms = {"flow_stage": flow_ms, "dyn_stage": dyn_ms, "encode_stage": enc_ms, "sigma_stage": sig_ms}
    top = max(stage_step_ms, key=stage_step_ms.get)          # the dominant kernel of the step
    top_bytes, top_kernel = table[top]
    top_launch_ms = stage_step_ms[top] * args.steps / n_launch   # average duration of one launch of it
    samples_per_launch = n_samples * args.steps / n_launch
    ncu = {}
    tr_path = os.path.join(ROOT, "profiles", "dominant_stage_ncu.json")
    if os.path.exists(tr_path):   # from the committed ncu --set full capture of this command
        ncu = json.load(open(tr_path))
    hbm_peak = float(pk["hbm_gbs"])

    def stage_entry(kernel, ms_step, alg_bytes_per_sample):
        """One kernel against the HBM roof.  `achieved` is the kernel's MEASURED DRAM traffic (ncu dram__bytes_read.sum
        + dram__bytes_write.sum per sample of the committed capture, scaled to this launch) over its live CUDA-event
        duration: the tables are L2 / shared-memory resident, so the algorithmic gather bytes are not HBM bytes and are
        reported apart, never as a fraction of the HBM peak.  `limiter` names the unit that does bound the kernel, with
        the ncu counters it was read from."""
        k = ncu.get(kernel, {})
        e = {"kernel": kernel, "ms_per_step": ms_step, "bound": "hbm", "peak": hbm_peak, "unit": "GB/s"}
        per_sample = k.get("dram_bytes_per_sample")
        if per_sample is not None and ms_step > 0.05:
            traffic = per_sample * samples_per_launch
            e["traffic"] = traffic
            e["achieved"] = traffic * (n_launch / args.steps) / (ms_step * 1e-3) / 1e9
            e["frac"] = e["achieved"] / hbm_peak
        else:
            e["traffic"], e["achieved"], e["frac"] = None, None, None
        e["algorithmic"] = {"bytes_per_sample": alg_bytes_per_sample,
                            "gbs": (alg_bytes_per_sample * n_samples / (ms_step * 1e-3) / 1e9 if ms_step > 0.05 else None),
                            "note": "table gathers served from L2 / shared memory; not HBM traffic"}
        e["limiter"] = k.get("limiter")
        e["ncu"] = {m: k.get(m) for m in ("l1tex_pct", "lts_pct", "dram_pct", "ipc", "occupancy_pct", "source") if m in k}
        # The on-chip roof of a gather kernel, from two measured ceilings of this chip (tools/ubench_gather.cu,
        # profiles/r02_ubench_gather.txt + _ncu.txt): random sector gathers that MISS L1 run at 1.00 sector per clock per
        # SM = 290 G sectors/s (the L1 -> crossbar request port is then 96-99 % busy, L2 78 %) whatever the occupancy,
        # the loads in flight or the access width; gathers that HIT L1 at >= 2.96 per clock per SM = 861 G sectors/s.
        # floor = misses / 290 + hits / 861 for the L1 sector counts of this kernel (ncu, committed capture);
        # frac = floor / live duration.  `data_pipe_pct` is the unit ncu reports closest to saturation in the real
        # kernel: the L1 data pipe (LSU wavefronts) — the 16-byte plane texels cost four wavefronts of register
        # write-back per load however coherent the warp's addresses are.
        miss, hit = k.get("l1_miss_sectors_ld_per_sample"), k.get("l1_hit_sectors_ld_per_sample")
        if miss is not None and hit is not None and ms_step > 0.05:
            floor_ms = (miss / GATHER_MISS_PEAK_GSECTORS + hit / GATHER_HIT_PEAK_GSECTORS) * n_samples * 1e-6
            e["gather"] = {"bound": "l1 sector gathers (measured miss / hit ceilings)", "unit": "G sectors/s",
                           "peak_miss": GATHER_MISS_PEAK_GSECTORS, "peak_hit": GATHER_HIT_PEAK_GSECTORS,
                           "l1_miss_sectors_per_sample": miss, "l1_hit_sectors_per_sample": hit,
                           "achieved": (miss + hit) * n_samples / (ms_step * 1e-3) / 1e9,
                           "floor_ms": floor_ms, "frac": floor_ms / ms_step,
                           "data_pipe_pct": k.get("l1_data_pipe_pct"), "xbar_req_pct": k.get("l1_xbar_req_pct"),
                           "peak_source": "profiles/r02_ubench_gather.txt, r02_ubench_gather_ncu.txt (tools/ubench_gather.cu "
                                          "on this pool's B200)"}
        return e

    stages = {k: stage_entry(table[k][1], stage_step_ms[k], table[k][0]) for k in table if table[k][1] != "-"}
    kernels_per_chunk = sum(1 for b, k in table.values() if k != "-")
    tensor_peak = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1590.0)))
    heads_kernel = {0: "k_render_composite", 1: "k_composite_tc", 6: "k_composite_ts"}.get(
        int(L.nvsf_get_option(b"heads_tc")), "k_composite_tc8")
    roof = dict(stages[top])
    roof.update({"density_mode": mode, "peak_source": pk_kind, "samples_per_launch": samples_per_launch,
                 "launch_ms": top_launch_ms, "launches_per_step": n_launch / args.steps,
                 "share_of_step": stage_step_ms[top] / (ms_total / args.steps),
                 "traffic_source": ncu.get("source"),
                 "survey_bytes_per_sample": SURVEY_BYTES_PER_SAMPLE,
                 "stages": stages,
                 "heads": {"bound": "tensor", "kernel": heads_kernel,
                           "ms_per_step": comp_ms, "flop_per_sample": HEADS_FLOP_PER_SAMPLE,
                           "executed_flop_per_sample": HEADS_EXECUTED_FLOP_PER_SAMPLE,
                           "achieved": HEADS_FLOP_PER_SAMPLE * n_samples / (comp_ms * 1e-3) / 1e12,
                           "achieved_executed": HEADS_EXECUTED_FLOP_PER_SAMPLE * n_samples / (comp_ms * 1e-3) / 1e12,
                           "peak": tensor_peak, "unit": "TFLOP/s", "peak_kind": "sustained dense bf16 (cuBLAS, measured)",
                           "frac": HEADS_FLOP_PER_SAMPLE * n_samples / (comp_ms * 1e-3) / 1e12 / tensor_peak,
                           "frac_executed": HEADS_EXECUTED_FLOP_PER_SAMPLE * n_samples / (comp_ms * 1e-3) / 1e12 / tensor_peak,
                           "ncu": ncu.get(heads_kernel, {}),
                           "note": "compositing + intensity / raydrop heads of every sample (all pass the w > 1e-4 mask "
                                   "with random-init weights); algorithmic flops are SURVEY 8(d)'s 2 nets x 2 (87*64 + "
                                   "64*64 + 64*1); executed = 2 nets x 2 (16*64 + 64*64 + 64*16): the direction columns "
                                   "of layer 1 are evaluated once per ray"}})
    if "camera_march_render" in train and "operators" in train["camera_march_render"]:
        roof["operators"] = train["camera_march_render"].pop("operators")
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "rays_per_gpu": N, "samples_per_ray": Sn, "parallelism": f"rays x{world} (one frame per GPU, no collective)",
                   "l2": "per-step working set 1.9 GB of per-sample scratch + 128 MB tables exceeds the 126 MB L2; no flush",
                   "kernel_ms": {"field_density": dens_ms, "flow_stage": flow_ms, "dyn_stage": dyn_ms, "encode_stage": enc_ms,
                                 "sigma_stage": sig_ms, "composite_heads": comp_ms,
                                 "time_collapse_and_gaps": ms_total / args.steps - dens_ms - comp_ms}},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(2 * N * 3 * 4), "d2h_bytes_per_step": int(N * 3 * 4)},
        "e2e_from_pose": {"value": pose_value, "unit": UNIT, "h2d_bytes_per_step": 64, "d2h_bytes_per_step": int(N * 3 * 4),
                          "what": "NeRFNetwork.render_frame: pinned 4x4 pose -> device, rays generated on the device in the "
                                  "renderer's stream (get_lidar_rays kernel), render, depth / image -> host"},
        "gpu_launches": (9 + 1 + kernels_per_chunk * n_launch // args.steps) * args.steps,
        "roofline": roof,
    }
    out.update(train)
    if want_cpu:
        out["cpu_baseline"], out["parity"] = cpu_baseline_and_parity(pkg, S, model, cfg_kw, dev, args)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
