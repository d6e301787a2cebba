"""Cost of the training-state features of FlatAdam at the full model size (bench.py's, 93.6 M parameters, one GPU):
  - update_ema(): nvsf_ema_update over the flat buffer (12 B of HBM traffic per parameter), against the
    per-tensor loop torch_ema runs (tmp = s - p; tmp.mul_(omd); s.sub_(tmp)) over the reference's parameter
    tensors — three kernels and a temporary per tensor;
  - state_dict() / load_state_dict(): host clock around the call and a device synchronise.
Prints one JSON line with the card's name and power limit; run on the GPU (no fallback)."""
import importlib
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("selfsupervised-nvsf_b200")


def gpu_time(fn, iters=20):
    """Median device time of one call, with the launches queued behind a spin kernel so that host-side
    launch cost does not sit between the events."""
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


def wall_time(fn, iters=5):
    fn()
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
    assert torch.cuda.is_available(), "bench_optim_state measures on the GPU"
    S = importlib.import_module("selfsupervised-nvsf_b200.synth")
    torch.manual_seed(0)
    # bench.py's model: the KITTI-360 configuration of the reference (93.6 M parameters)
    m = pkg.NeRFNetwork(bound=S.BOUND, num_frames=S.NUM_FRAMES, time_resolution=S.TIME_RESOLUTION).train()
    opt = pkg.optim.FlatAdam(m, lr=1e-2, ema_decay=0.95)
    n_params = sum(p.numel() for p in m.parameters())
    # the reference's EMA works on its parameter tensors: here the hot-path views in the reference layout
    params = [v for k, v in m.reference_state_dict().items() if not k.startswith("aabb")]
    shadow = [p.clone() for p in params]
    omd = 1.0 - 0.95

    def torch_ema_loop():
        for s, p in zip(shadow, params):
            tmp = s - p
            tmp.mul_(omd)
            s.sub_(tmp)

    # same bits as the per-tensor ops (one update from the same start, decay past its warm-up)
    opt.ema_num_updates = 1000
    opt.ema.copy_(torch.cat([opt.flat[lo:hi] for lo, hi in opt.owned]))
    with torch.no_grad():
        opt.flat.add_(1e-3)
    opt.update_ema()
    torch_ema_loop()
    ref = {k: s for k, s in zip([k for k in m.reference_state_dict() if not k.startswith("aabb")], shadow)}
    named = opt.state_dict()["ema"]
    same = all(torch.equal(named[name].view(-1)[off:off + n], ref[key].reshape(-1))
               for key, name, off, n, _ in m._reference_keys())

    t_ema = gpu_time(opt.update_ema)
    t_loop = gpu_time(torch_ema_loop)
    sd = opt.state_dict()
    t_save = wall_time(opt.state_dict)
    t_load = wall_time(lambda: opt.load_state_dict(sd))
    name, power = card()
    print(json.dumps({
        "gpu": name, "power_limit": power, "parameters": n_params, "ema_tensors_torch_ema": len(params),
        "ema_bit_identical_to_torch_ops": same,
        "update_ema_ms": round(t_ema, 4),
        "update_ema_GBps": round(12 * opt.ema.numel() / (t_ema * 1e-3) / 1e9, 1),
        "torch_ema_loop_ms": round(t_loop, 4),
        "state_dict_ms": round(t_save, 3), "load_state_dict_ms": round(t_load, 3)}))


if __name__ == "__main__":
    main()
