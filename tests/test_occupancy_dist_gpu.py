"""2-GPU: the occupancy-grid updates that use a cell list — the full update over the trainable cells after
mark_untrained_grid and torch-ngp's partial update — sharded over two ranks (each evaluates one slice of the list
and the ranks all_gather the values) equal the single-GPU update bit for bit, and the replicas stay identical.
Needs two visible GPUs; skipped otherwise."""
import importlib
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
import torch.distributed as dist
import torch.multiprocessing as mp

import field_cases as FC

S = FC.S


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _make(pkg, dev):
    m = pkg.NeRFNetwork(device=dev, time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND,
                        min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH).eval()
    m.load_flat_params(FC.oracle_params())
    return m


def _lidar_poses(dev):
    out = []
    for seed in (0, 1, 2):
        R, t = S.random_pose(seed)
        P = np.eye(4)
        P[:3, :3], P[:3, 3] = R, t
        out.append(P)
    return torch.from_numpy(np.stack(out).astype(np.float32)).to(dev)


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    pkg = importlib.import_module("selfsupervised-nvsf_b200")
    m = _make(pkg, dev)
    n = m.cascade * m.grid_size ** 3
    g = torch.Generator(device=dev).manual_seed(3)
    noise_full = torch.rand(n, 3, device=dev, generator=g)
    noise_part = torch.rand(n // 2, 3, device=dev, generator=g)
    m.update_extra_state(0.5, cal_lidar_color=True, perturb=False, shard=False)
    m.mark_untrained_grid(lidar_poses=_lidar_poses(dev), intrinsics_lidar=(S.LIDAR_FOV_UP, S.LIDAR_FOV),
                          intrinsics_hoz_lidar=(0.0, 360.0), cal_lidar_color=True)
    start = m.occupancy_state_dict()
    res = {}
    for name, kw in (("full_marked", dict(noise=noise_full)),
                     ("partial", dict(noise=noise_part, mode="partial", seed=11))):
        m.load_occupancy_state_dict(start)
        m.update_extra_state([0.1, 0.6], cal_lidar_color=True, **kw)                 # sharded over the ranks
        sharded = [t.clone() for t in (m.density_grid(True), m.density_bitfield(True), m._grid[True]["stats"])]
        m.load_occupancy_state_dict(start)
        m.update_extra_state([0.1, 0.6], cal_lidar_color=True, shard=False, **kw)    # one GPU
        single = (m.density_grid(True), m.density_bitfield(True), m._grid[True]["stats"])
        torch.cuda.synchronize()
        res[name] = all(torch.equal(a, b) for a, b in zip(sharded, single))
        chk = torch.stack([sharded[0].double().sum(), sharded[1].double().sum()])
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        res[name + "_replicas"] = bool(torch.equal(lo, hi))
        res[name + "_occupied"] = int(torch.count_nonzero(sharded[1]))
    np.save(os.path.join(out_dir, f"res{rank}.npy"), np.array([res], dtype=object), allow_pickle=True)
    dist.destroy_process_group()


def test_sharded_marked_and_partial_updates_equal_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, port = 2, _free_port()
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        res = np.load(tmp_path / f"res{r}.npy", allow_pickle=True)[0]
        print(res)
        for name in ("full_marked", "partial"):
            assert res[name] and res[name + "_replicas"] and res[name + "_occupied"] > 0, name
