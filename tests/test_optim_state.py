"""Checkpoint and resume of FlatAdam: the Adam moments, the applied-step count and the EMA of the parameters
(torch_ema's ExponentialMovingAverage in the reference trainer, trainer.py:112-114), in the native layout
(keyed by parameter name, any world size) and in the reference checkpoint's "optimizer" / "ema" entries
(utils.py:610-680), whose parameter groups and order are pinned by tests/golden/state_dict_manifest.json.

torch_ema is not a dependency: its update is restated below as the three tensor ops it runs."""
import importlib
import json
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import field_cases as FC
from conftest import GOLDEN

S = FC.S
BETAS, EPS = (0.9, 0.99), 1e-15
SMALL_CPU = dict(device="cpu", log2_hashmap_size=8, hash_size_dynamic=(6, 5, 5), flow_log2_hashmap_size=8,
                 base_resolution=16, max_resolution=64, min_resolution=4, time_resolution=2, num_frames=4,
                 flow_base_resolution=4, flow_max_resolution=32)
SMALL_GPU = dict(log2_hashmap_size=12, hash_size_dynamic=(10, 9, 9), flow_log2_hashmap_size=11,
                 time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND, min_near=S.MIN_NEAR,
                 min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
FULL = dict(time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND, min_near=S.MIN_NEAR,
            min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)


@pytest.fixture(scope="module")
def manifest():
    return json.load(open(os.path.join(GOLDEN, "state_dict_manifest.json")))


def _pkg():
    return importlib.import_module("selfsupervised-nvsf_b200")


def _omd(decay, num_updates):
    """torch_ema's 1 - decay of update number `num_updates` (1-based)."""
    return 1.0 - min(decay, (1 + num_updates) / (10 + num_updates))


class TorchEma:
    """torch_ema.ExponentialMovingAverage(params, decay) as the reference trainer uses it."""

    def __init__(self, params, decay):
        self.params, self.decay, self.num_updates = list(params), decay, 0
        self.shadow = [p.detach().clone() for p in self.params]

    @torch.no_grad()
    def update(self):
        self.num_updates += 1
        omd = _omd(self.decay, self.num_updates)
        for s, p in zip(self.shadow, self.params):
            tmp = s - p
            tmp.mul_(omd)
            s.sub_(tmp)

    def state_dict(self):
        return {"decay": self.decay, "num_updates": self.num_updates, "shadow_params": self.shadow,
                "collected_params": None}


def _exact_adam(opt, lr, grad_scale, found):
    """An injected FlatAdam step for the CPU tests of the collective choreography: Adam written with
    separately rounded element-wise ops only, so the result does not depend on how a range is sliced."""
    if found is not None and float(found) != 0.0:
        opt.state[3] = 1.0
        return
    opt.state[0] += 1
    b1, b2 = opt.betas
    for off, moff, k, scale in opt.launches:
        g = opt.sync.flat[off:off + k] * grad_scale
        m, v = opt.exp_avg[moff:moff + k], opt.exp_avg_sq[moff:moff + k]
        m.mul_(b1).add_(g * (1 - b1))
        v.mul_(b2).add_(g * g * (1 - b2))
        opt.flat[off:off + k].sub_(m / (v.sqrt() + opt.eps) * (lr * scale))


@torch.no_grad()
def _torch_ema_update(opt):
    """FlatAdam.update_ema() with torch_ema's tensor ops over the owned ranges (the CPU stand-in for the kernel)."""
    opt.ema_num_updates += 1
    omd = _omd(opt.ema_decay, opt.ema_num_updates)
    for _, lo, hi, s in opt._owned_parts(opt.ema):
        tmp = s - opt.flat[lo:hi]
        tmp.mul_(omd)
        s.sub_(tmp)


# ---------------------------------------------------------------------------------------------- CPU: layouts
def test_reference_param_groups_are_the_manifest_groups(manifest):
    m = _pkg().NeRFNetwork(device="cpu", **FULL)
    got = m.reference_param_groups()
    assert [g["params"] for g in got] == [g["params"] for g in manifest["optimizer_groups"]]
    assert [g["lr"] for g in got] == pytest.approx([g["lr"] for g in manifest["optimizer_groups"]])


def test_reference_parameters_are_the_manifest_keys_without_buffers(manifest):
    m = _pkg().NeRFNetwork(device="cpu", **FULL)
    want = [(k, tuple(s)) for k, s, _ in manifest["keys"] if k not in ("aabb_train", "aabb_infer")]
    assert [(k, tuple(s)) for k, s in m.reference_parameters()] == want


def _manifest_adam(manifest, steps, seed=0):
    """torch.optim.Adam over manifest-shaped tensors with the reference's groups, after `steps` random steps."""
    gen = torch.Generator().manual_seed(seed)
    shapes = {k: tuple(s) for k, s, _ in manifest["keys"]}
    tensors = {k: torch.nn.Parameter(torch.randn(shapes[k], generator=gen))
               for g in manifest["optimizer_groups"] for k in g["params"]}
    adam = torch.optim.Adam([{"params": [tensors[k] for k in g["params"]], "lr": 1e-2 * g["lr"]}
                             for g in manifest["optimizer_groups"]], betas=BETAS, eps=EPS)
    for _ in range(steps):
        _random_grads(tensors, gen)
        adam.step()
    return tensors, adam, gen


def _random_grads(tensors, gen):
    for t in tensors.values():
        t.grad = torch.randn(t.shape, generator=gen) if t.numel() else None   # tcnn view encodings: no grad


def test_reference_optimizer_state_round_trip_cpu(manifest):
    pkg = _pkg()
    tensors, adam, gen = _manifest_adam(manifest, steps=2)
    sd = adam.state_dict()
    opt = pkg.optim.FlatAdam(pkg.NeRFNetwork(device="cpu", **FULL), lr=0.5)
    opt.load_reference_optimizer_state({"optimizer": sd, "model": {}})
    assert opt.applied_steps() == 2 and opt.step_count == 2 and opt.lr == pytest.approx(1e-2)
    out = opt.reference_optimizer_state_dict()
    assert sorted(out["state"]) == sorted(sd["state"])
    for i, st in sd["state"].items():
        assert float(out["state"][i]["step"]) == float(st["step"])
        for k in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(out["state"][i][k], st[k]), (i, k)
    for a, b in zip(out["param_groups"], sd["param_groups"]):
        assert a["params"] == b["params"] and a["lr"] == pytest.approx(b["lr"], rel=1e-12)
        assert tuple(a["betas"]) == tuple(b["betas"]) and a["eps"] == b["eps"] and a["weight_decay"] == 0
    # the export loads into a fresh torch.optim.Adam of the reference's structure and continues like the original
    fresh_t = {k: torch.nn.Parameter(t.detach().clone()) for k, t in tensors.items()}
    fresh = torch.optim.Adam([{"params": [fresh_t[k] for k in g["params"]], "lr": 0.0}
                              for g in manifest["optimizer_groups"]], betas=BETAS, eps=EPS)
    fresh.load_state_dict(out)
    _random_grads(tensors, gen)
    for k, t in tensors.items():
        fresh_t[k].grad = None if t.grad is None else t.grad.clone()
    adam.step()
    fresh.step()
    for k in tensors:
        assert torch.equal(fresh_t[k], tensors[k]), k
    # one common step, matching betas / eps
    bad = adam.state_dict()
    bad["state"][0]["step"] = torch.tensor(7.0)
    with pytest.raises(pkg._lib.NvsfError):
        opt.load_reference_optimizer_state(bad)
    bad = adam.state_dict()
    bad["param_groups"][3]["betas"] = (0.9, 0.999)
    with pytest.raises(pkg._lib.NvsfError):
        opt.load_reference_optimizer_state(bad)


def test_reference_ema_state_round_trip_cpu():
    pkg = _pkg()
    m = pkg.NeRFNetwork(device="cpu", **FULL)
    ref = m.reference_parameters()
    gen = torch.Generator().manual_seed(3)
    sd = {"decay": 0.97, "num_updates": 12, "collected_params": None,
          "shadow_params": [torch.randn(s, generator=gen) for _, s in ref]}
    opt = pkg.optim.FlatAdam(m, ema_decay=0.5)
    opt.load_reference_ema_state({"ema": sd})
    assert opt.ema_decay == 0.97 and opt.ema_num_updates == 12
    out = opt.reference_ema_state_dict()
    assert set(out) == {"decay", "num_updates", "shadow_params", "collected_params"}
    assert out["decay"] == 0.97 and out["num_updates"] == 12 and out["collected_params"] is None
    hot = {k for k, *_ in m._reference_keys()}
    assert len(out["shadow_params"]) == len(ref)
    for (k, s), a, b in zip(ref, out["shadow_params"], sd["shadow_params"]):
        assert tuple(a.shape) == tuple(s), k
        # parameters the B200 model does not have come back as zeros
        assert torch.equal(a, b) if k in hot else not a.any(), k
    with pytest.raises(pkg._lib.NvsfError):   # count checked
        opt.load_reference_ema_state(dict(sd, shadow_params=sd["shadow_params"][:-1]))
    shadow = list(sd["shadow_params"])
    shadow[-1] = shadow[-1][:-4]
    with pytest.raises(pkg._lib.NvsfError):   # shapes checked
        opt.load_reference_ema_state(dict(sd, shadow_params=shadow))
    with pytest.raises(pkg._lib.NvsfError):   # no EMA without ema_decay
        pkg.optim.FlatAdam(pkg.NeRFNetwork(**SMALL_CPU)).load_reference_ema_state(sd)


def test_native_state_dict_rejects_foreign_states():
    pkg = _pkg()
    opt = pkg.optim.FlatAdam(pkg.NeRFNetwork(**SMALL_CPU), ema_decay=0.9, step_fn=_exact_adam)
    sd = opt.state_dict()
    assert set(sd["exp_avg"]) == set(opt.names) and sd["step"] == 0 and sd["ema_num_updates"] == 0
    for n, t in sd["ema"].items():
        assert torch.equal(t, getattr(opt.model, n).detach()), n
    bad = dict(sd, exp_avg=dict(sd["exp_avg"]))
    bad["exp_avg"]["sigma_net"] = bad["exp_avg"]["sigma_net"][:-4]
    with pytest.raises(pkg._lib.NvsfError):
        opt.load_state_dict(bad)
    bad = dict(sd, exp_avg_sq=dict(sd["exp_avg_sq"]))
    bad["exp_avg_sq"]["sigma"] = bad["exp_avg_sq"].pop("sigma_net")
    with pytest.raises(pkg._lib.NvsfError):
        opt.load_state_dict(bad)
    with pytest.raises(pkg._lib.NvsfError):
        opt.load_state_dict(dict(sd, ema=None))
    with pytest.raises(pkg._lib.NvsfError):
        opt.load_state_dict(dict(sd, eps=1e-8))
    with pytest.raises(pkg._lib.NvsfError):
        with pkg.optim.FlatAdam(pkg.NeRFNetwork(**SMALL_CPU)).ema_weights():
            pass


# ---------------------------------------------------------------------------------------------- CPU: gloo world 2
WORLD, STEPS, BAD_STEP, DECAY = 2, 4, 1, 0.9


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _grads(model, it, rank):
    g = torch.Generator().manual_seed(1000 * it + rank)
    out = {n: torch.randn(p.shape, generator=g) for n, p in model.named_parameters()}
    if it == BAD_STEP and rank == WORLD - 1:
        out["flow_mlp"].view(-1)[3] = float("inf")
    return out


def _history(opt, rank, world):
    """STEPS injected steps + EMA updates; rank `rank` of `world` contributes its own gradients (world 1: the
    average of all WORLD ranks' gradients, bit for bit what the reduce-scatter average gives)."""
    for it in range(STEPS):
        opt.zero_grad()
        if world == 1:
            gs = [_grads(opt.model, it, r) for r in range(WORLD)]
            for n, p in opt.model.named_parameters():
                p.grad.copy_(sum(g[n] for g in gs).mul_(1.0 / WORLD))
        else:
            for n, g in _grads(opt.model, it, rank).items():
                getattr(opt.model, n).grad.copy_(g)
        for grp in _pkg().dist.GROUPS:
            opt.sync.reduce_group(grp)
        opt.sync.wait()
        opt.step(lr=1e-2 * (it + 1))
        _torch_ema_update(opt)


def _same_state(a, b):
    ok = all(a[k] == b[k] for k in ("step", "lr", "eps", "ema_decay", "ema_num_updates"))
    ok = ok and tuple(a["betas"]) == tuple(b["betas"])
    for key in ("exp_avg", "exp_avg_sq", "ema"):
        ok = ok and set(a[key]) == set(b[key]) and all(torch.equal(a[key][n], b[key][n]) for n in a[key])
    return ok


def _worker_state(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    pkg = _pkg()
    one = torch.load(os.path.join(out_dir, "world1.pt"))
    res = {}
    torch.manual_seed(0)
    opt = pkg.optim.FlatAdam(pkg.NeRFNetwork(**SMALL_CPU), lr=1e-2, shard=True, skip_nonfinite=True,
                             step_fn=_exact_adam, ema_decay=DECAY)
    _history(opt, rank, world)
    res["applied"] = opt.applied_steps()
    # (1) the sharded state_dict (a collective) is the world-1 state of the same history
    res["sharded_equals_world1"] = _same_state(opt.state_dict(), one)
    # (2) a world-1 state loads on world 2 into this rank's slices
    torch.manual_seed(1)
    opt2 = pkg.optim.FlatAdam(pkg.NeRFNetwork(**SMALL_CPU), lr=3.0, shard=True, skip_nonfinite=True,
                              step_fn=_exact_adam, ema_decay=0.5)
    opt2.load_state_dict(one)
    res["loaded_slices"] = all(torch.equal(getattr(opt2, k), getattr(opt, k)) for k in ("exp_avg", "exp_avg_sq", "ema"))
    res["loaded_scalars"] = (opt2.applied_steps() == opt.applied_steps() and opt2.step_count == opt.applied_steps()
                             and opt2.lr == opt.last_lr and opt2.ema_num_updates == STEPS and opt2.ema_decay == DECAY)
    # (3) ema_weights(): every rank holds the FULL EMA parameters inside, the exact parameters after
    before = {n: p.detach().clone() for n, p in opt.model.named_parameters()}
    with opt.ema_weights():
        res["inside"] = all(torch.equal(p.detach(), one["ema"][n]) for n, p in opt.model.named_parameters())
        res["differs"] = any(not torch.equal(p.detach(), before[n]) for n, p in opt.model.named_parameters())
    res["restored"] = all(torch.equal(p.detach(), before[n]) for n, p in opt.model.named_parameters())
    np.save(os.path.join(out_dir, f"res{rank}.npy"), np.array([res], dtype=object), allow_pickle=True)
    dist.destroy_process_group()


def test_sharded_state_dict_and_ema_weights_gloo_world2(tmp_path):
    pkg = _pkg()
    torch.manual_seed(0)
    one = pkg.optim.FlatAdam(pkg.NeRFNetwork(**SMALL_CPU), lr=1e-2, skip_nonfinite=True, step_fn=_exact_adam,
                             ema_decay=DECAY)
    _history(one, 0, 1)
    assert one.applied_steps() == STEPS - 1
    torch.save(one.state_dict(), tmp_path / "world1.pt")
    mp.spawn(_worker_state, args=(WORLD, _free_port(), str(tmp_path)), nprocs=WORLD, join=True)
    for r in range(WORLD):
        res = np.load(tmp_path / f"res{r}.npy", allow_pickle=True)[0]
        assert res == {"applied": STEPS - 1, "sharded_equals_world1": True, "loaded_slices": True,
                       "loaded_scalars": True, "inside": True, "differs": True, "restored": True}, (r, res)


# ---------------------------------------------------------------------------------------------- GPU
def _inject(opt, it, bad=False):
    """Gradients of step `it` (rendered gradients use atomics and are not bit-reproducible)."""
    g = torch.Generator(device="cuda").manual_seed(100 + it)
    opt.zero_grad()
    for n, p in opt.model.named_parameters():
        p.grad.copy_(torch.randn(p.shape, generator=g, device="cuda"))
    if bad:
        opt.model.planes_camera.grad.view(-1)[11] = float("inf")


@pytest.mark.gpu
def test_ema_update_kernel_is_torch_ema(pkg):
    L = pkg._lib.lib()
    g = torch.Generator(device="cuda").manual_seed(0)
    n = 1 << 20
    p = torch.randn(n, generator=g, device="cuda")
    s = p.clone()
    ref = s.clone()
    for t in range(1, 6):    # decay warm-up: min(0.999, (1+t)/(10+t)) is still rising
        p.add_(torch.randn(n, generator=g, device="cuda"))
        omd = _omd(0.999, t)
        assert pkg._lib.check(L.nvsf_ema_update(s.data_ptr(), p.data_ptr(), n, omd, None), "ema") is None
        tmp = ref - p
        tmp.mul_(omd)
        ref.sub_(tmp)
        torch.cuda.synchronize()
        assert torch.equal(s, ref), t
    x = torch.zeros(16, device="cuda")
    assert L.nvsf_ema_update(x.data_ptr() + 4, x.data_ptr(), 8, 0.1, None) == -1      # misaligned shadow
    assert L.nvsf_ema_update(x.data_ptr(), x.data_ptr() + 4, 8, 0.1, None) == -1      # misaligned params
    assert L.nvsf_ema_update(x.data_ptr(), x.data_ptr(), 6, 0.1, None) == -1          # not a multiple of 4
    assert L.nvsf_ema_update(None, x.data_ptr(), 8, 0.1, None) == -1
    assert L.nvsf_ema_update(None, None, 0, 0.1, None) == 0


def _gpu_opt(pkg, seed=0):
    torch.manual_seed(seed)
    m = pkg.NeRFNetwork(**SMALL_GPU).train()
    return pkg.optim.FlatAdam(m, lr=1e-2, skip_nonfinite=True, ema_decay=0.95)


@pytest.mark.gpu
def test_resume_is_bit_exact(pkg, tmp_path):
    K, M, BAD = 4, 3, 1

    def run(opt, steps):
        for it in steps:
            _inject(opt, it, bad=it == BAD)
            opt.step(lr=1e-2 / (1 + it))
            opt.update_ema()

    a = _gpu_opt(pkg)
    run(a, range(K + M))
    b = _gpu_opt(pkg)
    run(b, range(K))
    torch.save({"model": b.model.state_dict(), "optimizer": b.state_dict()}, tmp_path / "ckpt.pt")
    ck = torch.load(tmp_path / "ckpt.pt")
    c = _gpu_opt(pkg, seed=7)
    c.model.load_state_dict(ck["model"])
    c.load_state_dict(ck["optimizer"])
    run(c, range(K, K + M))
    torch.cuda.synchronize()
    assert a.applied_steps() == c.applied_steps() == K + M - 1
    for k in ("flat", "exp_avg", "exp_avg_sq", "ema"):
        assert torch.equal(getattr(a, k), getattr(c, k)), k
    assert a.ema_num_updates == c.ema_num_updates == K + M


@pytest.mark.gpu
def test_reference_resume_matches_torch_adam_and_ema(pkg, manifest):
    from test_checkpoint import reference_layout_state_dict
    K, M = 3, 2
    sd = reference_layout_state_dict(FC.oracle_params(), manifest)
    tensors = {k: torch.nn.Parameter(sd[k].clone().cuda())
               for k, _, _ in manifest["keys"] if k not in ("aabb_train", "aabb_infer")}
    adam = torch.optim.Adam([{"params": [tensors[k] for k in g["params"]], "lr": 1e-2 * g["lr"]}
                             for g in manifest["optimizer_groups"]], betas=BETAS, eps=EPS)
    ema = TorchEma(tensors.values(), 0.95)      # over model.parameters(): the manifest order without buffers
    m = pkg.NeRFNetwork(**FULL).train()
    slices = {k: (name, off, n) for k, name, off, n, _ in m._reference_keys()}

    def grads(it):
        g = torch.Generator(device="cuda").manual_seed(200 + it)
        return {k: torch.randn(tensors[k].shape, generator=g, device="cuda") for k in slices}

    def ref_step(it):
        for k, gk in grads(it).items():
            tensors[k].grad = gk
        adam.step()
        ema.update()

    for it in range(K):
        ref_step(it)
    m.load_reference_state_dict({"model": dict({k: t.detach() for k, t in tensors.items()},
                                               aabb_train=sd["aabb_train"], aabb_infer=sd["aabb_infer"])})
    opt = pkg.optim.FlatAdam(m, lr=1e-2, ema_decay=0.5)
    opt.load_reference_optimizer_state({"optimizer": adam.state_dict()})
    opt.load_reference_ema_state({"ema": ema.state_dict()})
    for it in range(K, K + M):
        ref_step(it)
        opt.zero_grad()
        for k, gk in grads(it).items():
            name, off, n = slices[k]
            getattr(m, name).grad.view(-1)[off:off + n].copy_(gk.reshape(-1))
        opt.step()
        opt.update_ema()
    mine = m.reference_state_dict()
    shadow = dict(zip((k for k, _ in m.reference_parameters()), opt.reference_ema_state_dict()["shadow_params"]))
    ref_shadow = dict(zip(tensors, ema.shadow))
    for k in slices:
        np.testing.assert_allclose(mine[k].cpu().numpy(), tensors[k].detach().cpu().numpy(), rtol=2e-5, atol=1e-7,
                                   err_msg=k)
        np.testing.assert_allclose(shadow[k].cpu().numpy(), ref_shadow[k].cpu().numpy(), rtol=2e-5, atol=1e-7,
                                   err_msg="ema " + k)
    assert opt.applied_steps() == K + M and opt.ema_num_updates == K + M


@pytest.mark.gpu
def test_render_with_ema_weights(pkg):
    opt = _gpu_opt(pkg)
    for it in range(3):
        _inject(opt, it)
        opt.step(lr=1e-3)
        opt.update_ema()
    m = opt.model.eval()
    o, d = S.lidar_rays(2048, seed=4)
    o, d = torch.from_numpy(o).cuda()[None], torch.from_numpy(d).cuda()[None]
    t = torch.tensor([[0.4]], device="cuda")

    def render(model):
        with torch.no_grad():
            r = model.render(o, d, t, cal_lidar_color=True, staged=True, num_steps=64)
        return torch.cat([r["depth_lidar"].reshape(-1), r["image_lidar"].reshape(-1)])

    before = render(m)
    torch.manual_seed(5)
    shadow_model = pkg.NeRFNetwork(**SMALL_GPU).eval()
    with torch.no_grad():
        for n, v in opt.state_dict()["ema"].items():
            getattr(shadow_model, n).copy_(v)
    with opt.ema_weights():
        inside = render(m)
    after = render(m)
    assert torch.equal(inside, render(shadow_model))
    assert not torch.equal(inside, before)
    assert torch.equal(after, before)


def _worker_nccl(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    pkg = _pkg()
    small = dict(SMALL_GPU, device=dev)
    opts = []
    for shard in (False, True):
        torch.manual_seed(0)
        opts.append(pkg.optim.FlatAdam(pkg.NeRFNetwork(**small).train(), lr=1e-2, shard=shard, skip_nonfinite=True,
                                       ema_decay=0.95))
    for it in range(4):
        g = torch.Generator(device=dev).manual_seed(10 * it + rank)
        grads = {n: torch.randn(p.shape, generator=g, device=dev) for n, p in opts[0].model.named_parameters()}
        if it == 2 and rank == world - 1:
            grads["planes_camera"].view(-1)[7] = float("inf")
        for opt in opts:
            opt.zero_grad()
            for n, v in grads.items():
                getattr(opt.model, n).grad.copy_(v)
            for grp in pkg.dist.GROUPS:
                opt.sync.reduce_group(grp)
            opt.sync.wait()
            opt.step()
            opt.update_ema()
    full, sharded = opts[0].state_dict(), opts[1].state_dict()
    torch.cuda.synchronize()
    res = {"step": (full["step"], sharded["step"])}
    # the two paths differ only in the summation order of the gradient reduction
    res["diff"] = max(float((full[k][n] - sharded[k][n]).abs().max())
                      for k in ("exp_avg", "exp_avg_sq", "ema") for n in full[k])
    np.save(os.path.join(out_dir, f"res{rank}.npy"), np.array([res], dtype=object), allow_pickle=True)
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_state_dict_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mp.spawn(_worker_nccl, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        res = np.load(tmp_path / f"res{r}.npy", allow_pickle=True)[0]
        assert res["step"] == (3, 3) and res["diff"] < 1e-6, res
