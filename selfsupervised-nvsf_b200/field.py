"""Host side of the B200 field + uniform renderer: mirrors the reference's model interface.

`NeRFNetwork` here presents the surface of the reference's
``nvsf.nerf.models.network_dynamic.NeRFNetwork`` (which subclasses ``NeRFRenderer``,
renderer_dynamic.py:67-326) for the hot path:

    density(x, t, cal_lidar_color)           -> {"sigma", "geo_feat"}     network_dynamic.py:213-287
    flow(x, t)                               -> {"flow_forward", "flow_backward"}         :197-211
    color(x, d, geo_feat, mask, cal_lidar_color) -> [N, 2|3] f32                          :290-332
    run(rays_o, rays_d, time, cal_lidar_color, num_steps, upsample_steps, bg_color, perturb, **kw)
    render(rays_o, rays_d, time, cal_lidar_color, staged, max_ray_batch, **kw)
                                             -> dict with the reference's keys   renderer_dynamic.py:109-326
    update_extra_state(time, ...), run_cuda(rays_o, rays_d, time, ...)
                                             -> occupancy-grid update and the march_rays* / composite_rays*
                                                render loops around the operators of raymarching.py (the
                                                reference ships the operators but not these callers; they
                                                follow torch-ngp, where the operators come from)

Everything is computed by the sm_100a kernels behind include/nvsf_b200.h; there is no PyTorch
fallback.  Parameters are fp32 `nn.Parameter`s in the reference's own memory layouts (tcnn flat
`params`, Planes4D [1,F,H,W] tensors, nn.Linear weights), concatenated per encoder:

    hash_static_{lidar,camera}    == hash_encoder_*.hash_static.params
    hash_dynamic_{lidar,camera}   == cat(hash_encoder_*.hash_dynamic.{p}.hash_t.{k}.params  for p, k)
    planes_{lidar,camera}         == cat(planes_encoder_*.planes.{s}.{c}.flatten()       for s, c)
    flow_grid, flow_mlp           == flow_net.grid_enc.params, cat(flow_net.mlp.{0,2,4}.weight)
    sigma_net, intensity_net, raydrop_net, color_net  == the tcnn `params` of the same name
"""
import ctypes
import os
import math

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from . import raymarching
from ._lib import check, ptr, stream_ptr

MAX_LEVELS = 16
MAX_PLANE_SCALES = 8
PLANE_COMBS = [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]


class GridLevel(ctypes.Structure):
    _fields_ = [("scale", ctypes.c_float), ("res", ctypes.c_uint32), ("size", ctypes.c_uint32),
                ("offset", ctypes.c_uint32), ("hashed", ctypes.c_uint32)]


class FieldConfigC(ctypes.Structure):
    _fields_ = [
        ("bound", ctypes.c_float), ("density_scale", ctypes.c_float),
        ("active_sensor", ctypes.c_uint32), ("num_frames", ctypes.c_uint32),
        ("time_resolution", ctypes.c_uint32),
        ("hs_levels", ctypes.c_uint32), ("hs_entries", ctypes.c_uint32),
        ("hs", GridLevel * MAX_LEVELS),
        ("hd_levels", ctypes.c_uint32), ("hd_entries", ctypes.c_uint32 * 3),
        ("hd", (GridLevel * MAX_LEVELS) * 3),
        ("fl_levels", ctypes.c_uint32), ("fl_entries", ctypes.c_uint32),
        ("fl", GridLevel * MAX_LEVELS),
        ("pl_scales", ctypes.c_uint32), ("pl_res", ctypes.c_uint32 * MAX_PLANE_SCALES),
    ]


class FieldParamsC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in
                ("hash_static", "hash_dynamic", "planes", "flow_grid", "flow_mlp", "sigma_net",
                 "head_a", "head_b")]


def grid_levels(n_dims, n_levels, base_resolution, per_level_scale, log2_hashmap_size):
    """Per-level geometry of a tcnn multiresolution grid (tiny-cuda-nn GridEncoding):
    scale = exp2(l * log2(per_level_scale)) * base - 1, res = ceil(scale) + 1,
    size = min(next_multiple(res^D, 8), 2^log2_hashmap_size), hashed iff res^D > size."""
    log2_pls = np.log2(np.float32(per_level_scale), dtype=np.float32)
    out, offset = [], 0
    for l in range(n_levels):
        scale = np.float32(np.exp2(np.float32(l) * log2_pls, dtype=np.float32)
                           * np.float32(base_resolution) - np.float32(1.0))
        res = int(np.ceil(scale)) + 1
        dense = res ** n_dims
        size = min((min(dense, (2 ** 32 - 1) // 2) + 7) // 8 * 8, 1 << log2_hashmap_size)
        out.append((float(scale), res, size, offset, int(dense > size)))
        offset += size
    return out, offset


def _fill_levels(dst, levels):
    for i, (scale, res, size, offset, hashed) in enumerate(levels):
        dst[i].scale, dst[i].res, dst[i].size, dst[i].offset, dst[i].hashed = scale, res, size, offset, hashed


_L = None


def _setup_lib():
    global _L
    if _L is not None:
        return _L
    L = _lib.lib()
    P = ctypes.c_void_p
    cfgp, prmp = ctypes.POINTER(FieldConfigC), ctypes.POINTER(FieldParamsC)
    L.nvsf_field_workspace_bytes.argtypes = [cfgp]
    L.nvsf_field_pack_params.argtypes = [cfgp, prmp, ctypes.c_uint32, P, ctypes.c_size_t, P]
    L.nvsf_field_pack_time.argtypes = [cfgp, prmp, P, P, ctypes.c_size_t, P]
    L.nvsf_field_density.argtypes = [cfgp, P, P, ctypes.c_uint32, P, P, P, P, P, ctypes.c_size_t, P]
    L.nvsf_render_uniform_density.argtypes = [cfgp, P, P, P, P, P, P, ctypes.c_uint32, ctypes.c_uint32, P,
                                              ctypes.c_size_t, P]
    L.nvsf_render_uniform_composite.argtypes = [cfgp, P, ctypes.c_uint32, P, P, P, P, ctypes.c_uint32,
                                                ctypes.c_uint32, ctypes.c_float, P, ctypes.c_size_t, P, P,
                                                P, P, P, P]
    L.nvsf_render_uniform.argtypes = [cfgp, P, ctypes.c_uint32, P, P, P, P, P, ctypes.c_uint32,
                                      ctypes.c_uint32, ctypes.c_float, P, ctypes.c_size_t, P, P, P,
                                      P, P, P]
    L.nvsf_render_uniform_backward_scratch_bytes.argtypes = [cfgp, ctypes.c_uint32, ctypes.c_uint32]
    L.nvsf_render_uniform_train_forward.argtypes = [cfgp, P, ctypes.c_uint32, P, P, P, P, P, ctypes.c_uint32,
                                                    ctypes.c_uint32, ctypes.c_float, P, ctypes.c_size_t, P, P,
                                                    P, P, P, P]
    L.nvsf_render_uniform_backward.argtypes = [cfgp, P, prmp, ctypes.c_uint32, P, P, P, P, P, ctypes.c_uint32,
                                               ctypes.c_uint32, ctypes.c_float, P, ctypes.c_size_t, P, P, P, P,
                                               P, prmp, P, ctypes.c_size_t, P]
    L.nvsf_field_color.argtypes = [cfgp, P, ctypes.c_uint32, P, P, ctypes.c_uint32, ctypes.c_uint32, P,
                                   ctypes.c_uint32, P, ctypes.c_uint32, P]
    # development switches (A/B runs of the staged density evaluation): NVSF_OPT="density_mode=2,dyn_tile=8192"
    for kv in filter(None, os.environ.get("NVSF_OPT", "").split(",")):
        k, v = kv.split("=")
        check(L.nvsf_set_option(k.strip().encode(), int(v)), f"set_option({kv})")
    _L = L
    return L


PARAM_ORDER_SHARED = ("flow_grid", "flow_mlp", "sigma_net")


def _param_names(lidar):
    """Parameters a render of one modality depends on, in nvsf_field_params_t order."""
    m = "lidar" if lidar else "camera"
    return ([f"hash_static_{m}", f"hash_dynamic_{m}", f"planes_{m}"] + list(PARAM_ORDER_SHARED)
            + (["intensity_net", "raydrop_net"] if lidar else ["color_net"]))


class _RenderUniformTrain(torch.autograd.Function):
    """NeRFRenderer.run with autograd (what train_step differentiates, trainer.py:193-200,491-499):
    forward keeps the per-sample intermediates, backward calls nvsf_render_uniform_backward and
    returns the gradients of the fp32 master parameters in their own layouts.

    If a parameter already owns a contiguous `.grad` and `model.fused_grad_accumulation` is set,
    the kernels accumulate straight into it (no temporary, no extra add pass) and autograd
    receives None for that input."""

    @staticmethod
    @_lib.device_guard
    def forward(ctx, model, lidar, o, d, nears, fars, noise, S, bg, *params):
        L = _setup_lib()
        dev = o.device
        N = o.shape[0]
        nch = 2 if lidar else 3
        ws = model._ws[lidar]
        depth = torch.empty(N, dtype=torch.float32, device=dev)
        image = torch.empty(N, nch, dtype=torch.float32, device=dev)
        wsum = torch.empty(N, dtype=torch.float32, device=dev)
        weights = torch.empty(N, S, dtype=torch.float32, device=dev)
        z_vals = torch.empty(N, S, dtype=torch.float32, device=dev)
        nbytes = L.nvsf_render_uniform_saved_bytes(N, S)
        saved = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        check(L.nvsf_render_uniform_train_forward(ctypes.byref(model._cfg), ptr(ws), int(lidar), ptr(o), ptr(d),
                                                  ptr(nears), ptr(fars), ptr(noise), N, S, bg, ptr(saved),
                                                  saved.numel(), ptr(depth), ptr(image), ptr(wsum), ptr(weights),
                                                  ptr(z_vals), stream_ptr()), "render_uniform_train_forward")
        ctx.model, ctx.lidar, ctx.S, ctx.bg = model, lidar, S, bg
        ctx.tensors = (o, d, nears, fars, noise, saved, weights, ws)
        ctx.pack_gen = model._pack_gen.get(lidar, 0)
        ctx.mark_non_differentiable(z_vals)
        return depth, image, wsum, weights, z_vals

    @staticmethod
    @_lib.device_guard
    def backward(ctx, g_depth, g_image, g_wsum, g_weights, _g_z):
        with _lib.option_scope(ctx.model.options):   # the autograd thread runs under the model's own options too
            return _RenderUniformTrain._backward(ctx, g_depth, g_image, g_wsum, g_weights, _g_z)

    @staticmethod
    def _backward(ctx, g_depth, g_image, g_wsum, g_weights, _g_z):
        L = _setup_lib()
        model, lidar, S = ctx.model, ctx.lidar, ctx.S
        o, d, nears, fars, noise, saved, weights, ws = ctx.tensors
        if model._ws.get(lidar) is not ws or model._pack_gen.get(lidar, 0) != ctx.pack_gen:
            raise _lib.NvsfError("the packed field tables were rebuilt between forward and backward (another "
                                 "render / density / update_extra_state of the same modality ran in between): "
                                 "call backward() of a render before the next pack of that modality")
        dev, N = o.device, o.shape[0]
        names = _param_names(lidar)
        params = [getattr(model, n) for n in names]
        fused = bool(getattr(model, "fused_grad_accumulation", False))
        grads, ret = [], []
        for p in params:
            if fused and p.grad is not None and p.grad.is_contiguous() and p.grad.dtype == torch.float32:
                grads.append(p.grad)
                ret.append(None)
            else:
                g = torch.zeros_like(p, memory_format=torch.contiguous_format)
                grads.append(g)
                ret.append(g)
        gc = FieldParamsC()
        for field, g in zip(("hash_static", "hash_dynamic", "planes", "flow_grid", "flow_mlp", "sigma_net",
                             "head_a", "head_b"), grads + [None]):
            setattr(gc, field, ptr(g))

        def prep(g):
            return None if g is None else g.to(dtype=torch.float32).contiguous()

        g_depth, g_image, g_wsum, g_weights = prep(g_depth), prep(g_image), prep(g_wsum), prep(g_weights)
        pc = model._params_c(lidar)
        sbytes = L.nvsf_render_uniform_backward_scratch_bytes(ctypes.byref(model._cfg), N, S)
        scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
        check(L.nvsf_render_uniform_backward(ctypes.byref(model._cfg), ptr(ws), ctypes.byref(pc), int(lidar),
                                             ptr(o), ptr(d), ptr(nears), ptr(fars), ptr(noise), N, S, ctx.bg,
                                             ptr(saved), saved.numel(), ptr(weights), ptr(g_depth), ptr(g_image),
                                             ptr(g_wsum), ptr(g_weights), ctypes.byref(gc), ptr(scratch),
                                             scratch.numel(), stream_ptr()), "render_uniform_backward")
        if getattr(model, "_debug_keep", False):  # tests/tools: look at the intermediates
            model._debug = dict(saved=saved, scratch=scratch, N=N, S=S)
        ctx.tensors = None
        return (None,) * 9 + tuple(ret)


class _FlowTrain(torch.autograd.Function):
    """NeRFNetwork.flow with autograd (network_dynamic.py:197-211): the scene-flow loss of train_step
    (trainer.py:237-265) differentiates it with respect to flow_net's grid and MLP."""

    @staticmethod
    @_lib.device_guard
    def forward(ctx, model, x, flow_grid, flow_mlp):
        L = _setup_lib()
        n = x.shape[0]
        dev = x.device
        ws = model._ws[True]
        flow = torch.empty(n, 8, dtype=torch.float32, device=dev)
        flowfeat = torch.empty(n, 32, dtype=torch.float16, device=dev)
        sbytes = L.nvsf_field_flow_scratch_bytes(ctypes.byref(model._cfg), n)
        scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
        check(L.nvsf_field_flow_forward(ctypes.byref(model._cfg), ptr(ws), ptr(x), n, ptr(flow), ptr(flowfeat),
                                        ptr(scratch), sbytes, stream_ptr()), "field_flow_forward")
        ctx.model, ctx.pack_gen, ctx.tensors = model, model._pack_gen.get(True, 0), (x, flowfeat, ws, scratch)
        return flow[:, :6]

    @staticmethod
    @_lib.device_guard
    def backward(ctx, g_flow):
        with _lib.option_scope(ctx.model.options):
            return _FlowTrain._backward(ctx, g_flow)

    @staticmethod
    def _backward(ctx, g_flow):
        L = _setup_lib()
        model = ctx.model
        x, flowfeat, ws, scratch = ctx.tensors
        if model._ws.get(True) is not ws or model._pack_gen.get(True, 0) != ctx.pack_gen:
            raise _lib.NvsfError("the packed field tables were rebuilt between flow() and its backward")
        n = x.shape[0]
        dflow = torch.zeros(n, 8, dtype=torch.float32, device=x.device)
        dflow[:, :6] = g_flow.to(torch.float32)
        fused = bool(getattr(model, "fused_grad_accumulation", False))
        grads, ret = [], []
        for p in (model.flow_grid, model.flow_mlp):
            if fused and p.grad is not None and p.grad.is_contiguous() and p.grad.dtype == torch.float32:
                grads.append(p.grad)
                ret.append(None)
            else:
                g = torch.zeros_like(p, memory_format=torch.contiguous_format)
                grads.append(g)
                ret.append(g)
        check(L.nvsf_field_flow_backward(ctypes.byref(model._cfg), ptr(ws), ptr(model.flow_mlp), ptr(x), n,
                                         ptr(flowfeat), ptr(dflow), ptr(grads[0]), ptr(grads[1]), ptr(scratch),
                                         scratch.numel(), stream_ptr()), "field_flow_backward")
        ctx.tensors = None
        return None, None, ret[0], ret[1]


class NeRFNetwork(nn.Module):
    """B200 field + renderer with the reference NeRFNetwork's constructor arguments
    (network_dynamic.py:13-38; renderer kwargs renderer_dynamic.py:68-78)."""

    def __init__(self, min_resolution=32, base_resolution=512, max_resolution=32768,
                 time_resolution=25, n_levels_plane=4, n_features_per_level_plane=8,
                 n_levels_hash=8, n_features_per_level_hash=4, log2_hashmap_size=19,
                 num_layers_flow=3, hidden_dim_flow=64, num_layers_sigma=2, hidden_dim_sigma=64,
                 geo_feat_dim=15, num_layers_lidar=3, hidden_dim_lidar=64, num_layers_color=3,
                 hidden_dim_color=64, out_color_dim=3, out_lidar_color_dim=2, num_frames=51,
                 bound=1, density_scale=1, min_near=0.01, min_near_lidar=0.01,
                 lidar_max_depth=0.81, density_thresh=0.01, bg_radius=-1, active_sensor=False,
                 hash_size_dynamic=(15, 13, 13), flow_levels=16, flow_features=8,
                 flow_base_resolution=32, flow_max_resolution=8192, flow_log2_hashmap_size=18,
                 device="cuda", options=None, **kwargs):
        super().__init__()
        # per-model tuning options ({name: int}, the names of nvsf_set_option): applied around this model's launches
        # only (_lib.option_scope); None / {} = the process defaults
        self.options = dict(options) if options else {}
        fixed = dict(n_levels_plane=(n_levels_plane, 4), n_features_per_level_plane=(n_features_per_level_plane, 8),
                     n_levels_hash=(n_levels_hash, 8), n_features_per_level_hash=(n_features_per_level_hash, 4),
                     num_layers_flow=(num_layers_flow, 3), hidden_dim_flow=(hidden_dim_flow, 64),
                     num_layers_sigma=(num_layers_sigma, 2), hidden_dim_sigma=(hidden_dim_sigma, 64),
                     geo_feat_dim=(geo_feat_dim, 15), num_layers_lidar=(num_layers_lidar, 3),
                     hidden_dim_lidar=(hidden_dim_lidar, 64), num_layers_color=(num_layers_color, 3),
                     hidden_dim_color=(hidden_dim_color, 64), out_color_dim=(out_color_dim, 3),
                     out_lidar_color_dim=(out_lidar_color_dim, 2), flow_levels=(flow_levels, 16),
                     flow_features=(flow_features, 8))
        for k, (got, want) in fixed.items():
            if got != want:
                raise ValueError(f"nvsf_b200 kernels are built for {k}={want} (the reference default), got {got}")
        if bg_radius > 0:
            raise ValueError("bg_radius > 0 is not supported (the reference asserts bg_radius <= 0, main_nvsf.py:171)")
        self.bound = float(bound)
        self.cascade = 1 + math.ceil(math.log2(bound))
        self.grid_size = 128
        self.density_scale, self.min_near = float(density_scale), float(min_near)
        self.min_near_lidar, self.lidar_max_depth = float(min_near_lidar), float(lidar_max_depth)
        self.density_thresh, self.bg_radius, self.active_sensor = density_thresh, bg_radius, bool(active_sensor)
        self.out_color_dim, self.out_lidar_color_dim = 3, 2
        self.num_frames, self.time_resolution = int(num_frames), int(time_resolution)

        hash_pls = float(np.exp2(np.log2(max_resolution / base_resolution) / (n_levels_hash - 1)))
        flow_pls = float(np.exp2(np.log2(flow_max_resolution / flow_base_resolution) / (flow_levels - 1)))
        self._hs, hs_entries = grid_levels(3, 8, base_resolution, hash_pls, log2_hashmap_size)
        self._hd, hd_entries = [], []
        for h in hash_size_dynamic:
            lv, tot = grid_levels(2, 8, base_resolution, hash_pls, h)
            self._hd.append(lv)
            hd_entries.append(tot)
        self._fl, fl_entries = grid_levels(3, 16, flow_base_resolution, flow_pls, flow_log2_hashmap_size)
        self._pl_res = [min_resolution * 2 ** s for s in range(4)]

        c = FieldConfigC()
        c.bound, c.density_scale, c.active_sensor = self.bound, self.density_scale, int(self.active_sensor)
        c.num_frames, c.time_resolution = self.num_frames, self.time_resolution
        c.hs_levels, c.hs_entries = 8, hs_entries
        _fill_levels(c.hs, self._hs)
        c.hd_levels = 8
        for p in range(3):
            c.hd_entries[p] = hd_entries[p]
            _fill_levels(c.hd[p], self._hd[p])
        c.fl_levels, c.fl_entries = 16, fl_entries
        _fill_levels(c.fl, self._fl)
        c.pl_scales = 4
        for s in range(4):
            c.pl_res[s] = self._pl_res[s]
        self._cfg = c

        T = self.time_resolution
        n_planes = sum(8 * r[a] * r[b] for R in self._pl_res for r in [(R, R, R, T)] for (a, b) in PLANE_COMBS)
        sizes = dict(hash_static=hs_entries * 4, hash_dynamic=sum(T * e * 4 for e in hd_entries),
                     planes=n_planes)
        self.param_sizes = dict(sizes, flow_grid=fl_entries * 8, flow_mlp=64 * 32 + 64 * 64 + 6 * 64,
                                sigma_net=64 * 128 + 16 * 64, intensity_net=64 * 96 + 64 * 64 + 16 * 64,
                                raydrop_net=64 * 96 + 64 * 64 + 16 * 64, color_net=64 * 32 + 64 * 64 + 16 * 64)
        dev = torch.device(device)

        def table(n):  # tcnn grids: U(-1e-4, 1e-4)
            return nn.Parameter(torch.empty(n, device=dev).uniform_(-1e-4, 1e-4))

        def xavier(shapes, last_std=None):
            chunks = []
            for i, (o, k) in enumerate(shapes):
                if last_std is not None and i == len(shapes) - 1:
                    chunks.append(torch.randn(o * k, device=dev) * last_std)
                else:
                    b = math.sqrt(6.0 / (o + k))
                    chunks.append(torch.empty(o * k, device=dev).uniform_(-b, b))
            return nn.Parameter(torch.cat(chunks))

        for m in ("lidar", "camera"):
            setattr(self, f"hash_static_{m}", table(sizes["hash_static"]))
            setattr(self, f"hash_dynamic_{m}", table(sizes["hash_dynamic"]))
            chunks = []  # planes_field.py:47-50: time planes = 1, space planes U(0.1, 0.5)
            for R in self._pl_res:
                r = (R, R, R, T)
                for (a, b) in PLANE_COMBS:
                    n = 8 * r[a] * r[b]
                    chunks.append(torch.ones(n, device=dev) if 3 in (a, b)
                                  else torch.empty(n, device=dev).uniform_(0.1, 0.5))
            setattr(self, f"planes_{m}", nn.Parameter(torch.cat(chunks)))
        self.flow_grid = table(self.param_sizes["flow_grid"])
        self.flow_mlp = xavier([(64, 32), (64, 64), (6, 64)], last_std=1e-3)  # flow_field.py:103
        self.sigma_net = xavier([(64, 128), (16, 64)])
        self.intensity_net = xavier([(64, 96), (64, 64), (16, 64)])
        self.raydrop_net = xavier([(64, 96), (64, 64), (16, 64)])
        self.color_net = xavier([(64, 32), (64, 64), (16, 64)])
        self.register_buffer("aabb_train", torch.tensor([-bound, -bound, -bound, bound, bound, bound],
                                                        dtype=torch.float32, device=dev))
        self.register_buffer("aabb_infer", self.aabb_train.clone())
        self._ws = {}      # modality -> workspace tensor
        self._packed = {}  # modality -> (param versions, time key)
        self._pack_gen = {}  # modality -> number of times the workspace tables were (re)written; a training
                             # forward records it and its backward refuses to run against newer tables

    # ------------------------------------------------------------------ parameters
    def load_flat_params(self, p):
        """Load parameters given in the layout of this module's docstring
        ({'lidar': {...}, 'camera': {...}, 'flow_grid': ..., ...})."""
        with torch.no_grad():
            for m in ("lidar", "camera"):
                for k in ("hash_static", "hash_dynamic", "planes"):
                    getattr(self, f"{k}_{m}").copy_(torch.as_tensor(p[m][k]))
            for k in ("flow_grid", "flow_mlp", "sigma_net", "intensity_net", "raydrop_net", "color_net"):
                getattr(self, k).copy_(torch.as_tensor(p[k]))
        self._packed.clear()

    # reference checkpoint keys (Trainer.save_checkpoint stores model.state_dict() under "model",
    # nvsf/nerf/utils.py:610-650; key names pinned by tests/golden/state_dict_manifest.json)
    def _reference_keys(self):
        """[(reference key, parameter name, offset, numel, shape)] in this module's concatenation order."""
        T = self.time_resolution
        out = []
        for m in ("lidar", "camera"):
            out.append((f"hash_encoder_{m}.hash_static.params", f"hash_static_{m}", 0,
                        self.param_sizes["hash_static"], (self.param_sizes["hash_static"],)))
            off = 0
            for p in range(3):
                per = self._cfg.hd_entries[p] * 4
                for k in range(T):
                    out.append((f"hash_encoder_{m}.hash_dynamic.{p}.hash_t.{k}.params", f"hash_dynamic_{m}", off, per,
                                (per,)))
                    off += per
            off = 0
            for s, R in enumerate(self._pl_res):
                r = (R, R, R, T)
                for c, (a, b) in enumerate(PLANE_COMBS):
                    n = 8 * r[a] * r[b]
                    out.append((f"planes_encoder_{m}.planes.{s}.{c}", f"planes_{m}", off, n, (1, 8, r[b], r[a])))
                    off += n
        out.append(("flow_net.grid_enc.params", "flow_grid", 0, self.param_sizes["flow_grid"],
                    (self.param_sizes["flow_grid"],)))
        off = 0
        for li, (o, k) in zip((0, 2, 4), ((64, 32), (64, 64), (6, 64))):
            out.append((f"flow_net.mlp.{li}.weight", "flow_mlp", off, o * k, (o, k)))
            off += o * k
        for n in ("sigma_net", "intensity_net", "raydrop_net", "color_net"):
            out.append((f"{n}.params", n, 0, self.param_sizes[n], (self.param_sizes[n],)))
        return out

    def load_reference_state_dict(self, state_dict, strict=True):
        """Load a checkpoint of the REFERENCE model: `torch.load(path)["model"]` (or the bare state
        dict) as written by Trainer.save_checkpoint (utils.py:610-650) / read by load_checkpoint
        (:682-747).  Returns (missing_keys, unexpected_keys) like nn.Module.load_state_dict; keys of
        modules outside the hot path (the un-suffixed planes_encoder / hash_encoder that the reference
        constructs but never optimises, view encoders without parameters, the U-Net, aabb buffers,
        density grids) are reported as unexpected and ignored."""
        sd = state_dict.get("model", state_dict) if isinstance(state_dict, dict) else state_dict
        used, missing = set(), []
        with torch.no_grad():
            for key, name, off, n, shape in self._reference_keys():
                if key not in sd:
                    missing.append(key)
                    continue
                v = sd[key]
                if tuple(v.shape) != tuple(shape):
                    raise _lib.NvsfError(f"{key}: checkpoint shape {tuple(v.shape)} != {tuple(shape)}")
                getattr(self, name).view(-1)[off:off + n].copy_(v.reshape(-1).to(torch.float32))
                used.add(key)
            for key in ("aabb_train", "aabb_infer"):
                if key in sd:
                    getattr(self, key).copy_(sd[key].to(torch.float32))
                    used.add(key)
        self._packed.clear()
        unexpected = [k for k in sd.keys() if k not in used]
        if strict and missing:
            raise _lib.NvsfError(f"reference checkpoint lacks {len(missing)} keys, e.g. {missing[:3]}")
        return missing, unexpected

    def reference_state_dict(self):
        """The hot-path parameters under the reference's state_dict keys and shapes (the inverse of
        load_reference_state_dict; tensors are views of this module's parameters)."""
        out = {"aabb_train": self.aabb_train, "aabb_infer": self.aabb_infer}
        for key, name, off, n, shape in self._reference_keys():
            out[key] = getattr(self, name).detach().view(-1)[off:off + n].view(*shape)
        return out

    def get_params(self, lr):
        """Optimizer parameter groups of the reference (network_dynamic.py:335-357): encoders, sigma_net
        and color_net at lr; flow_net, intensity_net and raydrop_net at 0.1 lr."""
        g = lambda names, f: {"params": [getattr(self, n) for n in names], "lr": f * lr}
        return [g(["planes_lidar"], 1.0), g(["hash_static_lidar", "hash_dynamic_lidar"], 1.0),
                g(["planes_camera"], 1.0), g(["hash_static_camera", "hash_dynamic_camera"], 1.0),
                g(["flow_grid", "flow_mlp"], 0.1), g(["sigma_net"], 1.0), g(["intensity_net"], 0.1),
                g(["raydrop_net"], 0.1), g(["color_net"], 1.0)]

    def reference_param_groups(self):
        """The reference optimiser's 11 parameter groups (network_dynamic.py:335-357) as
        [{"params": [reference key, ...], "lr": lr factor}]: get_params' groups under the reference's
        checkpoint keys, plus the groups of the zero-size tcnn view encodings after the four encoder
        groups.  Pinned by tests/golden/state_dict_manifest.json ("optimizer_groups")."""
        name_of = {id(p): n for n, p in self.named_parameters()}
        keys_of = {}
        for key, name, _, _, _ in self._reference_keys():
            keys_of.setdefault(name, []).append(key)
        groups = [{"params": [k for p in g["params"] for k in keys_of[name_of[id(p)]]], "lr": g["lr"]}
                  for g in self.get_params(1.0)]
        groups[4:4] = [{"params": [f"view_encoder_{m}.params"], "lr": 1.0} for m in ("lidar", "camera")]
        return groups

    def reference_parameters(self):
        """[(reference key, shape)] of every parameter of the reference model in its `model.parameters()`
        order (the order of torch_ema's shadow_params): the state_dict keys without the aabb buffers.
        Besides the hot-path keys of _reference_keys this lists the un-suffixed planes_encoder /
        hash_encoder (shaped like the _lidar ones) and the (0,) view encodings, which the reference
        constructs but never reads or optimises."""
        hot = [(k, tuple(s)) for k, _, _, _, s in self._reference_keys()]
        pick = lambda *prefixes: [(k, s) for k, s in hot if k.startswith(prefixes)]
        enc = lambda m: pick(f"planes_encoder_{m}.") + pick(f"hash_encoder_{m}.")
        return ([(k.replace("_lidar.", ".", 1), s) for k, s in enc("lidar")] + enc("lidar") + enc("camera")
                + [("view_encoder_lidar.params", (0,))]
                + pick("flow_net.", "sigma_net.", "intensity_net.", "raydrop_net.")
                + [("view_encoder_camera.params", (0,))] + pick("color_net."))

    def _params_c(self, lidar):
        m = "lidar" if lidar else "camera"
        ps = FieldParamsC()
        ps.hash_static = ptr(getattr(self, f"hash_static_{m}"))
        ps.hash_dynamic = ptr(getattr(self, f"hash_dynamic_{m}"))
        ps.planes = ptr(getattr(self, f"planes_{m}"))
        ps.flow_grid, ps.flow_mlp, ps.sigma_net = ptr(self.flow_grid), ptr(self.flow_mlp), ptr(self.sigma_net)
        if lidar:
            ps.head_a, ps.head_b = ptr(self.intensity_net), ptr(self.raydrop_net)
        else:
            ps.head_a, ps.head_b = ptr(self.color_net), None
        return ps

    def _version_key(self, lidar):
        m = "lidar" if lidar else "camera"
        names = [f"hash_static_{m}", f"hash_dynamic_{m}", f"planes_{m}", "flow_grid", "flow_mlp", "sigma_net"]
        names += ["intensity_net", "raydrop_net"] if lidar else ["color_net"]
        return tuple((getattr(self, n)._version, getattr(self, n).data_ptr()) for n in names)

    def prepare(self, time, lidar, force=False):
        """Pack parameters (if they changed) and collapse the time-dependent tables for `time`
        (a float or the reference's [1,1] tensor; no host sync when it is a CUDA tensor)."""
        L = _setup_lib()
        dev = self.sigma_net.device
        nbytes = L.nvsf_field_workspace_bytes(ctypes.byref(self._cfg))
        if nbytes == 0:
            raise _lib.NvsfError("unsupported field configuration")
        ws = self._ws.get(lidar)
        if ws is None or ws.numel() < nbytes or ws.device != dev:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self._ws[lidar] = ws
            force = True
        if torch.is_tensor(time):
            t_dev = time.detach().to(device=dev, dtype=torch.float32).reshape(-1)[:1].contiguous()
            t_key = None  # unknown value on the host: always re-collapse (cheap)
        else:
            t_dev = torch.tensor([float(time)], dtype=torch.float32, device=dev)
            t_key = float(time)
        vkey = self._version_key(lidar)
        prev = self._packed.get(lidar)
        pc = self._params_c(lidar)
        st = stream_ptr()
        if force or prev is None or prev[0] != vkey:
            check(L.nvsf_field_pack_params(ctypes.byref(self._cfg), ctypes.byref(pc), int(lidar), ptr(ws),
                                           ws.numel(), st), "field_pack_params")
            prev = None
            self._pack_gen[lidar] = self._pack_gen.get(lidar, 0) + 1
        if prev is None or t_key is None or prev[1] != t_key:
            check(L.nvsf_field_pack_time(ctypes.byref(self._cfg), ctypes.byref(pc), ptr(t_dev), ptr(ws),
                                         ws.numel(), st), "field_pack_time")
            self._pack_gen[lidar] = self._pack_gen.get(lidar, 0) + 1
        self._packed[lidar] = (vkey, t_key)
        return ws

    # ------------------------------------------------------------------ field API
    def _density_raw(self, x, t, lidar, want_features=False, want_flow=False, prepared=False):
        """`prepared`: the caller has just run prepare(t, lidar) itself (a frame time given as a CUDA tensor is
        re-collapsed by every prepare() because its value is unknown on the host: once per frame is enough)."""
        L = _setup_lib()
        x = x.detach().to(device=self.sigma_net.device, dtype=torch.float32).contiguous().view(-1, 3)
        n = x.shape[0]
        ws = self._ws[lidar] if prepared and self._ws.get(lidar) is not None else self.prepare(t, lidar)
        sigma = torch.empty(n, dtype=torch.float32, device=x.device)
        geo = torch.empty(n, 16, dtype=torch.float16, device=x.device)
        feats = torch.empty(n, 128, dtype=torch.float16, device=x.device) if want_features else None
        flow = torch.empty(n, 6, dtype=torch.float32, device=x.device) if want_flow else None
        sbytes = L.nvsf_field_density_scratch_bytes(n)
        scratch = torch.empty(max(sbytes, 16), dtype=torch.uint8, device=x.device)
        check(L.nvsf_field_density(ctypes.byref(self._cfg), ptr(ws), ptr(x), n, ptr(sigma), ptr(geo),
                                   ptr(feats), ptr(flow), ptr(scratch), sbytes, stream_ptr()), "field_density")
        return sigma, geo, feats, flow

    def _no_autograd(self, what, lidar):
        """The per-sample entry points are forward-only (the differentiable path is run() / render() /
        flow()); called under autograd on trainable parameters they would silently contribute no
        gradient where the reference's versions do, so in training mode they refuse instead."""
        if self.training and torch.is_grad_enabled() and \
                any(getattr(self, n).requires_grad for n in _param_names(lidar)):
            raise _lib.NvsfError(f"NeRFNetwork.{what}() is forward-only: in training mode call it under "
                                 "torch.no_grad() (gradients flow through run() / render() / flow())")

    @_lib.device_guard
    @_lib.with_options
    def density(self, x, t=None, cal_lidar_color=False, **kwargs):
        """x [N,3] in [-bound,bound] -> {'sigma' [N] f32, 'geo_feat' [N,15] f16}."""
        self._no_autograd("density", bool(cal_lidar_color))
        with torch.no_grad():
            return self._density(x, t, cal_lidar_color)

    def _density(self, x, t, cal_lidar_color):
        sigma, geo, _, _ = self._density_raw(x, t, bool(cal_lidar_color))
        return {"sigma": sigma, "geo_feat": geo[:, 1:]}

    @_lib.device_guard
    @_lib.with_options
    def flow(self, x, t):
        """NeRFNetwork.flow (network_dynamic.py:197-211): x [N,3] in [-bound,bound] -> forward / backward
        scene flow [N,3] each.  Differentiable with respect to flow_grid / flow_mlp when autograd is
        enabled (the scene-flow loss, trainer.py:237-265); x itself is treated as data."""
        if torch.is_grad_enabled() and (self.flow_grid.requires_grad or self.flow_mlp.requires_grad):
            with torch.no_grad():
                xx = x.detach().to(device=self.sigma_net.device, dtype=torch.float32).contiguous().view(-1, 3)
                self.prepare(t, True)
            f = _FlowTrain.apply(self, xx, self.flow_grid, self.flow_mlp)
        else:
            with torch.no_grad():
                _, _, _, f = self._density_raw(x, t, True, want_flow=True)
        return {"flow_forward": f[:, :3], "flow_backward": f[:, 3:]}

    @torch.no_grad()
    @_lib.device_guard
    @_lib.with_options
    def features(self, x, t, cal_lidar_color=False):
        """Debug/test hook: the 120 sigma-net inputs [N,120] (fp16) and the flow [N,6]."""
        _, _, feats, f = self._density_raw(x, t, bool(cal_lidar_color), want_features=True, want_flow=True)
        return feats[:, :120], f

    def _color_raw(self, d, geo16, lidar, mask=None, out_ld=None, geo_ld=16, geo_off=1):
        """Heads on n samples; the workspace must be packed for `lidar` (prepare())."""
        L = _setup_lib()
        n = d.shape[0]
        nch = 2 if lidar else 3
        out_ld = out_ld or nch
        out = torch.empty(n, out_ld, dtype=torch.float32, device=d.device)
        check(L.nvsf_field_color(ctypes.byref(self._cfg), ptr(self._ws[lidar]), int(lidar), ptr(d), ptr(geo16),
                                 geo_ld, geo_off, ptr(mask), n, ptr(out), out_ld, stream_ptr()), "field_color")
        return out

    @_lib.device_guard
    @_lib.with_options
    def color(self, x, d, geo_feat, mask=None, cal_lidar_color=False, **kwargs):
        self._no_autograd("color", bool(cal_lidar_color))
        with torch.no_grad():
            return self._color(x, d, geo_feat, mask, cal_lidar_color)

    def _color(self, x, d, geo_feat, mask=None, cal_lidar_color=False):
        """NeRFNetwork.color (network_dynamic.py:290-332): d [N,3] view directions in [-1,1],
        geo_feat [N,15] (the slice `density()` returns, or any fp16/fp32 matrix), mask [N] bool
        or None -> [N, 2] (raydrop, intensity) or [N, 3] rgb, zeros where mask is False.  `x`
        is accepted and unused beyond its shape, as in the reference."""
        lidar = bool(cal_lidar_color)
        dev = self.sigma_net.device
        if self._ws.get(lidar) is None or self._packed.get(lidar) is None or \
                self._packed[lidar][0] != self._version_key(lidar):
            self.prepare(0.0 if self._packed.get(lidar) is None or self._packed[lidar][1] is None
                         else self._packed[lidar][1], lidar)
        d = d.detach().to(device=dev, dtype=torch.float32).contiguous().view(-1, 3)
        n = d.shape[0]
        g = geo_feat.detach()
        if (g.dtype == torch.float16 and g.dim() == 2 and g.shape == (n, 15) and g.stride() == (16, 1)
                and g.storage_offset() >= 1 and g.device == dev
                and (g.data_ptr() - 2) % 16 == 0):
            # the view density() returned: columns 1..15 of the kernel's geo16 rows, used in place
            base, geo_ld, geo_off = g.data_ptr() - 2, 16, 1
            geo_ptr = ctypes.c_void_p(base)
            keep = g
        else:
            keep = g.to(device=dev, dtype=torch.float16).contiguous().view(n, 15)
            geo_ptr, geo_ld, geo_off = ptr(keep), 15, 0
        m = None
        if mask is not None:
            m = mask.detach().to(device=dev).reshape(-1).to(torch.uint8).contiguous()
        L = _setup_lib()
        nch = 2 if lidar else 3
        out = torch.empty(n, nch, dtype=torch.float32, device=dev)
        check(L.nvsf_field_color(ctypes.byref(self._cfg), ptr(self._ws[lidar]), int(lidar), ptr(d), geo_ptr,
                                 geo_ld, geo_off, ptr(m), n, ptr(out), nch, stream_ptr()), "field_color")
        del keep
        return out

    @_lib.device_guard
    @_lib.with_options
    def forward(self, x, d, t=None, cal_lidar_color=False, out_ld=None, _prepared=False):
        """sigma [N] and colours [N, 2|3] of samples (x, d): density + color in two launches
        (what the march_rays* callers evaluate per batch of samples)."""
        lidar = bool(cal_lidar_color)
        with torch.no_grad():
            sigma, geo16, _, _ = self._density_raw(x, t, lidar, prepared=_prepared)
            d = d.detach().to(device=sigma.device, dtype=torch.float32).contiguous().view(-1, 3)
            rgbs = self._color_raw(d, geo16, lidar, out_ld=out_ld)
        return sigma, rgbs

    # ------------------------------------------------------------------ occupancy grid
    def _grid_state(self, lidar):
        st = getattr(self, "_grid", None)
        if st is None:
            st = self._grid = {}
        if lidar not in st:
            dev = self.sigma_net.device
            n = self.cascade * self.grid_size ** 3
            st[lidar] = dict(density_grid=torch.zeros(self.cascade, self.grid_size ** 3, device=dev),
                             density_bitfield=torch.zeros(n // 8, dtype=torch.uint8, device=dev),
                             stats=torch.zeros(2, device=dev), iter_density=0)
        return st[lidar]

    def density_bitfield(self, cal_lidar_color=False):
        return self._grid_state(bool(cal_lidar_color))["density_bitfield"]

    def density_grid(self, cal_lidar_color=False):
        return self._grid_state(bool(cal_lidar_color))["density_grid"]

    def mean_density(self, cal_lidar_color=False):
        """Device scalar (no host sync): mean of clamp(density_grid, 0) after the last update."""
        return self._grid_state(bool(cal_lidar_color))["stats"][0]

    @torch.no_grad()
    @_lib.device_guard
    @_lib.with_options
    def update_extra_state(self, time=0.0, cal_lidar_color=False, decay=0.95, perturb=True, noise=None,
                           process_group=None, shard=None, mode="full", seed=0):
        """Full occupancy-grid update (torch-ngp NeRFRenderer.update_extra_state, the caller the
        reference's morton3D / packbits operators were written for): evaluate sigma at one
        jittered point per cell and cascade, grid = max(grid*decay, sigma*density_scale),
        density_thresh' = min(mean(grid), density_thresh), density_bitfield = packbits(grid).
        `time` may be a list of frame times: a cell is kept if it is occupied at any of them
        (one bitfield serves a dynamic scene because march_rays* take no time argument).
        `noise` [C*H^3, 3] in [0,1) optionally supplies the jitter.

        After mark_untrained_grid the full update evaluates only the trainable cells (grid >= 0); `noise`
        rows are still those of the cells, and the result is bit-identical to evaluating every cell.

        mode="partial" is torch-ngp's partial update: per cascade H^3/4 uniformly drawn cells and H^3/4
        cells drawn from those with grid > 0 (nvsf_grid_draws: a hash of (seed, iter_density, cascade,
        slot), the same on every rank); only the drawn cells are decayed and refreshed, a cell drawn twice
        takes the larger value.  Explicit `noise` is then [C*H^3/2, 3], one row per draw.
        mode="ngp" is torch-ngp's schedule: full while iter_density < 16, partial after that.

        Multi-GPU (SURVEY 8e): with torch.distributed initialised (or `shard=True`) every rank
        evaluates the field on ONE contiguous slice of the C*H^3 cells (dist.cell_slice), the ranks
        all_gather the per-cell sigmas (4 B per cell) and each applies the decay / threshold /
        packbits to the whole grid, so all replicas end with the same grid and bitfield.  `noise`
        given explicitly is the full [C*H^3, 3] array on every rank (each uses its rows).  The list
        of trainable cells or of draws is sliced the same way."""
        from . import dist as nd
        if mode not in ("full", "partial", "ngp"):
            raise ValueError(f"update_extra_state: mode {mode!r} is not 'full', 'partial' or 'ngp'")
        L = _lib.lib()
        lidar = bool(cal_lidar_color)
        st = self._grid_state(lidar)
        dev = self.sigma_net.device
        C, H = self.cascade, self.grid_size
        n = C * H ** 3
        world, rank = nd.world_and_rank(process_group)
        if shard is None:
            shard = world > 1
        if not shard:
            world, rank = 1, 0
        if mode == "partial" or (mode == "ngp" and st["iter_density"] >= 16):
            return self._update_cells(st, self._partial_draws(st, seed), False, time, lidar, decay, perturb, noise,
                                      process_group, world, rank)
        if st.get("trainable") is not None:
            return self._update_cells(st, st["trainable"], True, time, lidar, decay, perturb, noise, process_group,
                                      world, rank)
        per, lo, hi = nd.cell_slice(n, rank, world)
        cnt = hi - lo
        if noise is None and perturb:
            noise = torch.rand(cnt, 3, dtype=torch.float32, device=dev)
        elif noise is not None:
            noise = noise.detach().to(device=dev, dtype=torch.float32).contiguous().view(-1, 3)
            if noise.shape[0] == n:
                noise = noise[lo:hi].contiguous()
            elif noise.shape[0] != cnt:
                raise _lib.NvsfError(f"noise has {noise.shape[0]} rows, expected {n} (all cells) or {cnt} (this slice)")
        xyz = torch.empty(cnt, 3, dtype=torch.float32, device=dev)
        check(L.nvsf_grid_cell_points_range(C, H, self.bound, ptr(noise), lo, cnt, ptr(xyz), stream_ptr()),
              "grid_cell_points_range")
        gathered = torch.zeros(world * per, dtype=torch.float32, device=dev) if world > 1 else None
        tmp = gathered[rank * per:rank * per + per] if world > 1 else torch.empty(n, dtype=torch.float32, device=dev)
        times = list(time) if isinstance(time, (list, tuple)) else [time]
        for k, t in enumerate(times):
            sigma, _, _, _ = self._density_raw(xyz, t, lidar)
            check(L.nvsf_grid_accumulate(ptr(tmp), ptr(sigma), cnt, self.density_scale, int(k == 0), stream_ptr()),
                  "grid_accumulate")
        if world > 1:
            import torch.distributed as tdist
            tdist.all_gather_into_tensor(gathered, tmp.clone(), group=process_group)
            tmp = gathered[:n]
        wbytes = L.nvsf_grid_update_workspace_bytes(n)
        ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
        check(L.nvsf_grid_update(ptr(st["density_grid"]), ptr(tmp), n, float(decay), float(self.density_thresh),
                                 ptr(st["density_bitfield"]), ptr(st["stats"]), ptr(ws), wbytes, stream_ptr()),
              "grid_update")
        st["iter_density"] += 1
        return st["density_bitfield"]

    def _update_cells(self, st, cells, by_cell, time, lidar, decay, perturb, noise, process_group, world, rank):
        """update_extra_state over a list of cells (int32 ids): sigma at the listed cells' jittered points,
        max over the times, scattered into tmp = -1 so that unlisted cells are neither decayed nor refreshed.
        Ranks evaluate one slice of the list each and all_gather the values.  by_cell: `noise` rows are
        cell ids ([C*H^3, 3]); otherwise list positions ([len(cells), 3])."""
        from . import dist as nd
        L = _lib.lib()
        dev = self.sigma_net.device
        C, H = self.cascade, self.grid_size
        n, m = C * H ** 3, cells.shape[0]
        per, lo, hi = nd.cell_slice(m, rank, world)
        cnt = hi - lo
        if noise is not None:
            noise = noise.detach().to(device=dev, dtype=torch.float32).contiguous().view(-1, 3)
            want = n if by_cell else m
            if noise.shape[0] != want:
                raise _lib.NvsfError(f"noise has {noise.shape[0]} rows, expected {want} "
                                     f"({'one per cell' if by_cell else 'one per draw'})")
            if not by_cell:
                noise = noise[lo:hi]
        elif perturb:
            noise, by_cell = torch.rand(cnt, 3, dtype=torch.float32, device=dev), False
        xyz = torch.empty(cnt, 3, dtype=torch.float32, device=dev)
        check(L.nvsf_grid_cell_points_list(C, H, self.bound, ptr(cells[lo:hi]), cnt, ptr(noise), int(by_cell),
                                           ptr(xyz), stream_ptr()), "grid_cell_points_list")
        gathered = torch.zeros(world * per, dtype=torch.float32, device=dev) if world > 1 else None
        vals = gathered[rank * per:rank * per + per] if world > 1 else torch.empty(m, dtype=torch.float32, device=dev)
        if cnt > 0:
            times = list(time) if isinstance(time, (list, tuple)) else [time]
            for k, t in enumerate(times):
                sigma, _, _, _ = self._density_raw(xyz, t, lidar)
                check(L.nvsf_grid_accumulate(ptr(vals), ptr(sigma), cnt, self.density_scale, int(k == 0),
                                             stream_ptr()), "grid_accumulate")
        if world > 1 and per > 0:
            import torch.distributed as tdist
            tdist.all_gather_into_tensor(gathered, vals.clone(), group=process_group)
            vals = gathered[:m]
        tmp = torch.full((n,), -1.0, dtype=torch.float32, device=dev)
        check(L.nvsf_grid_scatter_max(ptr(tmp), n, ptr(cells), ptr(vals), m, stream_ptr()), "grid_scatter_max")
        wbytes = L.nvsf_grid_update_workspace_bytes(n)
        ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
        check(L.nvsf_grid_update(ptr(st["density_grid"]), ptr(tmp), n, float(decay), float(self.density_thresh),
                                 ptr(st["density_bitfield"]), ptr(st["stats"]), ptr(ws), wbytes, stream_ptr()),
              "grid_update")
        st["iter_density"] += 1
        return st["density_bitfield"]

    def _cell_list(self, st, above):
        """(cells [n] int32 device, offsets [C+1] int32 device): the cells with grid >= 0 (above=False) or
        grid > 0 (above=True) in ascending order, cascade c's at cells[offsets[c]:offsets[c+1]]."""
        L = _lib.lib()
        dev = self.sigma_net.device
        C, H3 = self.cascade, self.grid_size ** 3
        cells = torch.empty(C * H3, dtype=torch.int32, device=dev)
        offsets = torch.empty(C + 1, dtype=torch.int32, device=dev)
        wbytes = L.nvsf_grid_cell_list_workspace_bytes(C * H3)
        ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
        check(L.nvsf_grid_cell_list(ptr(st["density_grid"]), C, H3, int(above), ptr(cells), ptr(offsets), ptr(ws),
                                    wbytes, stream_ptr()), "grid_cell_list")
        return cells, offsets

    def _partial_draws(self, st, seed):
        """The C*H^3/2 cells of a partial update (nvsf_grid_draws); no host read."""
        L = _lib.lib()
        C, H3 = self.cascade, self.grid_size ** 3
        occupied, offsets = self._cell_list(st, True)
        cells = torch.empty(C * (H3 // 2), dtype=torch.int32, device=occupied.device)
        check(L.nvsf_grid_draws(C, H3, int(seed) & (2 ** 64 - 1), st["iter_density"], ptr(occupied), ptr(offsets),
                                ptr(cells), stream_ptr()), "grid_draws")
        return cells

    def _refresh_trainable(self, st):
        """Rebuild the list of trainable cells (grid >= 0) after marks change; one host read of its length.
        No marked cell: no list, and the full update takes the all-cells path."""
        cells, offsets = self._cell_list(st, False)
        k = int(offsets[-1])
        st["trainable"] = cells[:k] if k < cells.shape[0] else None

    @torch.no_grad()
    @_lib.device_guard
    @_lib.with_options
    def mark_untrained_grid(self, camera_poses=None, intrinsics=None, H=None, W=None, lidar_poses=None,
                            intrinsics_lidar=None, intrinsics_hoz_lidar=None, cal_lidar_color=False):
        """torch-ngp's mark_untrained_grid: cells of the occupancy grid of the modality `cal_lidar_color`
        whose centre no given sensor pose sees (DESIGN.md §3.5: the image frustum of a pinhole camera, the
        elevation band, range and azimuth wedge of a LiDAR, each widened by two half-cells) get grid = -1
        and are never occupied; updates skip them.  camera_poses [B,4,4] cam2world with intrinsics (3x3
        pinhole matrix) and the image size H x W; lidar_poses [B,4,4] lidar2world with intrinsics_lidar =
        (fov_up, fov) and intrinsics_hoz_lidar = (., fov_hoz) in degrees, range [min_near_lidar,
        lidar_max_depth].  Either group may be omitted, not both.  Calls accumulate: the marks are those
        of the union of every pose given so far (a cell seen by a later call is restored to 0).
        Returns the number of marked cells as a device scalar."""
        if camera_poses is None and lidar_poses is None:
            raise _lib.NvsfError("mark_untrained_grid: give camera_poses and / or lidar_poses")
        L = _lib.lib()
        lidar = bool(cal_lidar_color)
        st = self._grid_state(lidar)
        dev = self.sigma_net.device
        C, Hg = self.cascade, self.grid_size
        n = C * Hg ** 3
        covered = torch.zeros(n // 8, dtype=torch.uint8, device=dev)
        if st.get("trainable") is not None:  # earlier marks: covered so far == grid >= 0 (marks hold -1)
            check(L.nvsf_packbits(ptr(st["density_grid"]), n // 8, -0.5, ptr(covered), stream_ptr()), "packbits")

        def poses_of(p, what):
            p = torch.as_tensor(p).detach().to(device=dev, dtype=torch.float32).contiguous()
            if p.dim() == 2:
                p = p.unsqueeze(0)
            if p.dim() != 3 or p.shape[1:] != (4, 4):
                raise _lib.NvsfError(f"mark_untrained_grid: {what} must be [B,4,4], got {tuple(p.shape)}")
            return p

        if camera_poses is not None:
            if intrinsics is None or H is None or W is None:
                raise _lib.NvsfError("mark_untrained_grid: camera_poses need intrinsics, H and W")
            p = poses_of(camera_poses, "camera_poses")
            K = torch.as_tensor(intrinsics, dtype=torch.float64).cpu()
            fx, fy, cx, cy = float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])
            check(L.nvsf_grid_coverage_camera(C, Hg, self.bound, ptr(p), p.shape[0], fx, fy, cx, cy, int(H), int(W),
                                              ptr(covered), stream_ptr()), "grid_coverage_camera")
        if lidar_poses is not None:
            if intrinsics_lidar is None or intrinsics_hoz_lidar is None:
                raise _lib.NvsfError("mark_untrained_grid: lidar_poses need intrinsics_lidar and intrinsics_hoz_lidar")
            p = poses_of(lidar_poses, "lidar_poses")
            check(L.nvsf_grid_coverage_lidar(C, Hg, self.bound, ptr(p), p.shape[0], float(intrinsics_lidar[0]),
                                             float(intrinsics_lidar[1]), float(intrinsics_hoz_lidar[1]),
                                             self.min_near_lidar, self.lidar_max_depth, ptr(covered), stream_ptr()),
                  "grid_coverage_lidar")
        n_marked = torch.empty(1, dtype=torch.int32, device=dev)
        check(L.nvsf_grid_apply_marks(ptr(st["density_grid"]), ptr(st["density_bitfield"]), ptr(covered), n,
                                      ptr(n_marked), stream_ptr()), "grid_apply_marks")
        self._refresh_trainable(st)
        return n_marked[0]

    def occupancy_state_dict(self):
        """The occupancy grids, apart from state_dict(): {"lidar" | "camera": {density_grid (with its -1 marks),
        density_bitfield, stats, iter_density}} for each modality that has a grid."""
        names = {True: "lidar", False: "camera"}
        return {names[k]: dict(density_grid=v["density_grid"].clone(), density_bitfield=v["density_bitfield"].clone(),
                               stats=v["stats"].clone(), iter_density=int(v["iter_density"]))
                for k, v in getattr(self, "_grid", {}).items()}

    @torch.no_grad()
    @_lib.device_guard
    @_lib.with_options
    def load_occupancy_state_dict(self, sd):
        """Load what occupancy_state_dict() returned (CPU or GPU tensors) and rebuild the trainable-cell list."""
        C, H3 = self.cascade, self.grid_size ** 3
        n = C * H3
        for name, v in sd.items():
            if name not in ("lidar", "camera"):
                raise _lib.NvsfError(f"load_occupancy_state_dict: unknown modality {name!r}")
            g, b, s = v["density_grid"], v["density_bitfield"], v["stats"]
            if g.numel() != n or b.numel() != n // 8 or b.dtype != torch.uint8 or s.numel() != 2:
                raise _lib.NvsfError(f"load_occupancy_state_dict: {name} grid has {g.numel()} cells / "
                                     f"{b.numel()} bitfield bytes, this model has C*H^3 = {n} / {n // 8}")
            st = self._grid_state(name == "lidar")
            st["density_grid"].view(-1).copy_(g.reshape(-1))
            st["density_bitfield"].copy_(b.reshape(-1))
            st["stats"].copy_(s.reshape(-1))
            st["iter_density"] = int(v["iter_density"])
            self._refresh_trainable(st)

    @torch.no_grad()
    @_lib.device_guard
    @_lib.with_options
    def extract_geometry(self, time, resolution=256, threshold=10.0, cal_lidar_color=False):
        """torch-ngp's extract_geometry / save_mesh on the device: sigma at `time` on the resolution^3 lattice
        torch.linspace(aabb_infer[a], aabb_infer[3 + a], resolution) per axis ('ij' order), marching cubes at
        `threshold` (mesh.marching_cubes) and the vertex transform v / (resolution - 1) * (b_max - b_min) + b_min
        in fp32.  Returns (vertices [V,3] fp32 world coordinates, triangles [T,3] int64), both on the device."""
        from . import mesh
        R = int(resolution)
        vol, b = self._density_volume(time, R, bool(cal_lidar_color))
        v, f = mesh.marching_cubes(vol, threshold)
        lo, hi = b[:3].to(vol.device), b[3:].to(vol.device)
        return v / float(R - 1) * (hi - lo) + lo, f

    @torch.no_grad()
    @_lib.device_guard
    @_lib.with_options
    def _density_volume(self, time, R, lidar):
        """(sigma [R,R,R] on the device, aabb_infer on the host): x-slabs of at most 2^24 lattice points."""
        if not 2 <= R <= 1024:
            raise _lib.NvsfError(f"extract_geometry: resolution {R} out of range [2, 1024]")
        dev = self.sigma_net.device
        b = self.aabb_infer.detach().to(torch.float32).cpu()
        axes = [torch.linspace(b[a], b[3 + a], R).to(dev) for a in range(3)]   # the reference's CPU linspace
        vol = torch.empty(R, R, R, dtype=torch.float32, device=dev)
        self.prepare(time, lidar)
        slab = max(1, (1 << 24) // (R * R))
        for i0 in range(0, R, slab):
            xs = axes[0][i0:i0 + slab]
            pts = torch.stack(torch.meshgrid(xs, axes[1], axes[2], indexing="ij"), -1).view(-1, 3)
            sigma, _, _, _ = self._density_raw(pts, time, lidar, prepared=True)
            vol[i0:i0 + len(xs)].view(-1).copy_(sigma)
        return vol, b

    # ------------------------------------------------------------------ march_rays* render loops
    @torch.no_grad()
    @_lib.device_guard
    @_lib.with_options
    def run_cuda(self, rays_o, rays_d, time, cal_lidar_color=False, dt_gamma=0.0, bg_color=None, perturb=False,
                 max_steps=1024, T_thresh=1e-4, one_shot=None, noises=None, density_bitfield=None,
                 step_scale=16, sample_capacity=None, **kwargs):
        """Occupancy-skipping render built from the raymarching operators (the `cuda_ray` path of
        torch-ngp's NeRFRenderer.run_cuda, which raymarching.py:171-510 was written for).

        one_shot=True  (default): near_far -> march_rays_train -> density -> color -> composite_rays_train
                       over ALL samples of the frame, one host read (the sample count).  torch-ngp's
                       training branch; on a B200 also the faster way to render a frame (measured:
                       camera frame 22.9 ms vs 29.2 ms for the loop, profiles/r01_march_render.jsonl).
        one_shot=False: torch-ngp's eval branch, the alive-ray loop march_rays(n_step) -> density ->
                       color -> composite_rays -> compaction until every ray has terminated; pays off
                       only when most rays terminate early.  n_step is `step_scale` x torch-ngp's
                       max(min(N // n_alive, 8), 1): the composited result does not depend on it (up to
                       fp32 rounding of the restart point), a B200 wants few, large launches.
        sample_capacity (one_shot only): number of sample rows to provision WITHOUT reading the sample count
                       back to the host (torch-ngp's `mean_count` protocol, raymarching.py:186-188,272-279): the
                       frame is rendered with no host synchronisation at all; rays that would not fit are treated
                       as empty by the operators (raymarching.cu:453,596).  `last_run_cuda_counter` keeps the
                       device-side count so the caller can verify `samples <= capacity` whenever it likes.
        Outputs use run()'s keys: depth = sum w*t (absolute distance along the ray, not normalised),
        image [.., 2|3], weights_sum.
        LiDAR: near/far are the constants of renderer_dynamic.py:141-146 and no background is added."""
        lidar = bool(cal_lidar_color)
        prefix = rays_o.shape[:-1]
        o, d, nears, fars, _ = self._rays_setup(rays_o, rays_d, lidar, 1, False, None)
        N = o.shape[0]
        dev = o.device
        nch = 2 if lidar else 3
        bits = density_bitfield if density_bitfield is not None else self.density_bitfield(lidar)
        self.prepare(time, lidar)
        if one_shot is None:
            one_shot = True
        if noises is None and perturb:
            noises = torch.rand(N, dtype=torch.float32, device=dev)
        if one_shot:
            cap = int(sample_capacity) if sample_capacity else -1
            xyzs, dirs, deltas, rays = raymarching.march_rays_train(
                o, d, self.bound, bits, self.cascade, self.grid_size, nears, fars, None, cap, noises is not None,
                -1, cap <= 0, dt_gamma, max_steps, noises)
            self.last_run_cuda_counter = raymarching.last_step_counter
            sigmas, rgbs = self.forward(xyzs, dirs, time, lidar, out_ld=3, _prepared=True)
            if self.density_scale != 1:
                sigmas = sigmas * self.density_scale
            weights_sum, depth, image = raymarching.composite_rays_train(sigmas, rgbs, deltas, rays, T_thresh)
            # composite_rays_train accumulates t from 0 at the ray's first marching position
            # (raymarching.cu:372-375,626-627) while composite_rays starts from rays_t = near
            # (:1003): make the one-shot depth absolute like run()'s sum(w * z)
            t0 = nears
            if noises is not None:
                dt_min = 2 * math.sqrt(3) / max_steps
                dt_max = 2 * math.sqrt(3) * 2 ** (self.cascade - 1) / self.grid_size
                t0 = nears + (nears * dt_gamma).clamp(dt_min, dt_max) * noises.to(nears.dtype)
            depth = depth + weights_sum * t0
            n_samples = xyzs.shape[0]
        else:
            L = _lib.lib()
            weights_sum = torch.zeros(N, dtype=torch.float32, device=dev)
            depth = torch.zeros(N, dtype=torch.float32, device=dev)
            image = torch.zeros(N, 3, dtype=torch.float32, device=dev)
            rays_alive = torch.arange(N, dtype=torch.int32, device=dev)
            spare = torch.empty(N, dtype=torch.int32, device=dev)
            rays_t = nears.clone()
            n_dev = torch.empty(1, dtype=torch.int32, device=dev)
            n_host = torch.empty(1, dtype=torch.int32).pin_memory()
            cbytes = L.nvsf_compact_alive_workspace_bytes(N)
            cws = torch.empty(max(cbytes, 16), dtype=torch.uint8, device=dev)
            n_alive, step, n_samples = N, 0, 0
            while step < max_steps and n_alive > 0:
                n_step = max(min(N // n_alive, 8), 1) * int(step_scale)
                nz = noises if (noises is not None and step == 0) else None
                xyzs, dirs, deltas = raymarching.march_rays(
                    n_alive, n_step, rays_alive, rays_t, o, d, self.bound, bits, self.cascade, self.grid_size,
                    nears, fars, -1, nz is not None, dt_gamma, max_steps, nz)
                sigmas, rgbs = self.forward(xyzs, dirs, time, lidar, out_ld=3, _prepared=True)
                if self.density_scale != 1:
                    sigmas = sigmas * self.density_scale
                raymarching.composite_rays(n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum,
                                           depth, image, T_thresh)
                check(L.nvsf_compact_alive(ptr(rays_alive), n_alive, ptr(spare), ptr(n_dev), ptr(cws), cbytes,
                                           stream_ptr()), "compact_alive")
                n_host.copy_(n_dev, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                rays_alive, spare = spare, rays_alive
                n_samples += n_alive * n_step
                n_alive = int(n_host[0])
                step += n_step
        image = image[:, :nch]
        if not lidar:
            bg = 1.0 if bg_color is None else bg_color
            image = image + (1 - weights_sum).unsqueeze(-1) * bg
        sfx = "_lidar" if lidar else ""
        self.last_run_cuda_samples = n_samples
        return {"depth" + sfx: depth.view(*prefix), "image" + sfx: image.reshape(*prefix, nch),
                "weights_sum" + sfx: weights_sum}

    # ------------------------------------------------------------------ renderer API
    @_lib.device_guard
    @_lib.with_options
    def run(self, rays_o, rays_d, time, cal_lidar_color=False, num_steps=768, upsample_steps=128,
            bg_color=None, perturb=False, noise=None, return_weights=True, **kwargs):
        """NeRFRenderer.run (renderer_dynamic.py:109-265).  `noise` [N,num_steps] optionally
        supplies the stratified-sampling jitter that perturb=True otherwise draws with torch.rand.
        With autograd enabled and parameters that require grad the call is differentiable
        w.r.t. the field parameters (depth, image, weights_sum, weights)."""
        if torch.is_grad_enabled() and any(getattr(self, n).requires_grad for n in _param_names(bool(cal_lidar_color))):
            return self._run_train(rays_o, rays_d, time, bool(cal_lidar_color), int(num_steps), bg_color, perturb,
                                   noise)
        with torch.no_grad():
            return self._run_infer(rays_o, rays_d, time, cal_lidar_color, num_steps, bg_color, perturb, noise,
                                   return_weights)

    def _rays_setup(self, rays_o, rays_d, lidar, S, perturb, noise):
        dev = self.sigma_net.device
        o = rays_o.detach().to(device=dev, dtype=torch.float32).contiguous().view(-1, 3)
        d = rays_d.detach().to(device=dev, dtype=torch.float32).contiguous().view(-1, 3)
        N = o.shape[0]
        if lidar:
            nears = torch.full((N,), self.min_near_lidar, dtype=torch.float32, device=dev)
            fars = torch.full((N,), self.lidar_max_depth, dtype=torch.float32, device=dev)
        else:
            aabb = self.aabb_train if self.training else self.aabb_infer
            nears, fars = raymarching.near_far_from_aabb(o, d, aabb, self.min_near)
        if noise is None and perturb:
            noise = torch.rand(N, S, dtype=torch.float32, device=dev)
        if noise is not None:
            noise = noise.detach().to(device=dev, dtype=torch.float32).contiguous()
        return o, d, nears, fars, noise

    @staticmethod
    def _split_bg(bg_color, n, dev):
        """bg_color as NeRFRenderer.run accepts it (renderer_dynamic.py:236-237; train_step passes 1 or a
        per-pixel random [B,N,3] tensor, trainer.py:484-489): a number goes to the kernel, a tensor is
        blended outside it as (1 - weights_sum) * bg (differentiable through weights_sum)."""
        if bg_color is None:
            return 1.0, None
        if torch.is_tensor(bg_color):
            if bg_color.numel() == 1:
                return float(bg_color), None
            bg = bg_color.detach().to(device=dev, dtype=torch.float32)
            return 0.0, (bg.reshape(-1, 3) if bg.numel() == 3 * n else bg.reshape(1, 3))
        return float(bg_color), None

    def _run_train(self, rays_o, rays_d, time, lidar, S, bg_color, perturb, noise):
        self.out_dim = self.out_lidar_color_dim if lidar else self.out_color_dim
        prefix = rays_o.shape[:-1]
        with torch.no_grad():
            o, d, nears, fars, noise = self._rays_setup(rays_o, rays_d, lidar, S, perturb, noise)
            self.prepare(time, lidar)
        bg, bg_t = self._split_bg(bg_color, o.shape[0], o.device)
        params = [getattr(self, n) for n in _param_names(lidar)]
        depth, image, wsum, weights, z_vals = _RenderUniformTrain.apply(self, lidar, o, d, nears, fars, noise, S,
                                                                        bg, *params)
        if bg_t is not None and not lidar:
            image = image + (1 - wsum).unsqueeze(-1) * bg_t
        sfx = "_lidar" if lidar else ""
        return {"depth" + sfx: depth.view(*prefix), "image" + sfx: image.view(*prefix, self.out_dim),
                "weights_sum" + sfx: wsum, "weights": weights, "z_vals": z_vals}

    def _run_infer(self, rays_o, rays_d, time, cal_lidar_color, num_steps, bg_color, perturb, noise,
                   return_weights):
        L = _setup_lib()
        lidar = bool(cal_lidar_color)
        self.out_dim = self.out_lidar_color_dim if lidar else self.out_color_dim
        dev = self.sigma_net.device
        prefix = rays_o.shape[:-1]
        S = int(num_steps)
        o, d, nears, fars, noise = self._rays_setup(rays_o, rays_d, lidar, S, perturb, noise)
        N = o.shape[0]
        ws = self.prepare(time, lidar)
        nch = self.out_dim
        depth = torch.empty(N, dtype=torch.float32, device=dev)
        image = torch.empty(N, nch, dtype=torch.float32, device=dev)
        wsum = torch.empty(N, dtype=torch.float32, device=dev)
        weights = torch.empty(N, S, dtype=torch.float32, device=dev) if return_weights else None
        z_vals = torch.empty(N, S, dtype=torch.float32, device=dev) if return_weights else None
        sbytes = L.nvsf_render_uniform_scratch_bytes(N, S)
        scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
        bg, bg_t = self._split_bg(bg_color, N, dev)
        check(L.nvsf_render_uniform(ctypes.byref(self._cfg), ptr(ws), int(lidar), ptr(o), ptr(d), ptr(nears),
                                    ptr(fars), ptr(noise), N, S, bg, ptr(scratch), sbytes, ptr(depth),
                                    ptr(image), ptr(wsum), ptr(weights), ptr(z_vals), stream_ptr()),
              "render_uniform")
        if bg_t is not None and not lidar:
            image = image + (1 - wsum).unsqueeze(-1) * bg_t
        sfx = "_lidar" if lidar else ""
        out = {"depth" + sfx: depth.view(*prefix), "image" + sfx: image.view(*prefix, nch),
               "weights_sum" + sfx: wsum}
        if return_weights:
            out["weights"], out["z_vals"] = weights, z_vals
        return out

    @_lib.device_guard
    @_lib.with_options
    def render(self, rays_o, rays_d, time, cal_lidar_color=False, staged=False, max_ray_batch=4096, **kwargs):
        """NeRFRenderer.render (renderer_dynamic.py:267-326).  staged=True returns only depth and
        image like the reference; the whole frame is rendered by one launch pair per
        `frame_ray_batch` rays (default: all) instead of a Python loop of 4096-ray chunks —
        `max_ray_batch` is accepted for signature compatibility."""
        if not staged:
            return self.run(rays_o, rays_d, time, cal_lidar_color=cal_lidar_color, **kwargs)
        with torch.no_grad():  # staged rendering is the evaluation path (trainer.py:658-903, under no_grad)
            return self._render_staged(rays_o, rays_d, time, cal_lidar_color, kwargs)

    @torch.no_grad()
    @_lib.device_guard
    @_lib.with_options
    def render_frame(self, pose, intrinsics, H, W, time, cal_lidar_color=False, intrinsics_hoz=None, **kwargs):
        """Full-frame render from a sensor pose: ray generation (SURVEY 8f rank 1; get_lidar_rays / get_rays,
        dataset_utils.py:369-687) runs on the device in the same stream as the renderer, so a frame's only
        host input is the 4x4 pose (64 B instead of 24 B per ray over PCIe) and nothing synchronises with the
        host between the pose upload and the finished image.  pose [4,4] (or [1,4,4]) sensor-to-world;
        LiDAR: intrinsics = (fov_up, fov), intrinsics_hoz = (fov_up, fov) in degrees (defaults to
        `intrinsics`); camera: intrinsics = 3x3 pinhole matrix.  Returns render(staged=True)'s dict reshaped to
        [H, W] / [H, W, C]."""
        from . import rays as R
        lidar = bool(cal_lidar_color)
        dev = self.sigma_net.device
        pose = torch.as_tensor(pose, dtype=torch.float32).to(dev, non_blocking=True).reshape(1, 4, 4)
        if lidar:
            r = R.get_lidar_rays(pose, intrinsics, intrinsics if intrinsics_hoz is None else intrinsics_hoz, H, W, -1)
        else:
            r = R.get_rays(pose, intrinsics, H, W, -1)
        out = self._render_staged(r["rays_o"], r["rays_d"], time, lidar, dict(kwargs))
        return {k: (v.view(H, W) if v.dim() == 2 else v.view(H, W, -1)) for k, v in out.items()}

    def _render_staged(self, rays_o, rays_d, time, cal_lidar_color, kwargs):
        lidar = bool(cal_lidar_color)
        B, N = rays_o.shape[:2]
        chunk = int(kwargs.pop("frame_ray_batch", 0)) or N
        keys = ["depth_lidar", "image_lidar"] if lidar else ["depth", "image"]
        depth, image = [], []
        for b in range(B):
            for head in range(0, N, chunk):
                r = self.run(rays_o[b:b + 1, head:head + chunk], rays_d[b:b + 1, head:head + chunk],
                             time[b:b + 1] if torch.is_tensor(time) else time, cal_lidar_color=lidar,
                             return_weights=False, **kwargs)
                depth.append(r[keys[0]])
                image.append(r[keys[1]])
        depth = torch.cat(depth, dim=1).view(B, N) if len(depth) > 1 else depth[0].view(B, N)
        image = torch.cat(image, dim=1).view(B, N, -1) if len(image) > 1 else image[0].view(B, N, -1)
        return {keys[0]: depth, keys[1]: image}
