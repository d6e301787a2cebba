"""Adam over the flat parameter / gradient buffers of a NeRFNetwork replica.

Mirrors the optimizer the reference builds (reference nvsf/scripts/main_nvsf.py:350-352 with the
parameter groups of NeRFNetwork.get_params, network_dynamic.py:335-357: encoders, sigma_net and
color_net at `lr`; flow_net, intensity_net and raydrop_net at 0.1 * lr), but as ONE streaming CUDA
pass per learning-rate segment (csrc/optim.cu) over buffers that already are flat: `GradSync`
(dist.py) owns the gradients, this class re-homes the parameters and the two moment buffers in the
same order.  There is no PyTorch fallback.

shard=True (SURVEY.md section 8f rank 4, "Adam fused with the all-reduce epilogue"): GradSync runs in
reduce_scatter mode, every rank keeps the Adam moments of — and updates — only its 1/world slice of each
group, and the updated parameter slices are all-gathered in place: the optimizer is the epilogue of the
gradient reduction, Adam's 28 B/parameter of HBM traffic and the moment memory shrink by the world size.

skip_nonfinite=True gives `scaler.step(optimizer)` semantics (trainer.py:1332-1334) without a host sync:
non-finite gradients are detected on the device, the 4-byte flag is all-reduced (MAX) so that every rank
agrees, and the guarded kernel leaves parameters, moments and the step count untouched.

ema_decay=d keeps the reference trainer's torch_ema.ExponentialMovingAverage (trainer.py:112-114) as one
more flat buffer laid out like the moments (sharded like them); `update_ema()` is its `ema.update()` and
`ema_weights()` its store / copy_to / restore around evaluation (trainer.py:1475-1477).

Checkpoints: `state_dict()` / `load_state_dict()` hold the moments and the EMA per parameter name, so a
state saved at one world size loads at another; `reference_optimizer_state_dict()` /
`load_reference_optimizer_state()` and `reference_ema_state_dict()` / `load_reference_ema_state()` speak
the reference checkpoint's "optimizer" (torch.optim.Adam) and "ema" (torch_ema) entries (utils.py:610-680)."""
import contextlib

import torch

from . import _lib
from ._lib import NvsfError, check, ptr, stream_ptr
from .dist import GROUPS, GradSync

LR_SCALE = {"flow_grid": 0.1, "flow_mlp": 0.1, "intensity_net": 0.1, "raydrop_net": 0.1}


class FlatAdam:
    def __init__(self, model, lr=1e-2, betas=(0.9, 0.99), eps=1e-15, grad_sync=None, shard=False,
                 skip_nonfinite=False, process_group=None, comm_dtype=None, step_fn=None, ema_decay=None):
        self.model, self.lr, self.betas, self.eps = model, float(lr), betas, float(eps)
        self.last_lr = self.lr   # the lr of the latest step(), stored in the checkpoint
        self.shard, self.skip_nonfinite = bool(shard), bool(skip_nonfinite)
        if grad_sync is None:
            grad_sync = GradSync(model, process_group=process_group, comm_dtype=comm_dtype,
                                 mode="reduce_scatter" if shard else "allreduce")
        if self.shard != (grad_sync.mode == "reduce_scatter"):
            raise ValueError("FlatAdam(shard=True) needs GradSync(mode='reduce_scatter') and vice versa")
        self.sync = grad_sync
        self._step_fn = step_fn   # tests of the sharding logic on CPU inject a step; None = the CUDA kernels
        params = dict(model.named_parameters())
        self.names = [n for g in GROUPS.values() for n in g]
        total = self.sync.flat.numel()
        dev = self.sync.flat.device
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.segments = []
        with torch.no_grad():
            for n in self.names:
                p = params[n]
                off, k = self.sync.param_offsets[n]
                self.flat[off:off + k].copy_(p.detach().reshape(-1))
                p.data = self.flat[off:off + k].view_as(p)   # parameters become views of the flat buffer
                # every tensor is padded to a multiple of 4 floats by construction of the field
                if off % 4 or k % 4:
                    raise ValueError(f"{n}: segment [{off}, {off + k}) is not 16-byte aligned")
                self.segments.append((n, off, k, LR_SCALE.get(n, 1.0)))
        # the part of the flat buffer this rank updates: its slice of every group (everything when not sharded)
        self.owned = [self.sync.shard(g) for g in GROUPS]
        n_owned = sum(hi - lo for lo, hi in self.owned)
        self.exp_avg = torch.zeros(n_owned, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n_owned, dtype=torch.float32, device=dev)
        self.state = torch.zeros(4, dtype=torch.float32, device=dev)      # see nvsf_adam_begin
        self.found_inf = torch.zeros(1, dtype=torch.float32, device=dev)
        self.step_count = 0   # steps requested on the host; the applied count is state[0] on the device
        # EMA shadow of the owned parameter ranges (torch_ema: shadow starts as a copy of the parameters)
        self.ema_decay, self.ema_num_updates, self.ema = None, 0, None
        if ema_decay is not None:
            self.ema_decay = float(ema_decay)
            self.ema = torch.cat([self.flat[lo:hi] for lo, hi in self.owned])
        # merge neighbours with the same learning rate: fewer, longer launches
        merged = []
        for n, o, k, s in self.segments:
            if merged and merged[-1][3] == s and merged[-1][1] + merged[-1][2] == o:
                merged[-1] = (merged[-1][0] + "+" + n, merged[-1][1], merged[-1][2] + k, s)
            else:
                merged.append((n, o, k, s))
        # ... intersected with the owned ranges: (flat offset, moment offset, length, lr scale)
        self.launches, moff = [], 0
        for lo, hi in self.owned:
            for _, o, k, s in merged:
                a, b = max(lo, o), min(hi, o + k)
                if a < b:
                    self.launches.append((a, moff + a - lo, b - a, s))
            moff += hi - lo

    def zero_grad(self):
        self.sync.zero_grad()

    def applied_steps(self):
        """Number of steps that were not skipped (host read of the device counter)."""
        return int(self.state[0].item())

    @torch.no_grad()
    def step(self, lr=None, grad_scale=1.0):
        """One Adam step (the reference's lr scheduler passes the current lr every step,
        trainer.py:1337-1338).  The gradient reduction of every group must have been started
        (GradSync.reduce_group) and waited for (GradSync.wait)."""
        self.step_count += 1
        lr = self.lr if lr is None else float(lr)
        self.last_lr = lr
        g = self.sync.flat
        if self._step_fn is not None:   # CPU tests of the partition / collective choreography
            found = None
            if self.skip_nonfinite:
                self.found_inf.zero_()
                for lo, hi in self.owned:
                    if not bool(torch.isfinite(g[lo:hi]).all()):
                        self.found_inf.fill_(1.0)
                found = self.sync.all_reduce_flag(self.found_inf)
            self._step_fn(self, lr, float(grad_scale), found)
        else:
            L = _lib.lib()
            st = stream_ptr()
            found = None
            if self.skip_nonfinite:
                self.found_inf.zero_()
                for lo, hi in self.owned:
                    check(L.nvsf_grad_found_inf(g.data_ptr() + 4 * lo, hi - lo, ptr(self.found_inf), st),
                          "grad_found_inf")
                found = self.sync.all_reduce_flag(self.found_inf)
            check(L.nvsf_adam_begin(ptr(self.state), ptr(found), self.betas[0], self.betas[1], st), "adam_begin")
            for off, moff, k, scale in self.launches:
                check(L.nvsf_adam_step_guarded(self.flat.data_ptr() + 4 * off, g.data_ptr() + 4 * off,
                                               self.exp_avg.data_ptr() + 4 * moff,
                                               self.exp_avg_sq.data_ptr() + 4 * moff, k, lr * scale, self.betas[0],
                                               self.betas[1], self.eps, ptr(self.state), float(grad_scale), st),
                      "adam_step_guarded")
        if self.shard:
            for gname in GROUPS:
                self.sync.all_gather_group(self.flat, gname)
        # the packed tables (fp16 hash, channel-last planes, MLP images) are stale now
        self.model._packed.clear()

    # ------------------------------------------------------------------ EMA of the parameters
    def _owned_parts(self, buf):
        """(group, lo, hi, slice of buf) for every owned range of a buffer laid out like exp_avg."""
        moff = 0
        for gname, (lo, hi) in zip(GROUPS, self.owned):
            yield gname, lo, hi, buf[moff:moff + hi - lo]
            moff += hi - lo

    def _need_ema(self):
        if self.ema is None:
            raise NvsfError("FlatAdam was built without ema_decay: there are no EMA weights")

    @torch.no_grad()
    def update_ema(self):
        """torch_ema's `ema.update()` (trainer.py:112-114) over this rank's parameter ranges: one
        nvsf_ema_update launch per owned range, with torch_ema's decay warm-up
        min(decay, (1 + t) / (10 + t)).  Unconditional, also after a skipped step, like torch_ema."""
        self._need_ema()
        if not self.ema.is_cuda:
            raise NvsfError("update_ema runs on the GPU: the model's parameters are not CUDA tensors")
        decay = self.ema_decay
        if self.ema_num_updates is not None:   # torch_ema(use_num_updates=False) keeps None: no warm-up
            self.ema_num_updates += 1
            decay = min(decay, (1 + self.ema_num_updates) / (10 + self.ema_num_updates))
        L, st = _lib.lib(), stream_ptr()
        for _, lo, hi, shadow in self._owned_parts(self.ema):
            # 1 - decay in double, rounded to float by ctypes as torch rounds the scalar of tmp.mul_(omd)
            check(L.nvsf_ema_update(shadow.data_ptr(), self.flat.data_ptr() + 4 * lo, hi - lo, 1.0 - decay, st),
                  "ema_update")

    def _set_owned(self, buf):
        """Copy a buffer laid out like exp_avg into the owned parameter ranges and all-gather them."""
        for gname, lo, hi, part in self._owned_parts(buf):
            self.flat[lo:hi].copy_(part)
            self.sync.all_gather_group(self.flat, gname)
        self.model._packed.clear()

    @contextlib.contextmanager
    def ema_weights(self):
        """Run the body with the EMA weights in the model (torch_ema's store / copy_to / restore around
        evaluation, trainer.py:1475-1477); the parameters are restored exactly on exit.  A collective
        when sharded: every rank must enter and leave together."""
        self._need_ema()
        with torch.no_grad():
            saved = torch.cat([self.flat[lo:hi] for lo, hi in self.owned])
            self._set_owned(self.ema)
        try:
            yield
        finally:
            with torch.no_grad():
                self._set_owned(saved)

    # ------------------------------------------------------------------ native checkpoint
    def _shapes(self):
        params = dict(self.model.named_parameters())
        return {n: tuple(params[n].shape) for n in self.names}

    def _gathered(self, buf):
        """{parameter name: tensor in the parameter's shape} of a buffer laid out like exp_avg: every rank
        all-gathers each group's padded range into a temporary (a collective when sharded)."""
        full = torch.zeros_like(self.flat)
        for gname, lo, hi, part in self._owned_parts(buf):
            full[lo:hi].copy_(part)
            self.sync.all_gather_group(full, gname)
        shapes = self._shapes()
        return {n: full[off:off + k].view(shapes[n]) for n, off, k, _ in self.segments}

    def _owned_from_named(self, named, what):
        """The inverse of _gathered for this rank: a new buffer laid out like exp_avg holding the owned
        ranges of {parameter name: tensor}; names and shapes are checked first."""
        shapes = self._shapes()
        if set(named) != set(shapes):
            raise NvsfError(f"{what}: parameters {sorted(set(named) ^ set(shapes))} are not those of the model")
        for n, t in named.items():
            if tuple(t.shape) != shapes[n]:
                raise NvsfError(f"{what}[{n}]: shape {tuple(t.shape)} != {shapes[n]}")
        buf = torch.zeros_like(self.exp_avg)
        for _, lo, hi, part in self._owned_parts(buf):
            for n, off, k, _ in self.segments:
                a, b = max(lo, off), min(hi, off + k)
                if a < b:
                    part[a - lo:b - lo].copy_(named[n].reshape(-1)[a - off:b - off])
        return buf

    def _check_hyper(self, betas, eps, what):
        if tuple(float(b) for b in betas) != tuple(float(b) for b in self.betas) or float(eps) != self.eps:
            raise NvsfError(f"{what}: betas {tuple(betas)} / eps {eps} != this optimizer's {tuple(self.betas)} / "
                            f"{self.eps}")

    def _set_step(self, step):
        # nvsf_adam_begin recomputes the bias corrections from the applied count state[0]
        self.state.zero_()
        self.state[0] = float(step)
        self.step_count = int(step)

    @torch.no_grad()
    def state_dict(self):
        """Adam and EMA state keyed by parameter name, in the parameters' shapes: {"step" (applied steps),
        "lr" (of the latest step), "betas", "eps", "exp_avg", "exp_avg_sq", "ema" (None without
        ema_decay), "ema_decay", "ema_num_updates"}.  When sharded this is a collective and every rank
        returns the full state, so it loads at any world size."""
        out = {"step": self.applied_steps(), "lr": self.last_lr, "betas": tuple(self.betas), "eps": self.eps,
               "ema_decay": self.ema_decay, "ema_num_updates": self.ema_num_updates}
        for key in ("exp_avg", "exp_avg_sq", "ema"):
            buf = getattr(self, key)
            out[key] = None if buf is None else self._gathered(buf)
        return out

    @torch.no_grad()
    def load_state_dict(self, sd):
        """Load a state_dict() (saved at any world size): this rank copies its owned ranges.  Names, shapes,
        betas and eps must match (NvsfError otherwise); the model's parameters are not touched."""
        self._check_hyper(sd["betas"], sd["eps"], "state_dict")
        keys = ("exp_avg", "exp_avg_sq") + (("ema",) if self.ema is not None else ())
        if self.ema is not None and sd.get("ema") is None:
            raise NvsfError("state_dict holds no EMA weights, but this FlatAdam has ema_decay set")
        new = {key: self._owned_from_named(sd[key], key) for key in keys}
        for key in keys:
            getattr(self, key).copy_(new[key])
        if self.ema is not None:
            self.ema_decay, self.ema_num_updates = float(sd["ema_decay"]), sd["ema_num_updates"]
        self._set_step(sd["step"])
        self.lr = self.last_lr = float(sd["lr"])

    # ------------------------------------------------------------------ reference checkpoint layouts
    def _reference_slices(self):
        """{reference key: (parameter name, offset, numel, shape)} of the hot-path keys (NeRFNetwork._reference_keys)."""
        return {k: (name, off, n, tuple(shape)) for k, name, off, n, shape in self.model._reference_keys()}

    def _named_from_reference(self, tensors, what):
        """{parameter name: tensor} assembled from {reference key: tensor}; every hot-path key is required."""
        shapes = self._shapes()
        out = {n: torch.empty(s, device=self.flat.device) for n, s in shapes.items()}
        for key, (name, off, n, shape) in self._reference_slices().items():
            v = tensors.get(key)
            if v is None:
                raise NvsfError(f"{what}: reference state lacks {key}")
            if tuple(v.shape) != shape:
                raise NvsfError(f"{what}[{key}]: shape {tuple(v.shape)} != {shape}")
            out[name].view(-1)[off:off + n].copy_(v.reshape(-1))
        return out

    @torch.no_grad()
    def load_reference_optimizer_state(self, sd):
        """Load the reference checkpoint's "optimizer" entry (`torch.load(path)["optimizer"]` or the whole
        checkpoint): torch.optim.Adam's state dict over the reference's 11 parameter groups
        (NeRFNetwork.reference_param_groups).  Every hot-path parameter needs state with one common step
        (a tensor or a number); the zero-size view encodings may have none.  Betas and eps must equal this
        optimizer's.  Sets lr to the first group's (whose factor is 1)."""
        if "param_groups" not in sd and "optimizer" in sd:
            sd = sd["optimizer"]
        groups, pg = self.model.reference_param_groups(), sd["param_groups"]
        if len(pg) != len(groups) or any(len(a["params"]) != len(b["params"]) for a, b in zip(pg, groups)):
            raise NvsfError(f"optimizer state has groups of sizes {[len(g['params']) for g in pg]}, the reference's "
                            f"are {[len(g['params']) for g in groups]}")
        for g in pg:
            self._check_hyper(g["betas"], g["eps"], "reference optimizer")
        hot = self._reference_slices()
        moments, steps = {"exp_avg": {}, "exp_avg_sq": {}}, set()
        for g, rg in zip(pg, groups):
            for idx, key in zip(g["params"], rg["params"]):
                if key not in hot:
                    continue
                st = sd["state"].get(idx)
                if st is None:
                    raise NvsfError(f"reference optimizer state lacks {key}")
                steps.add(float(st["step"]))
                for m in moments:
                    moments[m][key] = st[m]
        if len(steps) != 1:
            raise NvsfError(f"reference optimizer state has different steps {sorted(steps)[:4]}")
        new = {m: self._owned_from_named(self._named_from_reference(moments[m], m), m) for m in moments}
        self.exp_avg.copy_(new["exp_avg"])
        self.exp_avg_sq.copy_(new["exp_avg_sq"])
        self._set_step(int(steps.pop()))
        self.lr = self.last_lr = float(pg[0]["lr"]) / groups[0]["lr"]

    @torch.no_grad()
    def reference_optimizer_state_dict(self):
        """torch.optim.Adam's state dict of the reference's optimizer (the "optimizer" entry of its
        checkpoint): group lr = the latest lr x LR_SCALE, no state for the zero-size parameters (torch
        creates none for a parameter without gradient).  A collective when sharded."""
        step = float(self.applied_steps())
        avg, avg_sq = self._gathered(self.exp_avg), self._gathered(self.exp_avg_sq)
        hot = self._reference_slices()
        state, param_groups, idx = {}, [], 0
        for rg in self.model.reference_param_groups():
            ids = []
            for key in rg["params"]:
                if key in hot:
                    name, off, n, shape = hot[key]
                    state[idx] = {"step": torch.tensor(step),       # one tensor per parameter, as torch keeps it
                                  "exp_avg": avg[name].reshape(-1)[off:off + n].view(shape),
                                  "exp_avg_sq": avg_sq[name].reshape(-1)[off:off + n].view(shape)}
                ids.append(idx)
                idx += 1
            param_groups.append({"lr": self.last_lr * rg["lr"], "betas": tuple(self.betas), "eps": self.eps,
                                 "weight_decay": 0, "amsgrad": False, "params": ids})
        return {"state": state, "param_groups": param_groups}

    @torch.no_grad()
    def load_reference_ema_state(self, sd):
        """Load the reference checkpoint's "ema" entry (torch_ema.ExponentialMovingAverage.state_dict(), or
        the whole checkpoint): shadow_params in the reference's model.parameters() order
        (NeRFNetwork.reference_parameters); count and shapes are checked, the hot-path entries used."""
        if "shadow_params" not in sd and "ema" in sd:
            sd = sd["ema"]
        self._need_ema()
        ref, shadow = self.model.reference_parameters(), sd["shadow_params"]
        if len(shadow) != len(ref):
            raise NvsfError(f"EMA state has {len(shadow)} shadow parameters, the reference model {len(ref)}")
        for (key, shape), t in zip(ref, shadow):
            if tuple(t.shape) != tuple(shape):
                raise NvsfError(f"EMA shadow of {key}: shape {tuple(t.shape)} != {tuple(shape)}")
        named = self._named_from_reference({key: t for (key, _), t in zip(ref, shadow)}, "ema")
        self.ema.copy_(self._owned_from_named(named, "ema"))
        num = sd["num_updates"]
        self.ema_decay, self.ema_num_updates = float(sd["decay"]), None if num is None else int(num)

    @torch.no_grad()
    def reference_ema_state_dict(self):
        """torch_ema's state dict of the reference trainer's EMA: the parameters the B200 model does not have
        (un-suffixed planes_encoder / hash_encoder, the (0,) view encodings) are zeros of their shape.
        A collective when sharded."""
        self._need_ema()
        named, hot = self._gathered(self.ema), self._reference_slices()
        shadow = []
        for key, shape in self.model.reference_parameters():
            if key in hot:
                name, off, n, _ = hot[key]
                shadow.append(named[name].reshape(-1)[off:off + n].view(shape))
            else:
                shadow.append(torch.zeros(shape, device=self.flat.device))
        return {"decay": self.ema_decay, "num_updates": self.ema_num_updates, "shadow_params": shadow,
                "collected_params": None}
