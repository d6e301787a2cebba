"""TEST INFRASTRUCTURE.  Pure-PyTorch stand-in for the `tinycudann` module.

tiny-cuda-nn is an un-vendored, un-pinned dependency of the reference
(`git+https://github.com/NVlabs/tiny-cuda-nn/#subdirectory=bindings/torch`, reference
setup.py:98, readme.md:62) and cannot be installed here (no network, no source).  This file
restates the PUBLISHED algorithm of the four pieces the reference uses so that the
reference's own field code (hash_field.py, flow_field.py, network_dynamic.py) can be imported
by path and run on CPU.  PARITY UNPINNED for these pieces: nothing in the reference tests
them and tcnn itself is not available to compare against.

Call sites reproduced: hash_field.py:47-57,109-119 and flow_field.py:70-80 (HashGrid),
network_dynamic.py:108-114 (Frequency), :165-170 (SphericalHarmonics), :125-189 (FullyFusedMLP).

Semantics (tcnn `grid.h`, `frequency.h`, `spherical_harmonics.h`, `fully_fused_mlp.cu`):
  HashGrid   per level l: scale = exp2(l*log2(per_level_scale))*base - 1, res = ceil(scale)+1,
             level size = min(next_multiple(res^D, 8), 2^log2_hashmap_size) entries of F features;
             pos = scale*x + 0.5; cell = floor(pos); w = pos - cell; D-linear interpolation over
             the 2^D corners; corner index = sum_d cell_d*res^d (dense) when res^D <= size,
             else xor_d(cell_d*prime_d) with primes (1, 2654435761, 805459861); index %= size;
             output feature order is level-major.  Parameters are an fp32 master copy used in
             fp16 (here: rounded to fp16, arithmetic in fp32).
  Frequency  out[j] = sin(2^((j//2) % n_freq) * pi * x[j // (2 n_freq)] + (j % 2) * pi/2), n_freq=12.
  SH deg 4   16 real spherical-harmonics polynomials of 2x-1.
  FullyFusedMLP  weights row-major [out, in] per layer, input width padded to a multiple of 16,
             output padded to 16, no biases, ReLU hidden, linear output; fp16
             weights/activations (here: weights, inputs and every layer's output rounded to fp16,
             products accumulated in fp32 — tcnn's fully fused path even accumulates in fp16).
  Network    the torch binding's `tcnn.Network(n_in, n_out, cfg)` is `create_network`, which wraps
             the MLP in a NetworkWithInputEncoding with an "Identity" encoding (tcnn cpp_api.cu);
             tcnn's encodings fill their padded outputs with the constant 1 (identity.h: "data_out(j, i)
             = 1" for the padded columns; frequency.h documents "padding (value 1.f)"), so the padded
             INPUT columns of the MLP are 1 and the weight columns behind them act as a learned
             first-layer bias.  (Restated from the published source from memory: tcnn is not vendored.)
Outputs are returned as float32 (tcnn returns fp16): the comparison tolerance for anything that
passes through these modules is 1e-2 (BASELINE.json north_star), which covers that difference.
"""
import math

import numpy as np
import torch
import torch.nn as nn

PRIMES = (1, 2654435761, 805459861)


def grid_levels(n_dims, n_levels, base_resolution, per_level_scale, log2_hashmap_size):
    """Per-level (scale, resolution, size, offset) exactly as tcnn's GridEncoding derives them."""
    log2_pls = np.log2(np.float32(per_level_scale), dtype=np.float32)
    levels, offset = [], 0
    for l in range(n_levels):
        scale = np.float32(np.exp2(np.float32(l) * log2_pls, dtype=np.float32) * np.float32(base_resolution)
                           - np.float32(1.0))
        res = int(np.ceil(scale)) + 1
        dense = res ** n_dims
        size = min(dense, (2 ** 32 - 1) // 2)
        size = (size + 7) // 8 * 8
        size = min(size, 1 << log2_hashmap_size)
        levels.append(dict(scale=float(scale), res=res, size=size, offset=offset, hashed=dense > size))
        offset += size
    return levels, offset


def _fp16_round(p):
    return p.to(torch.float16).to(torch.float32)


class _HashGrid(nn.Module):
    def __init__(self, n_input_dims, cfg):
        super().__init__()
        self.D = n_input_dims
        self.L = int(cfg["n_levels"])
        self.F = int(cfg["n_features_per_level"])
        self.levels, total = grid_levels(self.D, self.L, cfg["base_resolution"], cfg["per_level_scale"],
                                         int(cfg["log2_hashmap_size"]))
        self.n_output_dims = self.L * self.F
        p = torch.empty(total * self.F, dtype=torch.float32).uniform_(-1e-4, 1e-4)
        self.params = nn.Parameter(p)

    def forward(self, x):
        # float32 like tcnn; float64 inputs stay float64 (tests/test_encoder_bwd_oracle.py differentiates the
        # encoders in float64) — the table is still the fp16-rounded parameters either way
        dt = torch.float64 if x.dtype == torch.float64 else torch.float32
        x = x.to(dt)
        N = x.shape[0]
        table = _fp16_round(self.params).to(dt).view(-1, self.F)
        outs = []
        for lv in self.levels:
            pos = x * np.float32(lv["scale"]) + 0.5
            cell = torch.floor(pos)
            w = pos - cell
            cell = cell.to(torch.int64)
            acc = torch.zeros(N, self.F, dtype=dt)
            for corner in range(1 << self.D):
                weight = torch.ones(N, dtype=dt)
                idx_dense = torch.zeros(N, dtype=torch.int64)
                idx_hash = torch.zeros(N, dtype=torch.int64)
                stride = 1
                for d in range(self.D):
                    bit = (corner >> d) & 1
                    c = (cell[:, d] + bit) & 0xFFFFFFFF          # uint32 wrap like the CUDA cast
                    weight = weight * (w[:, d] if bit else (1 - w[:, d]))
                    idx_dense = (idx_dense + c * stride) & 0xFFFFFFFF
                    idx_hash = idx_hash ^ ((c * PRIMES[d]) & 0xFFFFFFFF)
                    stride *= lv["res"]
                idx = (idx_hash if lv["hashed"] else idx_dense) % lv["size"]
                acc = acc + weight[:, None] * table[lv["offset"] + idx]
            outs.append(acc)
        return torch.cat(outs, dim=-1)


class _Frequency(nn.Module):
    def __init__(self, n_input_dims, cfg):
        super().__init__()
        self.n_freq = int(cfg.get("n_frequencies", 12))  # "degree" is not a tcnn key; default applies
        self.n_output_dims = n_input_dims * self.n_freq * 2
        self.params = nn.Parameter(torch.zeros(0))

    def forward(self, x):
        x = x.to(torch.float64)
        j = torch.arange(self.n_output_dims)
        feat = j // (2 * self.n_freq)
        log2f = (j // 2) % self.n_freq
        phase = (j % 2).to(torch.float64) * (math.pi / 2)
        arg = x[:, feat] * (2.0 ** log2f.to(torch.float64)) * math.pi + phase
        return torch.sin(arg).to(torch.float32)


def sh4(d):
    """16 real SH basis values of unit-ish vectors d (already mapped to [-1,1])."""
    x, y, z = d[:, 0], d[:, 1], d[:, 2]
    xy, xz, yz, x2, y2, z2 = x * y, x * z, y * z, x * x, y * y, z * z
    return torch.stack([
        torch.full_like(x, 0.28209479177387814),
        -0.48860251190291987 * y, 0.48860251190291987 * z, -0.48860251190291987 * x,
        1.0925484305920792 * xy, -1.0925484305920792 * yz,
        0.94617469575755997 * z2 - 0.31539156525251999, -1.0925484305920792 * xz,
        0.54627421529603959 * x2 - 0.54627421529603959 * y2,
        0.59004358992664352 * y * (-3.0 * x2 + y2), 2.8906114426405538 * xy * z,
        0.45704579946446572 * y * (1.0 - 5.0 * z2), 0.3731763325901154 * z * (5.0 * z2 - 3.0),
        0.45704579946446572 * x * (1.0 - 5.0 * z2), 1.4453057213202769 * z * (x2 - y2),
        0.59004358992664352 * x * (-x2 + 3.0 * y2)], dim=-1)


class _SphericalHarmonics(nn.Module):
    def __init__(self, n_input_dims, cfg):
        super().__init__()
        assert int(cfg.get("degree", 4)) == 4 and n_input_dims == 3
        self.n_output_dims = 16
        self.params = nn.Parameter(torch.zeros(0))

    def forward(self, x):
        return sh4(x.to(torch.float32) * 2.0 - 1.0)


def Encoding(n_input_dims, encoding_config, **_):
    otype = encoding_config["otype"]
    if otype == "HashGrid":
        return _HashGrid(n_input_dims, encoding_config)
    if otype == "Frequency":
        return _Frequency(n_input_dims, encoding_config)
    if otype == "SphericalHarmonics":
        return _SphericalHarmonics(n_input_dims, encoding_config)
    raise NotImplementedError(otype)


def mlp_layer_shapes(n_in, n_out, n_neurons, n_hidden_layers):
    pad_in = (n_in + 15) // 16 * 16
    pad_out = (n_out + 15) // 16 * 16
    shapes = [(n_neurons, pad_in)] + [(n_neurons, n_neurons)] * (n_hidden_layers - 1) + [(pad_out, n_neurons)]
    return shapes


class Network(nn.Module):
    def __init__(self, n_input_dims, n_output_dims, network_config, **_):
        super().__init__()
        assert network_config["otype"] == "FullyFusedMLP" and network_config["activation"] == "ReLU"
        assert network_config["output_activation"] == "None"
        self.n_input_dims, self.n_output_dims = n_input_dims, n_output_dims
        self.shapes = mlp_layer_shapes(n_input_dims, n_output_dims, int(network_config["n_neurons"]),
                                       int(network_config["n_hidden_layers"]))
        chunks = []
        for (o, i) in self.shapes:
            bound = math.sqrt(6.0 / (o + i))
            chunks.append(torch.empty(o * i, dtype=torch.float32).uniform_(-bound, bound))
        self.params = nn.Parameter(torch.cat(chunks))

    def forward(self, x):
        # tcnn is a native extension: an enclosing torch.autocast region does not change its arithmetic
        with torch.autocast("cpu", enabled=False):
            return self._forward(x)

    def _forward(self, x):
        x = x.to(torch.float32)
        pad = self.shapes[0][1] - x.shape[1]
        h = torch.nn.functional.pad(x, (0, pad), value=1.0) if pad else x   # Identity-encoding padding = 1
        h = _fp16_round(h)                    # the Identity encoding writes network_precision_t = __half
        w_all = _fp16_round(self.params)
        off = 0
        for li, (o, i) in enumerate(self.shapes):
            W = w_all[off:off + o * i].view(o, i)
            off += o * i
            h = h @ W.t()
            if li != len(self.shapes) - 1:
                h = torch.relu(h)
            h = _fp16_round(h)                # activations live in shared memory as __half; the output is __half
        return h[:, :self.n_output_dims]
