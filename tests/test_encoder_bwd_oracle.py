"""The float64 restatement of the encoder / flow-grid backward (oracle/encoder_bwd_oracle.py) against
torch.autograd in float64 of field_oracle's own encoder functions, on a shrunken field (dense and hashed
levels, four plane scales).  Both sides get the same float64 positions and the same per-sample gradients,
so they may differ by float64 rounding only: this pins the semantics, the corner order, the layouts and
grid_sample's border rule that tests/test_encoder_bwd_gpu.py then holds the CUDA kernels to."""
import numpy as np
import pytest
import torch

import field_cases as FC
from oracle import encoder_bwd_oracle as EB
from oracle import field_init
from oracle import field_oracle as FO
from oracle import tcnn_standin as TS


def small_config():
    return FC.oracle_config(min_resolution=6, base_resolution=16, max_resolution=512, log2_hashmap_size=12,
                            hash_size_dynamic=(10, 9, 9), flow_base=8, flow_max=256, flow_log2=11)


def make_params(cfg, h16):
    p = field_init.make_params(cfg, seed=3)
    out = {}
    for k, v in p.items():
        out[k] = {kk: vv.double() for kk, vv in v.items()} if isinstance(v, dict) else v.double()
    if h16:
        # the fp16 texels of the product rule: space planes fp16-exact and time planes constant along t,
        # so that the restatement's fp16 mirror of a time-collapsed row is the row the torch side blends
        for mod in ("lidar", "camera"):
            flat = out[mod]["planes"].float().half().double()
            off = 0
            for r in cfg.plane_res:
                for (a, b) in FO.PLANE_COMBS:
                    n = cfg.n_features_plane * r[a] * r[b]
                    if b == 3:
                        g = flat[off:off + n].view(cfg.n_features_plane, r[b], r[a])
                        g[:] = g[:, :1, :].clone()
                    off += n
            out[mod]["planes"] = flat
    return out


def make_samples(n, seed, x_on_one):
    """World positions: random inside the box, some on the -bound and +bound faces; flow that pushes warped
    queries outside [0, 1] and, for `x_on_one` rows, lands them exactly on 1.0."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-2.0, 2.0, size=(n, 3))
    x[: n // 16, 0] = 2.0
    x[n // 16: n // 8, 1] = -2.0
    x[n // 8: n // 8 + n // 16, 2] = 2.0
    flow = rng.normal(0.0, 0.02, size=(n, 6))
    flow[-n // 8:] *= 20.0                       # far outside the box
    xn = (x + 2.0) / 4.0
    i = np.arange(n)[x_on_one]
    for c in range(6):
        sel = i[(xn[i, c % 3] >= 0.5)]
        flow[sel, c] = 1.0 - xn[sel, c % 3]      # exact in float64 (Sterbenz): xn + flow == 1.0
        assert (xn[sel, c % 3] + flow[sel, c] == 1.0).all()
    return x, xn, flow


def torch_grads(cfg, params, mod, x, t, flow, dfeat, dflowfeat):
    """d/d(tables) of <features, dfeat> + <flow-MLP input, dflowfeat>, and d/d(flow) — field_oracle in float64."""
    # fp16 table values as in the stand-in, but a float64 gradient: the stand-in's cast would also round the
    # gradient to fp16 (like tcnn's half atomics), which the fp32 backward does not do
    real_round = TS._fp16_round
    TS._fp16_round = lambda p: p + (real_round(p).to(p.dtype) - p).detach()
    try:
        return _torch_grads(cfg, params, mod, x, t, flow, dfeat, dflowfeat)
    finally:
        TS._fp16_round = real_round


def _torch_grads(cfg, params, mod, x, t, flow, dfeat, dflowfeat):
    leaf = {mod: {k: v.clone().requires_grad_(True) for k, v in params[mod].items()},
            "flow_grid": params["flow_grid"].clone().requires_grad_(True), "flow_mlp": params["flow_mlp"]}
    fl = torch.from_numpy(flow).clone().requires_grad_(True)
    orc = FO.FieldOracle(cfg, leaf)
    orc.flow_net = lambda xn, t_: fl
    feats, _ = orc.features(torch.from_numpy(x), t, mod == "lidar")
    loss = (feats * torch.from_numpy(dfeat[:, :120])).sum()
    real_mlp = FO.mlp
    FO.mlp = lambda flat, shapes, h, n_out, fp16_weights=True: h   # flow_net up to the flow MLP's input
    try:
        h = FO.FieldOracle(cfg, leaf).flow_net(torch.from_numpy((x + cfg.bound) / (2 * cfg.bound)), t)
    finally:
        FO.mlp = real_mlp
    loss = loss + (h * torch.from_numpy(dflowfeat)).sum()
    loss.backward()
    g = {k: leaf[mod][k].grad.numpy() for k in ("hash_static", "hash_dynamic", "planes")}
    g["flow_grid"] = leaf["flow_grid"].grad.numpy()
    return g, fl.grad.numpy()


CASES = [  # (t, what it exercises)
    (0.0, "frame 0: no previous frame (valid2 = 0)"),
    (1.0, "last frame: no next frame (valid1 = 0)"),
    (float(np.float32(3 / 7)), "t * (T-1) an integer in fp32: k1 == k2"),
    (0.37, "interior t"),
]


@pytest.mark.parametrize("h16", [False, True])
@pytest.mark.parametrize("t", [c[0] for c in CASES])
@pytest.mark.parametrize("mod", ["lidar", "camera"])
def test_restatement_matches_autograd_float64(mod, t, h16):
    cfg = small_config()
    params = make_params(cfg, h16)
    n = 2048
    rng = np.random.default_rng(7)
    x, xn, flow = make_samples(n, 11, rng.random(n) < 0.25)
    dfeat = rng.normal(size=(n, 128))
    dflowfeat = rng.normal(size=(n, 32))
    dgeo16 = rng.normal(size=(n, 16)).astype(np.float32)
    dgeo16[rng.random(n) < 0.2] = 0.0       # dead rows: zero sigma-net output gradient ...
    dflow = rng.normal(size=(n, 8)).astype(np.float32)
    dflow[rng.random(n) < 0.2] = 0.0
    live, flive = EB.row_live(dgeo16, 1.0), EB.row_live(dflow[:, :6], 1.0)
    assert 0 < live.sum() < n and 0 < flive.sum() < n
    dfeat_k, dflowfeat_k = dfeat.copy(), dflowfeat.copy()
    dfeat_k[~live] = np.nan                  # ... whose dfeat / dflowfeat the backward never writes
    dflowfeat_k[~flive] = np.nan
    r = EB.encoder_bwd(cfg, params, mod, xn, t, np.concatenate([flow, np.zeros((n, 2))], 1), dfeat_k, dgeo16,
                       dflow, dflowfeat_k, 1.0, 1.0, h16=h16, exact=True)
    dfeat[~live] = 0.0
    dflowfeat[~flive] = 0.0
    g, gflow = torch_grads(cfg, params, mod, x, t, flow, dfeat, dflowfeat)
    for name in ("hash_static", "hash_dynamic", "planes", "flow_grid"):
        got, A, k = r["grads"][name]
        want = g[name].astype(np.float64)
        assert np.isfinite(got).all() and np.isfinite(A).all(), name
        assert ((A == 0) == (k == 0)).all(), name
        assert (got[A == 0] == 0).all(), name
        scale = np.abs(want).max()
        assert scale > 0, name
        err = np.abs(got - want).max()
        assert err <= 1e-12 * scale, (name, err, scale)
        # A bounds the entry and is not far above it where the terms do not cancel
        assert (np.abs(want) <= A * (1 + 1e-12) + 1e-300).all(), name
    # the only gradient the flow field gets: the coordinate gradient of the warped plane queries
    want = gflow
    assert np.abs(want).max() > 0
    assert np.abs(r["dflow"] - want).max() <= 1e-12 * np.abs(want).max(), np.abs(r["dflow"] - want).max()
    assert (np.abs(want) <= r["dflow_abs"] * (1 + 1e-12) + 1e-300).all()
    if t == 0.0:
        assert not want[:, 3:].any()         # no previous frame: no backward-flow gradient
    if t == 1.0:
        assert not want[:, :3].any()


def test_edge_samples_are_present():
    """The samples of the test above reach the edges the restatement has to get right."""
    cfg = small_config()
    n = 2048
    rng = np.random.default_rng(7)
    x, xn, flow = make_samples(n, 11, rng.random(n) < 0.25)
    q = xn[:, [0, 1, 2, 0, 1, 2]] + flow
    assert (xn == 1.0).any() and (xn == 0.0).any()       # samples on the +bound and -bound faces
    assert (q == 1.0).sum() > 50                          # warped queries exactly on the last texel
    assert (q < 0).any() and (q > 1).any()                # ... and outside [0, 1]
    # dense levels whose +1 corner of a +bound sample wraps (tcnn's % size)
    lv = [l for l in cfg.static_levels if not l["hashed"]]
    assert lv and lv[-1]["res"] ** 3 >= lv[-1]["size"] - 7
    assert any(l["hashed"] for l in cfg.static_levels)


def test_positions_and_fractions_are_the_kernel_fp32_arithmetic():
    """fp32 mode: positions via fma(d, z, o) and grid positions via fma(scale, x, 0.5); the emulated FMA
    rounds once (checked against exact rational arithmetic on random operands)."""
    from fractions import Fraction
    rng = np.random.default_rng(1)
    a, b, c = (rng.normal(size=2000).astype(np.float32) for _ in range(3))
    got = EB.fma32(a, b, c)
    for i in range(0, 2000, 7):
        exact = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        lo = np.float32(float(exact))
        cand = [np.nextafter(lo, np.float32(-np.inf)), lo, np.nextafter(lo, np.float32(np.inf))]
        best = min(cand, key=lambda v: (abs(Fraction(float(v)) - exact), int(np.float32(v).view(np.uint32)) & 1))
        assert got[i] == best, i
    z = EB.uniform_z(np.float32([0.01, 0.5]), np.float32([0.868, 3.0]), 768)
    assert z.dtype == np.float32 and (np.diff(z, axis=1) > 0).all()
    assert z[0, 0] == np.float32(0.01) and z[0, -1] == np.float32(0.868)
