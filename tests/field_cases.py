"""Shared helpers for field parity tests (oracle side)."""
import importlib

import numpy as np
import torch

S = importlib.import_module("selfsupervised-nvsf_b200.synth")
_cache = {}


def oracle_config(density_scale=1.0, **kw):
    from oracle.field_oracle import FieldConfig
    return FieldConfig(bound=S.BOUND, num_frames=S.NUM_FRAMES, time_resolution=S.TIME_RESOLUTION,
                       min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH,
                       density_scale=density_scale, **kw)


def oracle_params(seed=0, style="trained"):
    """Full-size parameters (62 M floats) from the numpy-seeded initialiser; cached per process."""
    key = (seed, style)
    if key not in _cache:
        from oracle import field_init
        _cache[key] = field_init.make_params(oracle_config(), seed=seed, style=style)
    return _cache[key]


def rel_err(a, b, floor=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float((np.abs(a - b) / (np.abs(b) + floor)).max())


def ulp16(a, b):
    """|a - b| in units of the fp16 spacing at |b| (2^(e-10), e = exponent of b; subnormal spacing 2^-24).
    MLP outputs of the reference are half-precision values (tcnn returns __half, the flow MLP runs under
    fp16 autocast): two correct evaluations whose fp32 accumulators differ in the last bit may round to
    neighbouring fp16 values."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    e = np.floor(np.log2(np.maximum(np.abs(b), 2.0 ** -14)))
    return np.abs(a - b) / 2.0 ** (e - 10)


def assert_fp16_close(a, b, what, max_ulp=2.0, max_frac=0.02):
    """Equal up to `max_ulp` fp16 spacings of the tensor's largest magnitude (one flipped fp16 rounding of a
    hidden activation moves every output of that row by about that much), and different at all in at most
    `max_frac` of the entries."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    spacing = 2.0 ** (np.floor(np.log2(max(float(np.abs(b).max()), 2.0 ** -14))) - 10)
    d = np.abs(a - b)
    assert d.max() <= max_ulp * spacing, (what, "fp16 spacings", float(d.max() / spacing))
    assert (d > 0).mean() <= max_frac, (what, "fraction of entries that differ", float((d > 0).mean()))


# ---- gradient cases (tests/golden/field_grad_ref.npz, oracle/make_golden_grad.py) -------------------
LOSS_SCALE = 4096.0
GRAD_CASES = ["l_mid", "c_mid", "l_first", "c_last"]
GRAD_SHARED = ("flow_grid", "flow_mlp", "sigma_net", "intensity_net", "raydrop_net", "color_net")
GRAD_NAMES = ("hash_static", "hash_dynamic", "planes") + GRAD_SHARED


def grad_case(gold, tag):
    k = tag + "_"
    lidar, t, ds, perturb = gold[k + "meta"].tolist()
    return dict(lidar=bool(lidar), t=float(t), ds=float(ds), o=gold[k + "o"], d=gold[k + "d"],
                noise=gold[k + "noise"] if perturb else None,
                coef={n: gold[k + "coef_" + n] for n in "abce"})


def linear_loss(out, coef, to=lambda a: torch.from_numpy(a)):
    """The fixed functional of the render outputs the gradient goldens were taken for."""
    n = coef["a"].shape[0]
    return ((to(coef["a"]) * out["depth"].reshape(-1)).sum() + (to(coef["b"]) * out["image"].reshape(n, -1)).sum()
            + (to(coef["c"]) * out["weights"]).sum() + (to(coef["e"]) * out["weights_sum"]).sum())


def oracle_grads(case, params=None, bg_color=1.0):
    """Autograd gradients of the CPU oracle for one gradient case, in the flat parameter layout (camera:
    background `bg_color`, a number or an [N,3] tensor)."""
    from oracle.field_oracle import FieldOracle
    from oracle import raymarching_oracle as RO
    base = params if params is not None else oracle_params()
    mod = "lidar" if case["lidar"] else "camera"
    leaf = {mod: {k: v.clone().requires_grad_(True) for k, v in base[mod].items()}}
    for k in GRAD_SHARED:
        leaf[k] = base[k].clone().requires_grad_(True)
    orc = FieldOracle(oracle_config(density_scale=case["ds"]), leaf)
    nears = fars = None
    if not case["lidar"]:
        n, f = RO.near_far_from_aabb(case["o"], case["d"], S.AABB, S.MIN_NEAR)
        nears, fars = torch.from_numpy(n), torch.from_numpy(f)
    S_ = case["coef"]["c"].shape[1]
    out = orc.run(torch.from_numpy(case["o"]), torch.from_numpy(case["d"]), case["t"], case["lidar"], S_, nears,
                  fars, None if case["noise"] is None else torch.from_numpy(case["noise"]), bg_color=bg_color)
    loss = linear_loss(out, case["coef"])
    (loss * LOSS_SCALE).backward()   # the goldens were taken with this loss scale (oracle/make_golden_grad.py)
    un = lambda v: (v.grad / LOSS_SCALE if v.grad is not None else torch.zeros_like(v)).numpy()
    g = {k: un(v) for k, v in leaf[mod].items()}
    for k in GRAD_SHARED:
        g[k] = un(leaf[k])
    return g, float(loss.item()), out


_floor_cache = {}


def oracle_grad_floor(case, tag):
    """Conditioning of the reference gradient itself: relative L2 change of every parameter gradient of the
    CPU oracle when the ray origins move by ONE fp32 ulp.  The finest hash levels have 32768 cells per unit
    (a 1-ulp move of a coordinate shifts the interpolation weights by ~0.3 %) and every MLP stores fp16
    activations whose rounding may flip, so the gradient of this field is only defined to 1-3 %: no
    implementation that evaluates o + z d in a different but equally valid fp32 order can agree better."""
    if tag not in _floor_cache:
        g0, _, _ = oracle_grads(case)
        moved = dict(case, o=np.nextafter(case["o"], np.float32(10.0)).astype(np.float32))
        g1, _, _ = oracle_grads(moved)
        _floor_cache[tag] = {k: float(np.linalg.norm(g1[k].astype(np.float64) - g0[k]) /
                                      max(np.linalg.norm(g0[k].astype(np.float64)), 1e-30)) for k in g0}
    return _floor_cache[tag]


def check_grad_summary(gold, tag, name, g, rtol, what):
    """Compare a full gradient tensor with the fixture's summary of the reference gradient."""
    k = f"{tag}_g_{name}_"
    idx, val, l2 = gold[k + "idx"], gold[k + "val"], float(gold[k + "l2"])
    if l2 == 0.0:
        assert not np.any(g), (what, tag, name, "expected an all-zero gradient")
        return
    got = np.asarray(g, np.float64).reshape(-1)
    err = np.sqrt(((got[idx] - val.astype(np.float64)) ** 2).sum()) / np.sqrt((val.astype(np.float64) ** 2).sum())
    assert err < rtol, (what, tag, name, "sampled entries", err)
    assert abs(np.sqrt((got ** 2).sum()) - l2) < rtol * l2, (what, tag, name, "l2", np.sqrt((got ** 2).sum()), l2)
    # an error vector of norm rtol*l2 over nnz entries changes the sum by at most rtol*l2*sqrt(nnz)
    bound = rtol * max(l2 * np.sqrt(float(gold[k + "nnz"])), abs(float(gold[k + "sum"])))
    assert abs(got.sum() - float(gold[k + "sum"])) < bound, (what, tag, name, "sum")
