"""Entry-by-entry check of the table gradients of the training backward (k_encode_bwd, k_flowgrid_bwd and the
k_expand_* transposes of the time collapse in csrc/train.cu) against the float64 restatement
oracle/encoder_bwd_oracle.py, fed the per-sample gradients the CUDA backward kept in its scratch buffer
(model._debug_keep): dfeat, dgeo16 and the sigma scale (liveness), dflow, dflowfeat and the flow scale, and the
forward's flow.  Those scatters are linear in what they are fed, so the only differences left are fp32 rounding
and the order of the atomic adds: every entry g of hash_static, hash_dynamic, planes and flow_grid must satisfy
|g - ref| <= 2^-16 * A (A: float64 sum of |terms| landing in that entry, about 256 fp32 ulps of it), entries
with A = 0 must be exactly zero, and the same bound holds per sample for the coordinate gradient dflow.

(tests/test_field_grad_gpu.py compares whole tensors in relative L2 at >= 1e-2 — the fp16 MLPs leave the CPU
oracle's own gradient only defined to 1-3 % — so an error in under ~1 % of a tensor's norm passes there.)

Also here: the camera background (bg_color 0, 0.3, a per-ray tensor) through k_composite_bwd and _split_bg."""
import ctypes
import importlib

import numpy as np
import pytest

import field_cases as FC
from oracle import encoder_bwd_oracle as EB
from oracle.field_oracle import PLANE_COMBS

torch = pytest.importorskip("torch")
S = FC.S
NAMES = ("hash_static", "hash_dynamic", "planes", "flow_grid")
BOUND_ULPS = 256.0            # |g - ref| <= BOUND_ULPS * 2^-24 * A
NOISE_EDGES = (0.0, float(np.float32(1.0) - np.float32(2.0 ** -24)))


# ---- cases -------------------------------------------------------------------------------------------------
def _rays(kind, N, seed):
    rng = np.random.default_rng(seed)
    if kind == "lidar":
        return S.lidar_rays(N, seed=seed)
    if kind == "camera":
        return S.camera_rays(N, seed=seed)
    if kind == "axis":
        # along +x with |d| chosen so that one sample step is 0.49 cells of static-hash level 2 (scale 1679):
        # 32 consecutive samples of a ray cover exactly 16 or exactly 17 cells of that level
        o = np.stack([rng.uniform(-0.6, -0.2, N), rng.uniform(-0.5, 0.5, N), rng.uniform(-0.5, 0.5, N)], 1)
        step = (np.float32(S.LIDAR_MAX_DEPTH) - np.float32(S.MIN_NEAR_LIDAR)) / 767 / (2 * S.BOUND)
        d = np.tile([0.49 / (1679.046875 * step), 0.0, 0.0], (N, 1))
        return o.astype(np.float32), d.astype(np.float32)
    if kind == "leave":
        # rays that leave the box through the +x, +y and +z faces: their last samples are clamped onto the faces
        o = rng.uniform(-0.3, 0.3, (N, 3))
        ax = np.arange(N) % 3
        o[np.arange(N), ax] = rng.uniform(1.45, 1.7, N)
        d = np.zeros((N, 3))
        d[np.arange(N), ax] = 1.0
        d += rng.normal(0, 0.05, (N, 3)) * (np.arange(N) % 2)[:, None]
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        return o.astype(np.float32), d.astype(np.float32)
    raise ValueError(kind)


# name: (lidar, ray kind, N, S, t, density_scale, noise, zero last flow layer, [(enc_bwd_h16, enc_bwd_ctas)])
CASES = {
    "lidar_256x768": (True, "lidar", 256, 768, 0.37, 60.0, True, False, [(1, 2), (0, 2), (1, 3), (0, 3)]),
    "camera_256x768_t0": (False, "camera", 256, 768, 0.0, 1.0, False, False, [(1, 2), (0, 3)]),
    "lidar_4099x1_t1": (True, "lidar", 4099, 1, 1.0, 1.0, True, False, [(1, 2), (0, 3)]),
    "camera_37x37_tslice": (False, "camera", 37, 37, float(np.float32(3 / 7)), 60.0, True, False, [(1, 3), (0, 2)]),
    "lidar_axis_16_17": (True, "axis", 64, 768, 0.61, 1.0, False, False, [(1, 2), (0, 3)]),
    "lidar_leave_box_t0": (True, "leave", 96, 256, 0.0, 1.0, True, False, [(1, 2), (0, 3)]),
    "camera_leave_box_zero_flow": (False, "leave", 96, 256, 0.37, 1.0, False, True, [(1, 2), (0, 2)]),
}


def make_case(name):
    lidar, kind, N, Sn, t, ds, perturb, zero_flow, opts = CASES[name]
    o, d = _rays(kind, N, seed=list(CASES).index(name) + 1)
    rng = np.random.default_rng(5)
    noise = None
    if perturb:
        noise = rng.random((N, Sn), dtype=np.float32)
        noise.reshape(-1)[::7] = NOISE_EDGES[0]
        noise.reshape(-1)[3::7] = NOISE_EDGES[1]
    nch = 2 if lidar else 3
    coef = dict(a=rng.normal(size=N).astype(np.float32), b=rng.normal(size=(N, nch)).astype(np.float32),
                c=(0.1 * rng.normal(size=(N, Sn))).astype(np.float32), e=rng.normal(size=N).astype(np.float32))
    for v in coef.values():
        v[::3] = 0.0                              # every third ray: no gradient at all
    return dict(lidar=lidar, N=N, S=Sn, t=t, ds=ds, o=o, d=d, noise=noise, coef=coef, zero_flow=zero_flow, opts=opts)


def _params(zero_flow):
    p = FC.oracle_params()
    if zero_flow:   # flow == 0: the warped queries sit on the un-warped ones, +bound samples exactly on 1.0
        p = dict(p)
        p["flow_mlp"] = p["flow_mlp"].clone()
        p["flow_mlp"][-6 * 64:] = 0
    return p


def geometry(case):
    """Host side of the sample positions (kernel fp32 arithmetic) and nears / fars as the model forms them."""
    N, Sn = case["N"], case["S"]
    if case["lidar"]:
        nears = np.full(N, S.MIN_NEAR_LIDAR, np.float32)
        fars = np.full(N, S.LIDAR_MAX_DEPTH, np.float32)
    else:
        from oracle import raymarching_oracle as RO
        nears, fars = RO.near_far_from_aabb(case["o"], case["d"], S.AABB, S.MIN_NEAR)
    x, z = EB.sample_positions(case["o"], case["d"], nears, fars, Sn, S.BOUND, case["noise"])
    return x, z, nears, fars


# ---- device run --------------------------------------------------------------------------------------------
def run_device(pkg, case, h16, ctas):
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    m = pkg.NeRFNetwork(time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND,
                        min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH,
                        density_scale=case["ds"], options={"enc_bwd_h16": h16, "enc_bwd_ctas": ctas})
    m.load_flat_params(_params(case["zero_flow"]))
    m.train()
    m._debug_keep = True
    lidar, sfx = case["lidar"], "_lidar" if case["lidar"] else ""
    out = m.render(dev(case["o"])[None], dev(case["d"])[None], torch.tensor([[case["t"]]], device="cuda"),
                   cal_lidar_color=lidar, staged=False, num_steps=case["S"],
                   noise=None if case["noise"] is None else dev(case["noise"]))
    std = dict(depth=out["depth" + sfx], image=out["image" + sfx], weights=out["weights"],
               weights_sum=out["weights_sum" + sfx])
    FC.linear_loss(std, case["coef"], to=dev).backward()
    torch.cuda.synchronize()
    mod = "lidar" if lidar else "camera"
    g = {n: getattr(m, f"{n}_{mod}" if n != "flow_grid" else n).grad for n in NAMES}
    g = {n: (np.zeros(1) if v is None else v.detach().double().cpu().numpy().reshape(-1)) for n, v in g.items()}
    N, Sn = m._debug["N"], m._debug["S"]
    n = N * Sn
    lay = (ctypes.c_size_t * 12)()
    F = importlib.import_module("selfsupervised-nvsf_b200.field")
    F._setup_lib().nvsf_render_uniform_debug_layout(ctypes.byref(m._cfg), N, Sn, lay)
    assert lay[10] >= N, "the backward ran in more than one chunk: only the last chunk's dfeat is kept"
    sc, sv = m._debug["scratch"], m._debug["saved"]

    def view(buf, off, cnt, w):
        return buf[off:off + cnt * w * 4].view(torch.float32).cpu().numpy().reshape(cnt, w)

    scales = sc[:64].view(torch.float32).cpu().numpy()   # BwdLayout::scales: 4 x {max bits, pad, scale, 1/scale}
    kept = dict(flow=view(sv, lay[2], n, 8), dgeo16=view(sc, lay[6], n, 16), dfeat=view(sc, lay[7], n, 128),
                dflow=view(sc, lay[8], n, 8), dflowfeat=view(sc, lay[9], n, 32),
                scale_sigma=float(scales[4 * 1 + 2]), scale_flow=float(scales[4 * 2 + 2]))
    return g, kept, out["z_vals"].detach().cpu().numpy()


# ---- comparison --------------------------------------------------------------------------------------------
def regions(cfg, name):
    """(label, start, stop) of the levels / scales of one master tensor."""
    if name == "hash_static":
        return [(f"L{i}", l["offset"] * 4, (l["offset"] + l["size"]) * 4) for i, l in enumerate(cfg.static_levels)]
    if name == "flow_grid":
        return [(f"L{i}", l["offset"] * 8, (l["offset"] + l["size"]) * 8) for i, l in enumerate(cfg.flow_grid_levels)]
    if name == "hash_dynamic":
        out, base = [], 0
        for p in range(3):
            per = cfg.dyn_entries[p] * 4
            for i, l in enumerate(cfg.dyn_levels[p]):
                # one level of plane p across all time slices: entries offset..offset+size of every slice
                idx = (base + np.arange(cfg.time_resolution)[:, None] * per + l["offset"] * 4
                       + np.arange(l["size"] * 4)[None, :]).reshape(-1)
                out.append((f"P{p}L{i}", idx, None))
            base += cfg.time_resolution * per
        return out
    out, off = [], 0
    for s, r in enumerate(cfg.plane_res):
        n = sum(8 * r[a] * r[b] for (a, b) in PLANE_COMBS)
        out.append((f"S{s}", off, off + n))
        off += n
    return out


def worst_ratio(got, ref, A, k):
    """max |g - ref| / (2^-24 A) over entries with A > 0, and the term count where it is reached."""
    nz = A > 0
    if not nz.any():
        return 0.0, 0
    r = np.abs(got[nz] - ref[nz]) / (2.0 ** -24 * A[nz])
    i = int(np.argmax(r))
    return float(r[i]), int(k[nz][i])


def check_case(name, case, cfg, h16, ctas, g, kept, ref, report):
    for tn in NAMES:
        rg, A, k = ref["grads"][tn]
        got = g[tn] if g[tn].size == rg.size else np.zeros_like(rg)
        zero = A == 0
        assert not got[zero].any(), (name, tn, "non-zero where no term lands", int((got[zero] != 0).sum()))
        per = []
        for label, a, b in regions(cfg, tn):
            sl = a if b is None else slice(a, b)
            per.append((label,) + worst_ratio(got[sl], rg[sl], A[sl], k[sl]))
        report.append(f"{name} h16={h16} ctas={ctas} {tn}: " +
                      " ".join(f"{lb}={r:.1f}(k={kk})" for lb, r, kk in per))
        bad = [(lb, r, kk) for lb, r, kk in per if r > BOUND_ULPS]
        assert not bad, (name, h16, ctas, tn, "entries off by more than 2^-16 A", bad)
    d, da = kept["dflow"][:, :6].astype(np.float64), ref["dflow_abs"]
    zero = da == 0
    assert not d[zero].any(), (name, "dflow non-zero where no term lands")
    r, kk = worst_ratio(d.reshape(-1), ref["dflow"].reshape(-1), da.reshape(-1), np.zeros(da.size, np.int64))
    report.append(f"{name} h16={h16} ctas={ctas} dflow: {r:.1f}")
    assert r <= BOUND_ULPS, (name, h16, ctas, "dflow", r)


_REPORT = []


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_table_gradients_entry_by_entry(pkg, name):
    case = make_case(name)
    cfg = FC.oracle_config(density_scale=case["ds"])
    x, z, nears, fars = geometry(case)
    mod = "lidar" if case["lidar"] else "camera"
    params = _params(case["zero_flow"])
    refs = {}
    for h16, ctas in case["opts"]:
        g, kept, zdev = run_device(pkg, case, h16, ctas)
        # the position arithmetic of the restatement is the kernels': z bit for bit
        assert np.array_equal(zdev.view(np.uint32), z.view(np.uint32)), (name, "z_vals differ")
        if h16 not in refs:
            refs[h16] = EB.encoder_bwd(cfg, params, mod, x, case["t"], kept["flow"], kept["dfeat"], kept["dgeo16"],
                                       kept["dflow"], kept["dflowfeat"], kept["scale_sigma"], kept["scale_flow"],
                                       h16=bool(h16))
            ref = refs[h16]
            assert ref["live"].any() and ref["flow_live"].any(), name
            _coverage(name, case, ref)
        check_case(name, case, cfg, h16, ctas, g, kept, refs[h16], _REPORT)
    print("\n" + "\n".join(_REPORT[-len(case["opts"]) * 5:]))


def _coverage(name, case, ref):
    """The edges each case is there for are really exercised (cell indices and live mask of the reference)."""
    n = case["N"] * case["S"]
    runs, live = ref["runs"]["hash_static"], ref["live"]
    wl = np.zeros(((n + 31) // 32) * 32, bool)
    wl[:n] = live
    wl = wl.reshape(-1, 32)
    if name == "lidar_256x768":
        assert (runs <= 16).any() and (runs > 16).any()
        mixed = wl.any(1) & ~wl.all(1)
        assert mixed.any(), "no warp with live and dead rows"
    if name == "lidar_axis_16_17":
        assert (runs == 16).any() and (runs == 17).any(), "no warp with exactly 16 and 17 runs"
    if name == "lidar_4099x1_t1":
        assert n % 32 != 0 and n % 256 != 0
    if name == "camera_37x37_tslice":
        assert n % 32 != 0 and (~live).any() and live.any()


def test_axis_rays_put_16_and_17_cells_in_a_warp():
    """Host-only: the axis-aligned rays give warps of exactly 16 and exactly 17 cells of static-hash level 2."""
    case = make_case("lidar_axis_16_17")
    cfg = FC.oracle_config()
    x, _, _, _ = geometry(case)
    lv = cfg.static_levels[2]
    cx = np.floor(EB.fma32(np.float32(lv["scale"]), x[:, 0], np.float32(0.5))).astype(np.int64)
    heads = EB.warp_heads(cx, np.ones(len(cx), bool))
    assert (heads == 16).any() and (heads == 17).any()


def test_leaving_rays_pile_onto_the_faces():
    """Host-only: the box-leaving rays clamp samples onto the +bound faces (normalised coordinate exactly 1.0)."""
    case = make_case("lidar_leave_box_t0")
    x, _, _, _ = geometry(case)
    assert ((x == 1.0).sum(0) > 100).all()


# ---- camera background -------------------------------------------------------------------------------------
RTOL = {"hash_static": 1e-2, "hash_dynamic": 1e-2, "planes": 1e-2, "flow_grid": 5e-2, "flow_mlp": 2e-2,
        "sigma_net": 1e-2, "intensity_net": 1e-2, "raydrop_net": 1e-2, "color_net": 1e-2}  # test_field_grad_gpu


@pytest.mark.gpu
@pytest.mark.parametrize("bg", ["0", "0.3", "tensor"])
def test_camera_background_forward_and_gradients(pkg, bg):
    """k_composite_bwd subtracts bg * sum(g_image) from the weights_sum gradient; a per-ray [N,3] background is
    blended outside the kernel (_split_bg).  Forward against FieldOracle.run(bg_color=...) at 1e-2, parameter
    gradients against the oracle's autograd at test_field_grad_gpu's tolerances."""
    import os
    from conftest import GOLDEN
    gold = np.load(os.path.join(GOLDEN, "field_grad_ref.npz"))
    case = FC.grad_case(gold, "c_mid")
    N = case["o"].shape[0]
    bgv = {"0": 0.0, "0.3": 0.3}.get(bg)
    bg_np = np.random.default_rng(9).random((N, 3), dtype=np.float32) if bg == "tensor" else None
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    m = pkg.NeRFNetwork(time_resolution=S.TIME_RESOLUTION, num_frames=S.NUM_FRAMES, bound=S.BOUND,
                        min_near=S.MIN_NEAR, min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH,
                        density_scale=case["ds"])
    m.load_flat_params(FC.oracle_params())
    m.train()
    out = m.render(dev(case["o"])[None], dev(case["d"])[None], torch.tensor([[case["t"]]], device="cuda"),
                   cal_lidar_color=False, staged=False, num_steps=case["coef"]["c"].shape[1],
                   noise=None if case["noise"] is None else dev(case["noise"]),
                   bg_color=dev(bg_np)[None] if bg_np is not None else bgv)
    std = dict(depth=out["depth"], image=out["image"], weights=out["weights"], weights_sum=out["weights_sum"])
    loss = FC.linear_loss(std, case["coef"], to=dev)
    loss.backward()
    e, eloss, eout = FC.oracle_grads(case, bg_color=torch.from_numpy(bg_np) if bg_np is not None else bgv)
    img = out["image"].detach().cpu().numpy().reshape(N, 3)
    eimg = eout["image"].detach().numpy()
    assert np.abs(img - eimg).max() <= 1e-2 * max(1.0, np.abs(eimg).max()), np.abs(img - eimg).max()
    assert abs(float(loss.detach()) - eloss) <= 1e-2 * max(abs(eloss), 1.0), (float(loss.detach()), eloss)
    floor = FC.oracle_grad_floor(case, "c_mid")
    for name in FC.GRAD_NAMES:
        p = getattr(m, f"{name}_camera" if name in ("hash_static", "hash_dynamic", "planes") else name)
        got = np.zeros(p.numel()) if p.grad is None else p.grad.detach().double().cpu().numpy().reshape(-1)
        ref = e[name].reshape(-1).astype(np.float64)
        if not ref.any():
            assert not got.any(), name
            continue
        err = np.linalg.norm(got - ref) / np.linalg.norm(ref)
        assert err < max(RTOL[name], 2.0 * floor[name]), (bg, name, err)
