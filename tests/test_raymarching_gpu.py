"""Parity of the sm_100a ray-marching operators (through the C ABI / Python operator module)
against (a) the CPU oracle and (b) the reference's own extension rebuilt for sm_100a: its stored
outputs (tests/golden/raymarching_ref_sm100a.npz) always, the live extension when oracle/_ref/ holds
a build of it (oracle/build_ref.sh).

Bar: bit-exact for sample ids/offsets/counts, positions, deltas, near/far, Morton codes and
bitfields; 1e-5 relative for compositing against the oracle (the oracle's exp2f is not the
GPU's ex2.approx), bit-exact against the reference extension."""
import os

import numpy as np
import pytest

import cases
from conftest import GOLDEN, assert_bits_equal

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

C, H = cases.S.CASCADE, cases.S.GRID_SIZE
BOUND = cases.S.BOUND


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def rel_close(a, b, rtol=1e-5, atol=1e-7, what=""):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    err = np.abs(a - b)
    tol = atol + rtol * np.maximum(np.abs(a), np.abs(b))
    assert (err <= tol).all(), f"{what}: max err {err.max():.3e} (rel {(err / (np.abs(b) + 1e-30)).max():.3e})"


# ------------------------------------------------------------------ near_far / sph
@pytest.mark.parametrize("n", [0, 1, 255, 256, 4096, 67980])
def test_near_far_from_aabb(pkg, oracle, ref_ext, n):
    rm = pkg.raymarching
    o, d = cases.S.camera_rays(n if n else 8, seed=3)
    o, d = o[:n], d[:n]
    if n >= 255:
        o = o.copy(); d = d.copy()
        o[::7] *= 9.0           # origins outside the box -> some misses
        d[5::11, 0] = 0.0       # axis-parallel rays (1/0 = inf)
        d[3::13] *= -1.0
    aabb = cases.S.AABB
    nears, fars = rm.near_far_from_aabb(dev(o).view(-1, 3), dev(d).view(-1, 3), dev(aabb), cases.S.MIN_NEAR)
    en, ef = oracle.near_far_from_aabb(o, d, aabb, cases.S.MIN_NEAR)
    assert_bits_equal(host(nears), en, "nears"); assert_bits_equal(host(fars), ef, "fars")
    if ref_ext is not None and n:
        rn, rf = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
        ref_ext.near_far_from_aabb(dev(o), dev(d), dev(aabb), n, cases.S.MIN_NEAR, rn, rf)
        assert_bits_equal(host(nears), host(rn), "nears vs ref"); assert_bits_equal(host(fars), host(rf), "fars vs ref")


def test_near_far_unaligned_and_cpu_inputs(pkg, oracle):
    rm = pkg.raymarching
    o, d = cases.S.camera_rays(1001, seed=4)
    big_o, big_d = dev(np.concatenate([o[:1], o])), dev(np.concatenate([d[:1], d]))
    nears, fars = rm.near_far_from_aabb(big_o[1:], big_d[1:], dev(cases.S.AABB), 0.05)  # 12-byte offset
    en, ef = oracle.near_far_from_aabb(o, d, cases.S.AABB, 0.05)
    assert_bits_equal(host(nears), en); assert_bits_equal(host(fars), ef)
    n2, f2 = rm.near_far_from_aabb(torch.from_numpy(o), torch.from_numpy(d), dev(cases.S.AABB), 0.05)  # CPU tensors
    assert n2.is_cuda and torch.equal(n2, nears) and torch.equal(f2, fars)


def test_sph_from_ray(pkg, oracle, ref_ext):
    rm = pkg.raymarching
    o, d = cases.S.camera_rays(5000, seed=5)
    got = host(rm.sph_from_ray(dev(o), dev(d), 3.0))
    exp = oracle.sph_from_ray(o, d, 3.0)
    assert got.shape == (5000, 2)
    np.testing.assert_allclose(got, exp, rtol=0, atol=2e-6)
    if ref_ext is not None:
        r = torch.empty(5000, 2, device="cuda")
        ref_ext.sph_from_ray(dev(o), dev(d), 3.0, 5000, r)
        np.testing.assert_allclose(got, host(r), rtol=0, atol=1e-6)


# ------------------------------------------------------------------ morton / packbits
def test_morton_roundtrip_and_oracle(pkg, oracle, ref_ext):
    rm = pkg.raymarching
    rng = np.random.default_rng(0)
    for hi, n in [(128, 100003), (1024, 4097)]:
        coords = rng.integers(0, hi, size=(n, 3)).astype(np.int32)
        idx = rm.morton3D(dev(coords))
        assert idx.dtype == torch.int32
        assert_bits_equal(host(idx), oracle.morton3D(coords), "morton3D")
        back = rm.morton3D_invert(idx)
        assert_bits_equal(host(back), coords, "roundtrip")
        assert_bits_equal(host(back), oracle.morton3D_invert(host(idx)), "invert")
    # out-of-range / negative values must still agree with the reference arithmetic
    wild = rng.integers(-2**31, 2**31 - 1, size=(1000, 3)).astype(np.int32)
    assert_bits_equal(host(rm.morton3D(dev(wild))), oracle.morton3D(wild), "morton3D wild")
    wi = rng.integers(-2**31, 2**31 - 1, size=1000).astype(np.int32)
    assert_bits_equal(host(rm.morton3D_invert(dev(wi))), oracle.morton3D_invert(wi), "invert wild")
    if ref_ext is not None:
        r = torch.empty(1000, dtype=torch.int32, device="cuda")
        ref_ext.morton3D(dev(wild), 1000, r)
        assert_bits_equal(host(rm.morton3D(dev(wild))), host(r))
    # all 128^3 cells: a permutation
    ax = np.arange(128, dtype=np.int32)
    full = np.stack(np.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)
    idx = host(rm.morton3D(dev(full)))
    assert np.array_equal(np.sort(idx), np.arange(128 ** 3))


@pytest.mark.parametrize("fill", ["full", "random5", "shell", "empty"])
def test_packbits_fills(pkg, oracle, ref_ext, fill):
    rm = pkg.raymarching
    g = cases.S.density_grid(fill, seed=1)
    got = rm.packbits(dev(g), cases.THRESH)
    assert got.dtype == torch.uint8 and got.shape == (C * H ** 3 // 8,)
    assert_bits_equal(host(got), cases.S.packbits_np(g, cases.THRESH), "vs numpy")
    assert_bits_equal(host(got), oracle.packbits(g, cases.THRESH), "vs oracle")
    if ref_ext is not None:
        r = torch.empty_like(got)
        ref_ext.packbits(dev(g), r.numel(), cases.THRESH, r)
        assert torch.equal(r, got)


def test_packbits_ragged_sizes_thresholds_and_preallocated(pkg):
    rm = pkg.raymarching
    rng = np.random.default_rng(7)
    for cells in [8, 64, 1016, 1024, 1032, 8 * 4099]:
        g = rng.normal(size=(1, cells)).astype(np.float32)
        g[0, ::5] = 0.25  # values equal to the threshold are NOT occupied (strict >)
        out = torch.full((cells // 8,), 0xAA, dtype=torch.uint8, device="cuda")
        ret = rm.packbits(dev(g), 0.25, out)
        assert ret.data_ptr() == out.data_ptr()
        assert_bits_equal(host(out), cases.S.packbits_np(g, 0.25), f"cells={cells}")
    # unaligned grid pointer (4-byte offset) takes the scalar path
    g = rng.normal(size=(1, 8 * 513 + 1)).astype(np.float32)
    gd = dev(g)[:, 1:]
    gd = torch.as_strided(dev(g).flatten()[1:], (1, 8 * 513), (8 * 513, 1))
    assert_bits_equal(host(rm.packbits(gd, 0.0)), cases.S.packbits_np(g[:, 1:], 0.0))


# ------------------------------------------------------------------ march_rays_train
def run_ref_march_train(ref_ext, o, d, bf, nears, fars, noises, dt_gamma, max_steps, M):
    N = o.shape[0]
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda")
    deltas = torch.zeros(M, 2, device="cuda")
    rays = torch.empty(N, 3, dtype=torch.int32, device="cuda")
    counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    ref_ext.march_rays_train(dev(o), dev(d), dev(bf), BOUND, dt_gamma, max_steps, N, C, H, M,
                             dev(nears), dev(fars), xyzs, dirs, deltas, rays, counter, dev(noises))
    torch.cuda.synchronize()
    return host(xyzs), host(dirs), host(deltas), host(rays), host(counter)


@pytest.mark.parametrize("fill", ["full", "random5", "shell", "empty"])
@pytest.mark.parametrize("kind,perturb,dt_gamma", [("lidar", False, cases.S.DT_GAMMA),
                                                   ("lidar", True, 0.0),
                                                   ("camera", True, cases.S.DT_GAMMA)])
def test_march_rays_train_bit_exact(pkg, oracle, ref_ext, fill, kind, perturb, dt_gamma):
    rm = pkg.raymarching
    N, max_steps = 4096, 1024
    o, d, nears, fars, noises = cases.march_inputs(kind, N, seed=11, perturb=perturb)
    bf = cases.bitfield(fill, seed=2)
    counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    xyzs, dirs, deltas, rays = rm.march_rays_train(
        dev(o), dev(d), BOUND, dev(bf), C, H, dev(nears), dev(fars), counter, -1, perturb, -1,
        True, dt_gamma, max_steps, dev(noises))
    ex, ed, el, er, ec = oracle.march_rays_train(o, d, BOUND, bf, C, H, nears, fars, noises,
                                                 dt_gamma=dt_gamma, max_steps=max_steps)
    m = int(ec[0])
    assert host(counter).tolist() == [m, N]
    assert xyzs.shape == (m, 3) and dirs.shape == (m, 3) and deltas.shape == (m, 2)
    assert_bits_equal(host(rays), er, "rays")
    assert_bits_equal(host(xyzs), ex[:m], "xyzs")
    assert_bits_equal(host(dirs), ed[:m], "dirs")
    assert_bits_equal(host(deltas), el[:m], "deltas")
    if fill == "empty":
        assert m == 0
    if ref_ext is not None:
        M = max(m, 1)
        rx, rd, rl, rr, rc = run_ref_march_train(ref_ext, o, d, bf, nears, fars, noises, dt_gamma, max_steps, M)
        assert rc.tolist() == [m, N]
        cr, (cx, cd, cl) = cases.canonical_from_rays(rr, [rx, rd, rl])
        assert_bits_equal(host(rays), cr, "rays vs reference (canonical order)")
        assert_bits_equal(host(xyzs), cx, "xyzs vs reference")
        assert_bits_equal(host(dirs), cd, "dirs vs reference")
        assert_bits_equal(host(deltas), cl, "deltas vs reference")


def test_march_rays_train_wrapper_semantics(pkg, oracle):
    """align padding, mean_count buffers with dropped rays, accumulated step_counter, perturb."""
    rm = pkg.raymarching
    N = 1000
    o, d, nears, fars, noises = cases.march_inputs("lidar", N, seed=12, perturb=True)
    bf = cases.bitfield("shell", seed=0)
    args = (dev(o), dev(d), BOUND, dev(bf), C, H, dev(nears), dev(fars))
    ex, ed, el, er, ec = oracle.march_rays_train(o, d, BOUND, bf, C, H, nears, fars, noises,
                                                 dt_gamma=cases.S.DT_GAMMA)
    m = int(ec[0])
    # align: a full `align` is added when already aligned (raymarching.py:278-279)
    for align in (128, 1, m if m > 0 else 7):
        x, dd, l, r = rm.march_rays_train(*args, None, -1, False, align, True, cases.S.DT_GAMMA, 1024, dev(noises))
        exp_m = m + (align - m % align)
        assert x.shape[0] == exp_m
        assert_bits_equal(host(x)[:m], ex[:m]); assert not host(x)[m:].any() and not host(l)[m:].any()
    # mean_count too small: trailing rays dropped, buffer size = padded mean_count
    mc = max(m // 2, 1)
    x, dd, l, r = rm.march_rays_train(*args, None, mc, False, 128, False, cases.S.DT_GAMMA, 1024, dev(noises))
    Mbuf = mc + (128 - mc % 128)
    assert x.shape[0] == Mbuf
    ox, od, ol, orr, oc = oracle.march_rays_train(o, d, BOUND, bf, C, H, nears, fars, noises,
                                                  dt_gamma=cases.S.DT_GAMMA, M=Mbuf)
    assert_bits_equal(host(r), orr); assert_bits_equal(host(x), ox); assert_bits_equal(host(l), ol)
    # accumulated counter: the second call's offsets start where the first ended
    counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    rm.march_rays_train(*args, counter, -1, False, -1, True, cases.S.DT_GAMMA, 1024, dev(noises))
    assert host(counter).tolist() == [m, N]
    counter[1] = 0
    x2, _, _, r2 = rm.march_rays_train(*args, counter, -1, False, -1, True, cases.S.DT_GAMMA, 1024, dev(noises))
    assert host(counter).tolist() == [2 * m, N]
    assert x2.shape[0] == 2 * m
    r2 = host(r2)
    assert np.array_equal(r2[:, 1], er[:, 1] + m) and np.array_equal(r2[:, 2], er[:, 2])
    assert_bits_equal(host(x2)[m:], ex[:m])
    # perturb=True draws noises internally: counts stay within one step of the unperturbed ones
    xp, _, _, rp = rm.march_rays_train(*args, None, -1, True, -1, True, cases.S.DT_GAMMA, 1024)
    assert rp.shape == (N, 3) and xp.shape[0] == int(host(rp)[:, 2].sum())


def test_march_rays_train_degenerate_rays(pkg, oracle):
    rm = pkg.raymarching
    o, d, nears, fars, noises = cases.march_inputs("camera", 300, seed=13, perturb=True)
    d = d.copy(); o = o.copy()
    d[::3, 1] = 0.0; d[1::5, 2] = -0.0; o[2::7] *= 4.0
    fars[4::9] = nears[4::9]            # empty interval
    nears[5::10] = np.float32(3.4e38); fars[5::10] = np.float32(3.4e38)   # "miss" rays from near_far
    bf = cases.bitfield("random5", seed=5)
    x, dd, l, r = rm.march_rays_train(dev(o), dev(d), BOUND, dev(bf), C, H, dev(nears), dev(fars),
                                      None, -1, False, -1, True, cases.S.DT_GAMMA, 64, dev(noises))
    ex, ed, el, er, ec = oracle.march_rays_train(o, d, BOUND, bf, C, H, nears, fars, noises,
                                                 dt_gamma=cases.S.DT_GAMMA, max_steps=64)
    m = int(ec[0])
    assert_bits_equal(host(r), er); assert_bits_equal(host(x), ex[:m]); assert_bits_equal(host(l), el[:m])
    assert er[:, 2].max() <= 64


# ------------------------------------------------------------------ composite_rays_train
def _march_for_composite(pkg, fill, N, seed):
    o, d, nears, fars, noises = cases.march_inputs("lidar", N, seed=seed, perturb=True)
    bf = cases.bitfield(fill, seed=3)
    x, dd, l, r = pkg.raymarching.march_rays_train(dev(o), dev(d), BOUND, dev(bf), C, H, dev(nears), dev(fars),
                                                   None, -1, False, -1, True, cases.S.DT_GAMMA, 1024, dev(noises))
    return l, r


@pytest.mark.parametrize("fill,T_thresh,scale", [("full", 1e-4, 1.0), ("shell", 1e-4, 30.0),
                                                 ("random5", 1e-2, 200.0), ("full", 0.5, 50.0)])
def test_composite_rays_train_forward_backward(pkg, oracle, ref_ext, fill, T_thresh, scale):
    rm = pkg.raymarching
    N = 4096
    deltas, rays = _march_for_composite(pkg, fill, N, seed=21)
    M = deltas.shape[0]
    sig, rgb = cases.field_values(M, seed=1)
    sig = sig * np.float32(scale)
    rng = np.random.default_rng(5)
    # shuffle the rows like the reference's atomics would, add an empty and an overflowing ray
    rays_h = host(rays).copy()
    rays_h = rays_h[rng.permutation(N)]
    rays_h[0, 2] = 0
    rays_h[1, 1] = M - 1; rays_h[1, 2] = 5
    sig_t = dev(sig).requires_grad_(True); rgb_t = dev(rgb).requires_grad_(True)
    ws, depth, image = rm.composite_rays_train(sig_t, rgb_t, deltas, dev(rays_h), T_thresh)
    ews, edepth, eimage = oracle.composite_rays_train_forward(sig, rgb, host(deltas), rays_h, T_thresh)
    rel_close(host(ws), ews, what="weights_sum"); rel_close(host(depth), edepth, what="depth")
    rel_close(host(image), eimage, what="image")
    assert host(ws)[rays_h[0, 0]] == 0 and host(ws)[rays_h[1, 0]] == 0
    g_ws = rng.normal(size=N).astype(np.float32); g_img = rng.normal(size=(N, 3)).astype(np.float32)
    (ws * dev(g_ws)).sum().add((image * dev(g_img)).sum()).add(depth.sum()).backward()
    egs, egr = oracle.composite_rays_train_backward(g_ws, g_img, sig, rgb, host(deltas), rays_h,
                                                    host(ws), host(image), T_thresh)
    # per-sample gradients carry alpha = 1 - exp(-sigma*delta) un-summed: for tiny sigma*delta the
    # oracle's exp2f and the GPU's ex2.approx differ by ~2^-22 ABSOLUTE in alpha, so the bound is
    # absolute here (the reference-extension comparison below is bit-exact).
    rel_close(host(sig_t.grad), egs, rtol=2e-5, atol=2e-5, what="grad_sigmas")
    rel_close(host(rgb_t.grad), egr, rtol=1e-5, atol=5e-6, what="grad_rgbs")
    if ref_ext is not None:
        rws = torch.empty(N, device="cuda"); rde = torch.empty(N, device="cuda"); rim = torch.empty(N, 3, device="cuda")
        ref_ext.composite_rays_train_forward(dev(sig), dev(rgb), deltas, dev(rays_h), M, N, T_thresh, rws, rde, rim)
        assert_bits_equal(host(ws), host(rws), "weights_sum vs reference")
        assert_bits_equal(host(depth), host(rde), "depth vs reference")
        assert_bits_equal(host(image), host(rim), "image vs reference")
        rgs = torch.zeros(M, device="cuda"); rgr = torch.zeros(M, 3, device="cuda")
        ref_ext.composite_rays_train_backward(dev(g_ws), dev(g_img), dev(sig), dev(rgb), deltas, dev(rays_h),
                                              rws, rim, M, N, T_thresh, rgs, rgr)
        assert_bits_equal(host(sig_t.grad), host(rgs), "grad_sigmas vs reference")
        assert_bits_equal(host(rgb_t.grad), host(rgr), "grad_rgbs vs reference")


def test_composite_rays_train_properties_full_frame(pkg):
    """Size-independent properties at the full LiDAR frame (67 980 rays)."""
    rm = pkg.raymarching
    deltas, rays = _march_for_composite(pkg, "shell", -1, seed=22)
    N, M = rays.shape[0], deltas.shape[0]
    assert N == 67980
    r = host(rays)
    assert np.array_equal(r[:, 0], np.arange(N)) and r[:, 2].sum() == M
    assert np.array_equal(r[:, 1], np.concatenate([[0], np.cumsum(r[:, 2])[:-1]]))
    sig, rgb = cases.field_values(M, seed=2)
    sig *= 40
    ws, depth, image = rm.composite_rays_train(dev(sig), dev(rgb), deltas, rays)
    w = host(ws)
    assert (w >= 0).all() and (w <= 1 + 1e-5).all()
    assert not w[r[:, 2] == 0].any()
    # zero density -> nothing accumulates; linear in rgbs
    z = rm.composite_rays_train(torch.zeros(M, device="cuda"), dev(rgb), deltas, rays)
    assert not host(z[0]).any() and not host(z[2]).any()
    rgb2 = np.random.default_rng(3).random((M, 3), dtype=np.float32)
    i1 = host(image); i2 = host(rm.composite_rays_train(dev(sig), dev(rgb2), deltas, rays)[2])
    i3 = host(rm.composite_rays_train(dev(sig), dev(0.25 * rgb + 0.5 * rgb2), deltas, rays)[2])
    np.testing.assert_allclose(i3, 0.25 * i1 + 0.5 * i2, rtol=1e-4, atol=1e-6)
    # constant colour c -> image == c * weights_sum
    ic = host(rm.composite_rays_train(dev(sig), torch.full((M, 3), 0.5, device="cuda"), deltas, rays)[2])
    np.testing.assert_allclose(ic, 0.5 * w[:, None].repeat(3, 1), rtol=1e-5, atol=1e-7)


# ------------------------------------------------------------------ inference pair
@pytest.mark.parametrize("fill,n_step_cap", [("shell", 8), ("full", 40), ("random5", 1)])
def test_inference_loop_matches_oracle(pkg, oracle, ref_ext, fill, n_step_cap):
    """torch-ngp style run_cuda loop: march_rays -> field -> composite_rays -> compaction."""
    rm = pkg.raymarching
    N = 3000
    o, d, nears, fars, _ = cases.march_inputs("lidar", N, seed=31, perturb=False)
    bf = cases.bitfield(fill, seed=4)
    rng = np.random.default_rng(9)

    def field(x):  # deterministic pseudo-field of position
        s = (np.abs(np.sin(x * 37.0)).sum(1) * 20).astype(np.float32)
        c = np.abs(np.cos(x * 11.0)).astype(np.float32)
        return s, c

    t_o, t_d, t_bf, t_n, t_f = dev(o), dev(d), dev(bf), dev(nears), dev(fars)
    g = dict(ws=torch.zeros(N, device="cuda"), depth=torch.zeros(N, device="cuda"), image=torch.zeros(N, 3, device="cuda"))
    e = dict(ws=np.zeros(N, np.float32), depth=np.zeros(N, np.float32), image=np.zeros((N, 3), np.float32))
    r = None
    if ref_ext is not None:
        r = dict(ws=torch.zeros(N, device="cuda"), depth=torch.zeros(N, device="cuda"), image=torch.zeros(N, 3, device="cuda"),
                 t=t_n.clone(), alive=torch.arange(N, dtype=torch.int32, device="cuda"))
    g_alive = torch.arange(N, dtype=torch.int32, device="cuda"); g_t = t_n.clone()
    e_alive = np.arange(N, dtype=np.int32); e_t = nears.copy()
    it = 0
    while len(e_alive) > 0 and it < 200:
        n_alive = len(e_alive)
        n_step = max(min(N // n_alive, n_step_cap), 1)
        noises = rng.random(n_alive, dtype=np.float32)
        gx, gd, gl = rm.march_rays(n_alive, n_step, g_alive, g_t, t_o, t_d, BOUND, t_bf, C, H, t_n, t_f,
                                   128, True, cases.S.DT_GAMMA, 1024, dev(noises))
        M = gx.shape[0]
        assert M == n_alive * n_step + (128 - (n_alive * n_step) % 128)
        ex, ed, el = oracle.march_rays(n_alive, n_step, e_alive, e_t, o, d, BOUND, bf, C, H, nears, fars, noises,
                                       dt_gamma=cases.S.DT_GAMMA, M=M)
        assert_bits_equal(host(gx), ex, f"xyzs it={it}"); assert_bits_equal(host(gd), ed, "dirs")
        assert_bits_equal(host(gl), el, f"deltas it={it}")
        s, c = field(ex)
        rm.composite_rays(n_alive, n_step, g_alive, g_t, dev(s), dev(c), gl, g["ws"], g["depth"], g["image"], 1e-2)
        e_alive, e_t, e["ws"], e["depth"], e["image"] = oracle.composite_rays(
            n_alive, n_step, e_alive, e_t, s, c, el, e["ws"], e["depth"], e["image"], 1e-2)
        if r is not None:
            rx = torch.zeros(M, 3, device="cuda"); rd = torch.zeros(M, 3, device="cuda"); rl = torch.zeros(M, 2, device="cuda")
            ref_ext.march_rays(n_alive, n_step, r["alive"], r["t"], t_o, t_d, BOUND, cases.S.DT_GAMMA, 1024, C, H,
                               t_bf, t_n, t_f, rx, rd, rl, dev(noises))
            assert_bits_equal(host(gx), host(rx), "xyzs vs reference"); assert_bits_equal(host(gl), host(rl), "deltas vs reference")
            ref_ext.composite_rays(n_alive, n_step, 1e-2, r["alive"], r["t"], dev(s), dev(c), rl, r["ws"], r["depth"], r["image"])
            assert torch.equal(r["alive"][:n_alive], g_alive[:n_alive])
            assert_bits_equal(host(g["ws"]), host(r["ws"]), "ws vs reference")
            assert_bits_equal(host(g["depth"]), host(r["depth"]), "depth vs reference")
            assert_bits_equal(host(g["image"]), host(r["image"]), "image vs reference")
            assert_bits_equal(host(g_t), host(r["t"]), "rays_t vs reference")
            r["alive"] = r["alive"][:n_alive][r["alive"][:n_alive] >= 0].contiguous()
        assert np.array_equal(host(g_alive)[:n_alive], e_alive), f"alive flags it={it}"
        rel_close(host(g["ws"]), e["ws"], what="ws"); rel_close(host(g["depth"]), e["depth"], what="depth")
        rel_close(host(g["image"]), e["image"], what="image")
        # adopt the GPU state on the CPU side so rounding differences of exp cannot drift
        e_t = host(g_t).copy(); e["ws"] = host(g["ws"]).copy(); e["depth"] = host(g["depth"]).copy(); e["image"] = host(g["image"]).copy()
        g_alive = g_alive[:n_alive][g_alive[:n_alive] >= 0].contiguous()
        e_alive = e_alive[e_alive >= 0]
        it += 1
    assert len(e_alive) == 0 or it == 200
    assert host(g["ws"]).max() <= 1 + 1e-5


def test_errors_are_loud(pkg):
    L = pkg._lib.lib()
    st = L.nvsf_near_far_from_aabb(None, None, None, 5, 0.1, None, None, None)
    assert st == -1
    with pytest.raises(pkg._lib.NvsfError):
        pkg._lib.check(st, "near_far")
    # Morton grid larger than 10 bits per axis is rejected
    z = torch.zeros(8, device="cuda")
    st = L.nvsf_march_rays_train_count(z.data_ptr(), z.data_ptr(), z.data_ptr(), 1.0, 0.0, 16, 1, 1, 2048,
                                       z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(),
                                       z.data_ptr(), 32, None)
    assert st == -1
    st = L.nvsf_march_rays_train_count(z.data_ptr(), z.data_ptr(), z.data_ptr(), 1.0, 0.0, 16, 1, 1, 128,
                                       z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(),
                                       z.data_ptr(), 4, None)
    assert st == -2


# ------------------------------------------------------------------ stored outputs of the reference extension
@pytest.fixture(scope="module")
def gold():
    """Inputs and outputs of the reference's own extension (raymarching.cu built for sm_100a, run on a B200 by
    oracle/make_golden_raymarching.py): the comparison with the reference that needs nothing outside the tree."""
    return np.load(os.path.join(GOLDEN, "raymarching_ref_sm100a.npz"))


def test_operators_match_reference_golden(pkg, gold):
    rm = pkg.raymarching
    g = gold
    nears, fars = rm.near_far_from_aabb(dev(g["nf_o"]), dev(g["nf_d"]), dev(cases.S.AABB), cases.S.MIN_NEAR)
    assert_bits_equal(host(nears), g["nf_nears"], "nears"); assert_bits_equal(host(fars), g["nf_fars"], "fars")
    np.testing.assert_allclose(host(rm.sph_from_ray(dev(g["sph_o"]), dev(g["sph_d"]), 3.0)), g["sph_coords"],
                               rtol=0, atol=1e-6)
    assert_bits_equal(host(rm.morton3D(dev(g["mt_coords"]))), g["mt_indices"], "morton3D")
    assert_bits_equal(host(rm.morton3D_invert(dev(g["mt_indices"]))), g["mt_back"], "morton3D_invert")
    assert_bits_equal(host(rm.packbits(dev(g["pb_grid"]), 0.25)), g["pb_bits"], "packbits")


@pytest.mark.parametrize("ci", [0, 1, 2, 3])
def test_march_and_composite_train_match_reference_golden(pkg, gold, ci):
    rm = pkg.raymarching
    p = f"mt{ci}_"
    _, N, max_steps, perturb, m = gold[p + "meta"].tolist()
    bf = cases.bitfield(str(gold[p + "fill"]), seed=6)
    counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    xyzs, dirs, deltas, rays = rm.march_rays_train(
        dev(gold[p + "o"]), dev(gold[p + "d"]), BOUND, dev(bf), C, H, dev(gold[p + "nears"]), dev(gold[p + "fars"]),
        counter, -1, bool(perturb), -1, True, float(gold[p + "dt_gamma"]), max_steps, dev(gold[p + "noises"]))
    assert host(counter).tolist() == [m, N]
    assert_bits_equal(host(rays), gold[p + "rays"], "rays (canonical order)")
    assert_bits_equal(host(xyzs), gold[p + "xyzs"], "xyzs"); assert_bits_equal(host(deltas), gold[p + "deltas"], "deltas")
    sig, rgb = cases.field_values(m, seed=int(gold[p + "sig_seed"])); sig *= np.float32(30.0)
    sig_t = dev(sig).requires_grad_(True); rgb_t = dev(rgb).requires_grad_(True)
    ws, depth, image = rm.composite_rays_train(sig_t, rgb_t, deltas, rays, 1e-4)
    assert_bits_equal(host(ws), gold[p + "ws"], "weights_sum"); assert_bits_equal(host(depth), gold[p + "depth"], "depth")
    assert_bits_equal(host(image), gold[p + "image"], "image")
    ((ws * dev(gold[p + "g_ws"])).sum() + (image * dev(gold[p + "g_im"])).sum()).backward()
    assert_bits_equal(host(sig_t.grad), gold[p + "grad_sigmas"], "grad_sigmas")
    assert_bits_equal(host(rgb_t.grad), gold[p + "grad_rgbs"], "grad_rgbs")


def test_inference_step_matches_reference_golden(pkg, gold):
    rm = pkg.raymarching
    g = gold
    n_alive, n_step = g["inf_meta"].tolist()
    bf = cases.bitfield("shell", seed=6)
    x, d, l = rm.march_rays(n_alive, n_step, dev(g["inf_alive"]), dev(g["inf_rays_t"]), dev(g["inf_o"]), dev(g["inf_d"]),
                            BOUND, dev(bf), C, H, dev(g["inf_nears"]), dev(g["inf_fars"]), -1, True, cases.S.DT_GAMMA,
                            1024, dev(g["inf_noises"]))
    assert_bits_equal(host(x), g["inf_xyzs"], "xyzs"); assert_bits_equal(host(d), g["inf_dirs"], "dirs")
    assert_bits_equal(host(l), g["inf_deltas"], "deltas")
    sig, rgb = cases.field_values(n_alive * n_step, seed=71); sig *= np.float32(60.0)
    alive, rays_t = dev(g["inf_alive"]), dev(g["inf_rays_t"])
    ws, depth, image = dev(g["inf_ws0"]), dev(g["inf_de0"]), dev(g["inf_im0"])
    rm.composite_rays(n_alive, n_step, alive, rays_t, dev(sig), dev(rgb), l, ws, depth, image, 1e-2)
    assert np.array_equal(host(alive), g["inf_alive_out"])
    assert_bits_equal(host(rays_t), g["inf_t_out"], "rays_t"); assert_bits_equal(host(ws), g["inf_ws"], "weights_sum")
    assert_bits_equal(host(depth), g["inf_depth"], "depth"); assert_bits_equal(host(image), g["inf_image"], "image")
