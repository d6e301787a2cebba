"""Marching cubes on the device (csrc/mesh.cu) bit for bit against the numpy oracle, and
NeRFNetwork.extract_geometry against the field's own density on the reference's lattice."""
import importlib

import numpy as np
import pytest
import torch

from conftest import assert_bits_equal
from oracle import mesh_oracle as M

gpu = pytest.mark.gpu
TAU = 0.5


def _pkg():
    return importlib.import_module("selfsupervised-nvsf_b200")


def _smooth(shape, rng):
    """A random smooth field (a few random plane waves) plus a little noise: a surface of moderate size."""
    idx = np.meshgrid(*[np.arange(s, dtype=np.float64) for s in shape], indexing="ij")
    u = np.zeros(shape)
    for _ in range(6):
        k = rng.normal(size=3) * 0.08
        u += np.cos(k[0] * idx[0] + k[1] * idx[1] + k[2] * idx[2] + rng.uniform(0, 2 * np.pi))
    return (u / 6 + 0.5 + 0.02 * rng.random(shape)).astype(np.float32)


def _volume(kind, shape, seed):
    rng = np.random.default_rng(seed)
    # uniform noise puts a surface in nearly every cell; at 257^3 that is ~5e7 triangles for the oracle, so the
    # large shape uses the smooth field (it still spans every CTA and scan chunk)
    base = rng.random(shape, dtype=np.float32) if np.prod(shape) <= 64 ** 3 else _smooth(shape, rng)
    if kind == "random":
        return base
    if kind == "exact":            # values exactly at the threshold are not above
        return np.round(base * 4).astype(np.float32) / np.float32(4)
    if kind == "nonfinite":
        pick = rng.random(shape)
        u = base.copy()
        u[pick < 0.05] = np.nan
        u[(pick >= 0.05) & (pick < 0.1)] = np.inf
        u[(pick >= 0.1) & (pick < 0.15)] = -np.inf
        return u
    if kind == "all_above":
        return np.full(shape, 1.0, np.float32)
    assert kind == "all_below"
    return np.full(shape, TAU, np.float32)


SHAPES = [(2, 2, 2), (37, 53, 29), (64, 64, 64), (257, 257, 257)]
KINDS = ["random", "exact", "nonfinite", "all_above", "all_below"]


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("kind", KINDS)
def test_marching_cubes_matches_oracle(shape, kind):
    mesh = _pkg().mesh
    u = _volume(kind, shape, seed=10 * SHAPES.index(shape) + KINDS.index(kind))
    ev, et = M.marching_cubes(u, TAU)
    uu = torch.from_numpy(u).cuda()
    v, t = mesh.marching_cubes(uu, TAU)
    assert v.shape == ev.shape and t.shape == et.shape, (v.shape, ev.shape, t.shape, et.shape)
    assert v.dtype == torch.float32 and t.dtype == torch.int64 and v.is_cuda and t.is_cuda
    assert_bits_equal(v.cpu().numpy(), ev, f"{kind} {shape} vertices")
    assert_bits_equal(t.cpu().numpy(), et, f"{kind} {shape} triangles")
    if kind in ("all_above", "all_below"):
        assert len(ev) == 0 and len(et) == 0
    elif shape != (2, 2, 2):
        assert len(et) > 0
    v2, t2 = mesh.marching_cubes(uu, TAU)          # no atomics: a second run is bit-identical
    assert torch.equal(v2.view(torch.int32), v.view(torch.int32)) and torch.equal(t2, t)


@gpu
def test_every_case_of_the_table():
    """Each of the 256 corner cases once, as separate 2x2x2 cells inside one volume."""
    mesh = _pkg().mesh
    cases = np.arange(256)
    u = np.zeros((2 * 256, 2, 2), np.float32)
    for c in range(8):
        dx, dy, dz = c & 1, (c >> 1) & 1, (c >> 2) & 1
        u[2 * cases + dx, dy, dz] = ((cases >> c) & 1).astype(np.float32) + np.float32(0.25) * c / 8
    ev, et = M.marching_cubes(u, TAU)
    v, t = mesh.marching_cubes(torch.from_numpy(u).cuda(), TAU)
    assert_bits_equal(v.cpu().numpy(), ev, "vertices")
    assert_bits_equal(t.cpu().numpy(), et, "triangles")


@gpu
def test_inputs_and_errors():
    pkg = _pkg()
    mesh = pkg.mesh
    u = _volume("random", (9, 10, 11), 5)
    ev, et = M.marching_cubes(u, TAU)
    # a non-contiguous fp64 view is converted
    d = torch.from_numpy(u.astype(np.float64)).cuda().permute(2, 1, 0).contiguous().permute(2, 1, 0)
    v, t = mesh.marching_cubes(d, TAU)
    assert_bits_equal(v.cpu().numpy(), ev, "vertices")
    assert np.array_equal(t.cpu().numpy(), et)
    for bad in (torch.zeros(1, 4, 4, device="cuda"), torch.zeros(4, 4, device="cuda"),
                torch.zeros(4, 4, 1025, device="cuda"), torch.zeros(4, 4, 4)):
        with pytest.raises(pkg._lib.NvsfError):
            mesh.marching_cubes(bad, 0.0)


def _closed_oriented_torch(t):
    """The directed edges are distinct and each one's reverse is present (on the device)."""
    if t.numel() == 0:
        return True
    n = int(t.max()) + 1
    e = torch.cat([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])
    fwd = torch.sort(e[:, 0] * n + e[:, 1]).values
    if (fwd[1:] == fwd[:-1]).any():
        return False
    rev = e[:, 1] * n + e[:, 0]
    pos = torch.searchsorted(fwd, rev).clamp_max(fwd.numel() - 1)
    return bool((fwd[pos] == rev).all())


@gpu
def test_full_size_volume():
    """1024^3: the 4 GiB workspace and the two-level 64-bit offsets at full size (closed, oriented, counts)."""
    mesh = _pkg().mesh
    n = 1024
    g = torch.arange(n, device="cuda", dtype=torch.float32) - 511.3
    u = torch.empty(n, n, n, device="cuda")
    for i in range(0, n, 128):   # a sphere with ripples, built in slabs
        x = g[i:i + 128, None, None]
        r = torch.sqrt(x * x + g[None, :, None] ** 2 + g[None, None, :] ** 2)
        u[i:i + 128] = 400.0 - r + 6.0 * torch.sin(g[None, :, None] * 0.05) * torch.cos(g[None, None, :] * 0.07)
    v, t = mesh.marching_cubes(u, 0.0)
    A = u > 0
    V = int((A[1:] != A[:-1]).sum() + (A[:, 1:] != A[:, :-1]).sum() + (A[:, :, 1:] != A[:, :, :-1]).sum())
    count = torch.from_numpy(M.TRI_COUNT.astype(np.int64)).cuda()
    T = 0
    for i in range(0, n - 1, 64):
        a = A[i:min(i + 65, n)].to(torch.int64)
        m = a.shape[0] - 1
        cube = torch.zeros(m, n - 1, n - 1, dtype=torch.int64, device="cuda")
        for c in range(8):
            dx, dy, dz = c & 1, (c >> 1) & 1, (c >> 2) & 1
            cube |= a[dx:dx + m, dy:dy + n - 1, dz:dz + n - 1] << c
        T += int(count[cube].sum())
    del A
    assert v.shape == (V, 3) and t.shape == (T, 3) and T > 10 ** 6
    assert int(t.min()) == 0 and int(t.max()) == V - 1
    assert _closed_oriented_torch(t)
    assert bool(torch.isfinite(v).all()) and float(v.min()) >= 0 and float(v.max()) <= n - 1


@gpu
def test_extract_geometry_matches_density_and_oracle():
    import field_cases as FC
    pkg = _pkg()
    S = FC.S
    kw = dict(bound=S.BOUND, num_frames=S.NUM_FRAMES, time_resolution=S.TIME_RESOLUTION, min_near=S.MIN_NEAR,
              min_near_lidar=S.MIN_NEAR_LIDAR, lidar_max_depth=S.LIDAR_MAX_DEPTH)
    model = pkg.NeRFNetwork(**kw).eval()
    model.load_flat_params(FC.oracle_params(style="trained"))
    R, t = 128, 0.4
    b = model.aabb_infer.detach().float().cpu()
    axes = [torch.linspace(b[a], b[3 + a], R) for a in range(3)]
    pts = torch.stack(torch.meshgrid(*axes, indexing="ij"), -1).view(-1, 3).cuda()
    with torch.no_grad():
        vol = model.density(pts, t, cal_lidar_color=True)["sigma"].view(R, R, R)
    got, _ = model._density_volume(t, R, True)              # the slabbed volume extract_geometry meshes
    assert torch.equal(got.view(torch.int32), vol.view(torch.int32))
    tau = float(vol.float().median())       # a threshold with a surface, whatever the scale of sigma
    ev, et = M.marching_cubes(vol.cpu().numpy(), tau)
    assert len(et) > 1000
    v, f = model.extract_geometry(t, resolution=R, threshold=tau, cal_lidar_color=True)
    assert np.array_equal(f.cpu().numpy(), et)
    lo, hi = b[:3].cuda(), b[3:].cuda()
    want = torch.from_numpy(ev).cuda() / float(R - 1) * (hi - lo) + lo
    assert_bits_equal(v.cpu().numpy(), want.cpu().numpy(), "world vertices")
    # the transform is torch-ngp's v / (R - 1) * (b_max - b_min) + b_min
    ref = ev.astype(np.float64) / (R - 1) * (b[3:] - b[:3]).double().numpy() + b[:3].double().numpy()
    assert np.abs(v.cpu().numpy() - ref).max() <= 1e-6 * max(1.0, float(np.abs(ref).max()))
    # a time given as the reference's [1, 1] CUDA tensor gives the same mesh
    v2, f2 = model.extract_geometry(torch.tensor([[t]], device="cuda"), resolution=R, threshold=tau,
                                    cal_lidar_color=True)
    assert torch.equal(f2, f) and torch.equal(v2.view(torch.int32), v.view(torch.int32))


@gpu
def test_write_respects_the_caps():
    """_write stores only the rows below v_cap / t_cap; the leading rows are the full result's and the rest of the
    buffers keeps its sentinel."""
    pkg = _pkg()
    L, ptr = pkg._lib.lib(), pkg._lib.ptr
    u = _volume("random", (37, 53, 29), 7)
    ev, et = M.marching_cubes(u, TAU)
    uu = torch.from_numpy(u).cuda()
    X, Y, Z = u.shape
    wb = L.nvsf_marching_cubes_workspace_bytes(X, Y, Z)
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
    counts = torch.empty(2, dtype=torch.int64, device="cuda")
    assert L.nvsf_marching_cubes_count(ptr(uu), X, Y, Z, TAU, ptr(counts), ptr(ws), wb, None) == 0
    assert counts.tolist() == [len(ev), len(et)]
    for vc, tc in ((len(ev) // 3, len(et) // 2), (0, 5), (7, 0), (len(ev), len(et) - 1)):
        v = torch.full((len(ev), 3), -7.0, device="cuda")
        t = torch.full((len(et), 3), -7, dtype=torch.int64, device="cuda")
        assert L.nvsf_marching_cubes_write(ptr(uu), X, Y, Z, TAU, ptr(v), vc, ptr(t), tc, ptr(ws), wb, None) == 0
        v, t = v.cpu().numpy(), t.cpu().numpy()
        assert_bits_equal(v[:vc], ev[:vc], f"vertices below cap {vc}")
        assert np.array_equal(t[:tc], et[:tc]), tc
        assert (v[vc:] == -7.0).all() and (t[tc:] == -7).all(), (vc, tc)
