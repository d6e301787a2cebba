"""Mesh extraction on the CPU side: the generated marching-cubes table (it matches its generator and has the
properties the surface relies on), the numpy oracle on analytic and random volumes, write_ply, and the C ABI's
argument checks (they fire before any launch, so they run without a device)."""
import ctypes
import importlib
import struct

import numpy as np
import pytest
import torch

from oracle import make_mc_tables as G
from oracle import mesh_oracle as M


def _pkg():
    p = importlib.import_module("selfsupervised-nvsf_b200")
    importlib.import_module("selfsupervised-nvsf_b200.build").build()
    return p


# ------------------------------------------------------------------------------------------------- the table
def test_generated_header_is_committed():
    with open(G.HEADER) as f:
        assert f.read() == G.render(), "csrc/mc_tables.cuh differs from oracle/make_mc_tables.py's output"


def _crossing(case):
    return [e for e in range(12)
            if (case >> G.EDGES[e][0]) & 1 != (case >> (G.EDGES[e][0] | 1 << G.EDGES[e][1])) & 1]


def test_table_invariants():
    count, tris, mx = G.tables()
    assert count[0] == 0 and count[255] == 0 and mx == tris.shape[1]
    for case in range(256):
        loops = G.case_loops(case)
        flat = [e for lp in loops for e in lp]
        assert sorted(flat) == _crossing(case), case                     # every crossing edge in exactly one loop
        assert count[case] == sum(len(lp) - 2 for lp in loops), case
        used = tris[case, :count[case]]
        assert (tris[case, count[case]:] == -1).all()
        for lp in loops:                                                 # each loop's triangles use its own edges
            assert sum(set(t.tolist()) <= set(lp) for t in used) == len(lp) - 2
        # complementing the case keeps the crossing edges (the surface of the other side)
        assert _crossing(255 - case) == _crossing(case)


def test_ambiguous_face_rule_depends_on_the_face_only():
    """On a face with four crossing edges each above corner is cut off by its own segment; the choice is a
    function of the face's corners, so the two cells sharing the face agree."""
    seen = 0
    for case in range(256):
        above = [(case >> c) & 1 for c in range(8)]
        for axis, side, corners, edges in G.FACES:
            ce = [e for e in edges if e in _crossing(case)]
            if len(ce) != 4:
                continue
            seen += 1
            loops = G.case_loops(case)
            nxt = {lp[i]: lp[(i + 1) % len(lp)] for lp in loops for i in range(len(lp))}
            segs = {frozenset((a, b)) for a, b in nxt.items() if a in edges and b in edges}
            want = {frozenset(e for e in edges if c in (G.EDGES[e][0], G.EDGES[e][0] | 1 << G.EDGES[e][1]))
                    for c in corners if above[c]}
            assert segs == want, (case, axis, side)
    assert seen > 0


# ------------------------------------------------------------------------------------------------ the oracle
def _grid(n, c):
    g = np.arange(n, dtype=np.float64) - c
    return np.meshgrid(g, g, g, indexing="ij")


def _normals(v, t):
    a, b, c = v[t[:, 0]].astype(np.float64), v[t[:, 1]].astype(np.float64), v[t[:, 2]].astype(np.float64)
    return np.cross(b - a, c - a), (a + b + c) / 3.0


def test_sphere():
    n, r0, c = 48, 16.0, 23.3
    x, y, z = _grid(n, c)
    u = (r0 - np.sqrt(x * x + y * y + z * z)).astype(np.float32)
    v, t = M.marching_cubes(u, 0.0)
    assert len(t) > 1000 and M.is_closed_oriented(t)
    assert M.euler_characteristic(len(v), t) == 2
    r = np.linalg.norm(v.astype(np.float64) - c, axis=1)
    # linear interpolation of u = r0 - |x| along a unit edge errs by at most max|u''| / 8 <= 1 / (8 (r0 - 1))
    assert np.abs(r - r0).max() <= 1.0 / (8.0 * (r0 - 1.0)) + 1e-5
    nrm, cen = _normals(v, t)
    area = np.linalg.norm(nrm, axis=1)
    big = area > 1e-3
    assert big.mean() > 0.9
    assert (np.einsum("ij,ij->i", nrm[big], cen[big] - c) > 0).all()    # along -grad u: out of the inside


def test_torus():
    n, R, r = 56, 16.0, 6.0
    x, y, z = _grid(n, 27.6)
    u = (r - np.sqrt((np.sqrt(x * x + y * y) - R) ** 2 + z * z)).astype(np.float32)
    v, t = M.marching_cubes(u, 0.0)
    assert M.is_closed_oriented(t)
    assert M.euler_characteristic(len(v), t) == 0


def _bordered(u, value=-1.0):
    u[0] = u[-1] = value
    u[:, 0] = u[:, -1] = value
    u[:, :, 0] = u[:, :, -1] = value
    return u


@pytest.mark.parametrize("kind", ["uniform", "binary", "exact"])
def test_random_volumes_are_closed_and_oriented(kind):
    rng = np.random.default_rng({"uniform": 0, "binary": 1, "exact": 2}[kind])
    for s in range(6):
        shape = tuple(rng.integers(3, 14, size=3))
        if kind == "uniform":
            u = rng.random(shape, dtype=np.float32)
        elif kind == "binary":       # many ambiguous faces
            u = rng.integers(0, 2, size=shape).astype(np.float32)
        else:                        # values exactly at the threshold are not above
            u = rng.integers(0, 3, size=shape).astype(np.float32) * np.float32(0.5)
        v, t = M.marching_cubes(_bordered(u), 0.5)
        assert M.is_closed_oriented(t), (kind, s, shape)
        assert len(t) == 0 or t.max() < len(v)
        # every vertex is used and lies on its lattice edge
        assert len(t) == 0 or np.unique(t).size == len(v)
        frac = v - np.floor(v)
        assert ((frac != 0).sum(1) <= 1).all()


def test_nonfinite_values_give_finite_vertices():
    rng = np.random.default_rng(3)
    u = rng.normal(size=(17, 13, 11)).astype(np.float32)
    pick = rng.random(u.shape)
    u[pick < 0.08] = np.nan
    u[(pick >= 0.08) & (pick < 0.16)] = np.inf
    u[(pick >= 0.16) & (pick < 0.24)] = -np.inf
    v, t = M.marching_cubes(_bordered(u, -np.inf), 0.0)
    assert len(v) > 0 and np.isfinite(v).all()
    assert M.is_closed_oriented(t)
    # a NaN corner is below: an edge from NaN to an above corner lands on the NaN end (t = 0 from a NaN t)
    assert M.edge_bits(np.array([[[np.nan]], [[1.0]]], np.float32), 0.0)[0][0, 0, 0, 0]


def test_empty_volumes():
    for val in (-1.0, 1.0):
        v, t = M.marching_cubes(np.full((5, 4, 3), val, np.float32), 0.0)
        assert v.shape == (0, 3) and t.shape == (0, 3)


# ------------------------------------------------------------------------------------------------------ PLY
def _read_ply(path):
    with open(path, "rb") as f:
        data = f.read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    head = data[:end].decode("ascii").split("\n")
    assert head[0] == "ply" and head[1] == "format binary_little_endian 1.0"
    nv = int(next(h for h in head if h.startswith("element vertex")).split()[-1])
    nf = int(next(h for h in head if h.startswith("element face")).split()[-1])
    assert "property list uchar int vertex_indices" in head
    v = np.frombuffer(data, "<f4", nv * 3, end).reshape(nv, 3)
    off, faces = end + nv * 12, []
    for _ in range(nf):
        k = data[off]
        faces.append(struct.unpack_from(f"<{k}i", data, off + 1))
        off += 1 + 4 * k
    assert off == len(data)
    return v, np.array(faces, dtype=np.int64).reshape(-1, 3)


def test_write_ply_round_trip(tmp_path):
    mesh = importlib.import_module("selfsupervised-nvsf_b200.mesh")
    x, y, z = _grid(12, 5.5)
    v, t = M.marching_cubes((4.0 - np.sqrt(x * x + y * y + z * z)).astype(np.float32), 0.0)
    p = tmp_path / "sphere.ply"
    mesh.write_ply(str(p), torch.from_numpy(v), torch.from_numpy(t))
    rv, rt = _read_ply(p)
    assert np.array_equal(rv.view(np.uint32), v.view(np.uint32)) and np.array_equal(rt, t)
    mesh.write_ply(str(p), np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int64))
    rv, rt = _read_ply(p)
    assert rv.shape == (0, 3) and rt.shape == (0, 3)
    with pytest.raises(Exception):
        mesh.write_ply(str(p), v, t + len(v))


# ------------------------------------------------------------------------------------------------------ C ABI
def test_c_abi_rejects_invalid_arguments():
    """Every argument check fires before anything is launched, so it runs without a device; the pointers are
    never dereferenced."""
    L = _pkg()._lib.lib()
    p = ctypes.c_void_p(256)
    wsb = L.nvsf_marching_cubes_workspace_bytes
    for dims in ((1, 4, 4), (4, 1, 4), (4, 4, 1), (1025, 4, 4), (4, 1025, 4), (4, 4, 1025), (0, 0, 0)):
        assert wsb(*dims) == 0, dims
    assert wsb(2, 2, 2) > 0 and wsb(1024, 1024, 1024) >= 4 * 1024 ** 3
    assert wsb(1024, 1024, 1024) <= 4 * 1024 ** 3 + 16 * 1024 ** 2 + 4096       # 4 B per point + 8 per 1024
    assert wsb(64, 64, 64) <= wsb(64, 64, 65)
    need = wsb(8, 8, 8)
    ok = dict(vol=p, X=8, Y=8, Z=8, counts=p, ws=p, wb=need)

    def count(**kw):
        a = {**ok, **kw}
        return L.nvsf_marching_cubes_count(a["vol"], a["X"], a["Y"], a["Z"], 0.5, a["counts"], a["ws"], a["wb"],
                                           None)

    for bad in (dict(vol=None), dict(counts=None), dict(ws=None), dict(X=1), dict(Z=1025), dict(ws=ctypes.c_void_p(264))):
        assert count(**bad) == -1, bad
    assert count(wb=need - 1) == -2

    okw = dict(vol=p, X=8, Y=8, Z=8, v=p, vc=10, t=p, tc=10, ws=p, wb=need)

    def write(**kw):
        a = {**okw, **kw}
        return L.nvsf_marching_cubes_write(a["vol"], a["X"], a["Y"], a["Z"], 0.5, a["v"], a["vc"], a["t"], a["tc"],
                                           a["ws"], a["wb"], None)

    for bad in (dict(vol=None), dict(ws=None), dict(v=None), dict(t=None), dict(Y=0), dict(X=2048),
                dict(ws=ctypes.c_void_p(260))):
        assert write(**bad) == -1, bad
    assert write(wb=need - 1) == -2
