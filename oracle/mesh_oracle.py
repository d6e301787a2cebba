"""numpy restatement of nvsf_marching_cubes (csrc/mesh.cu; contract in DESIGN.md §3.5), bit for bit.

Vertices: one per lattice edge whose endpoints differ in "above" (u > threshold; NaN is not above), ordered by
the owning point's linear index (i*Y + j)*Z + k and then by axis; t = (threshold - u_a) / (u_b - u_a) in float32,
clamped with fmin(fmax(t, 0), 1) (a NaN t lands on a), and the edge's axis coordinate is float32(index) + t.
Triangles: per cell in linear order, the case's triangles of oracle/make_mc_tables.py in table order, as int64
indices into the vertices."""
import numpy as np

from oracle.make_mc_tables import EDGES, tables

TRI_COUNT, TRIS, MAX_TRIS = tables()
EDGE_CORNER = np.array([c for c, _ in EDGES], dtype=np.int64)
EDGE_AXIS = np.array([a for _, a in EDGES], dtype=np.int64)
EDGE_OFF = np.stack([EDGE_CORNER & 1, (EDGE_CORNER >> 1) & 1, (EDGE_CORNER >> 2) & 1], 1)


def edge_bits(u, threshold):
    """[X,Y,Z,3] bool: the point's +x / +y / +z edge has a vertex."""
    A = u > np.float32(threshold)
    b = np.zeros(u.shape + (3,), dtype=bool)
    b[:-1, :, :, 0] = A[:-1] != A[1:]
    b[:, :-1, :, 1] = A[:, :-1] != A[:, 1:]
    b[:, :, :-1, 2] = A[:, :, :-1] != A[:, :, 1:]
    return b, A


def marching_cubes(u, threshold, slab=32):
    """(vertices [V,3] float32 in index space, triangles [T,3] int64)."""
    u = np.ascontiguousarray(u, dtype=np.float32)
    assert u.ndim == 3 and min(u.shape) >= 2
    tau = np.float32(threshold)
    X, Y, Z = u.shape
    bits, A = edge_bits(u, tau)
    flat = bits.reshape(-1)
    idx = np.flatnonzero(flat)
    p, ax = idx // 3, idx % 3
    uf = u.reshape(-1)
    ua, ub = uf[p], uf[p + np.array([Y * Z, Z, 1], dtype=np.int64)[ax]]
    with np.errstate(all="ignore"):
        t = (tau - ua) / (ub - ua)
    t = np.fmin(np.fmax(t, np.float32(0)), np.float32(1))
    verts = np.stack([p // (Y * Z), (p // Z) % Y, p % Z], 1).astype(np.float32)
    rows = np.arange(len(idx))
    verts[rows, ax] = verts[rows, ax] + t
    vid = (np.cumsum(flat, dtype=np.int64) - 1).reshape(X, Y, Z, 3)

    tris = []
    for i0 in range(0, X - 1, slab):
        i1 = min(i0 + slab, X - 1)
        a = A[i0:i1 + 1]
        cube = np.zeros((i1 - i0, Y - 1, Z - 1), dtype=np.int64)
        for c in range(8):
            dx, dy, dz = c & 1, (c >> 1) & 1, (c >> 2) & 1
            cube |= a[dx:dx + i1 - i0, dy:dy + Y - 1, dz:dz + Z - 1].astype(np.int64) << c
        cells = np.flatnonzero(TRI_COUNT[cube].reshape(-1))
        if not len(cells):
            continue
        cc = cube.reshape(-1)[cells]
        ci = cells // ((Y - 1) * (Z - 1)) + i0
        cj = (cells // (Z - 1)) % (Y - 1)
        ck = cells % (Z - 1)
        e = TRIS[cc].astype(np.int64)                      # [M, MAX_TRIS, 3]
        live = np.arange(MAX_TRIS)[None, :] < TRI_COUNT[cc][:, None]
        e = e[live]                                         # cell-major, then table order
        rep = np.repeat(np.arange(len(cells)), TRI_COUNT[cc].astype(np.int64))
        off = EDGE_OFF[e]                                   # [T, 3, 3]
        tris.append(vid[ci[rep][:, None] + off[..., 0], cj[rep][:, None] + off[..., 1],
                        ck[rep][:, None] + off[..., 2], EDGE_AXIS[e]])
    tri = np.concatenate(tris) if tris else np.zeros((0, 3), dtype=np.int64)
    return verts, tri.astype(np.int64)


# ---- mesh checks shared by the tests ------------------------------------------------------------------------
def directed_edge_counts(tri):
    """{(a, b): number of triangles with the directed edge a -> b}."""
    e = np.concatenate([tri[:, [0, 1]], tri[:, [1, 2]], tri[:, [2, 0]]])
    keys, counts = np.unique(e, axis=0, return_counts=True)
    return keys, counts


def is_closed_oriented(tri):
    """Every directed edge occurs once and its reverse occurs once: a closed, consistently oriented surface."""
    if len(tri) == 0:
        return True
    keys, counts = directed_edge_counts(tri)
    if (counts != 1).any():
        return False
    n = int(tri.max()) + 1
    fwd = keys[:, 0] * n + keys[:, 1]
    rev = keys[:, 1] * n + keys[:, 0]
    return bool(np.isin(rev, fwd).all())


def euler_characteristic(verts_used, tri):
    keys, _ = directed_edge_counts(tri)
    undirected = np.unique(np.sort(keys, axis=1), axis=0)
    return int(verts_used) - len(undirected) + len(tri)
