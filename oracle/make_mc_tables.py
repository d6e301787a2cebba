"""Generate csrc/mc_tables.cuh: the marching-cubes case table of nvsf_b200's mesh extraction (DESIGN.md §3.5).

The table is derived, not typed in.  Numbering:
  corner c = x | y << 1 | z << 2, at offset (c & 1, c >> 1 & 1, c >> 2 & 1) from the cell origin;
  edge   e = 4 * axis + (o0 + 2 * o1), o0 / o1 the corner offsets along the two other axes in increasing order
            (x-edges 0-3, y-edges 4-7, z-edges 8-11); its start corner has offset 0 along `axis`;
  case     = sum of 1 << c over the corners that are above the threshold.

For each case: every cube face is cut into segments between its crossing edges (on a face with four crossing
edges each above corner is cut off by its own segment); each segment is oriented so that, seen from outside the
cell, the above side is on its right; the segments chain into simple closed loops (each crossing edge lies on two
faces and has one segment on each), taken in order of their lowest edge and started there; each loop is
fan-triangulated from its first edge, or, when that fan would draw a chord between two edges of one face, from the
first edge after it along the loop whose fan draws none (every loop of every case has one).  A triangle's normal (v1 - v0) x (v2 - v0) then points out of the above
region, and neighbouring cells cut a shared face the same way, so the surface is closed and consistently oriented.

    python oracle/make_mc_tables.py            # rewrite the header
    python oracle/make_mc_tables.py --check    # exit 1 if the committed header differs
"""
import os
import sys

import numpy as np

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                      "selfsupervised-nvsf_b200", "csrc", "mc_tables.cuh")


def corner_pos(c):
    return np.array([c & 1, (c >> 1) & 1, (c >> 2) & 1], dtype=np.int64)


def _others(axis):
    return [a for a in range(3) if a != axis]


def edge_def(e):
    """(start corner, axis) of edge e."""
    axis, o = e >> 2, e & 3
    b0, b1 = _others(axis)
    return ((o & 1) << b0) | (((o >> 1) & 1) << b1), axis


EDGES = [edge_def(e) for e in range(12)]


def edge_mid(e):
    c, axis = EDGES[e]
    p = corner_pos(c).astype(np.float64)
    p[axis] = 0.5
    return p


def faces():
    """(axis, side, corners, edges) of the six faces."""
    out = []
    for axis in range(3):
        for side in (0, 1):
            corners = [c for c in range(8) if (c >> axis) & 1 == side]
            edges = [e for e in range(12) if EDGES[e][1] != axis and (EDGES[e][0] >> axis) & 1 == side]
            out.append((axis, side, corners, edges))
    return out


FACES = faces()


def _edge_corners(e):
    c, axis = EDGES[e]
    return c, c | (1 << axis)


def case_loops(case):
    above = [(case >> c) & 1 for c in range(8)]
    crossing = [e for e in range(12) if above[_edge_corners(e)[0]] != above[_edge_corners(e)[1]]]
    nxt, prv = {}, {}
    for axis, side, corners, edges in FACES:
        ce = [e for e in edges if e in crossing]
        if not ce:
            continue
        if len(ce) == 2:
            segs = [(ce[0], ce[1], next(c for c in corners if above[c]))]
        else:  # ambiguous face: each above corner is cut off by its own segment
            assert len(ce) == 4
            segs = [tuple(e for e in edges if c in _edge_corners(e)) + (c,) for c in corners if above[c]]
        n = np.zeros(3)
        n[axis] = 2 * side - 1
        for a, b, c in segs:
            P, Q = edge_mid(a), edge_mid(b)
            if np.dot(np.cross(n, Q - P), corner_pos(c) - P) > 0:
                a, b = b, a
            assert a not in nxt and b not in prv, (case, a, b)
            nxt[a], prv[b] = b, a
    assert sorted(nxt) == crossing and sorted(prv) == crossing, case
    loops, seen = [], set()
    for e in crossing:
        if e in seen:
            continue
        loop = [e]
        seen.add(e)
        while nxt[loop[-1]] != e:
            loop.append(nxt[loop[-1]])
            seen.add(loop[-1])
        loops.append(loop)
    return loops


FACES_OF_EDGE = [{f for f, (_, _, _, edges) in enumerate(FACES) if e in edges} for e in range(12)]


def _fan_apex(loop):
    """Position of the fan's apex: the first edge along the loop whose chords join no two edges of a common face.
    Such a chord lies in a face (one with four crossing edges) and the neighbouring cell may draw it too, which
    would leave that mesh edge in four triangles."""
    n = len(loop)
    for r in range(n):
        if not any(FACES_OF_EDGE[loop[r]] & FACES_OF_EDGE[loop[(r + i) % n]] for i in range(2, n - 1)):
            return r
    raise AssertionError(f"no valid fan apex for loop {loop}")


def case_triangles(case):
    tris = []
    for loop in case_loops(case):
        r = _fan_apex(loop)
        loop = loop[r:] + loop[:r]
        tris += [(loop[0], loop[i], loop[i + 1]) for i in range(1, len(loop) - 1)]
    return tris


def tables():
    """(tri_count [256] uint8, tris [256, max_tris, 3] int8 padded with -1, max_tris)."""
    per = [case_triangles(c) for c in range(256)]
    mx = max(len(t) for t in per)
    tris = np.full((256, mx, 3), -1, dtype=np.int8)
    for c, t in enumerate(per):
        if t:
            tris[c, :len(t)] = t
    return np.array([len(t) for t in per], dtype=np.uint8), tris, mx


def render():
    count, tris, mx = tables()
    lines = [
        "// Generated by oracle/make_mc_tables.py; do not edit.  Numbering and construction: that script and",
        "// DESIGN.md §3.5.",
        "#pragma once",
        "#include <stdint.h>",
        "",
        f"constexpr int kMcMaxTris = {mx};  // most triangles any case emits",
        "",
        "// edge e: start corner (x | y << 1 | z << 2) and axis",
        "__constant__ uint8_t c_mc_edge_corner[12] = {" + ", ".join(str(EDGES[e][0]) for e in range(12)) + "};",
        "__constant__ uint8_t c_mc_edge_axis[12] = {" + ", ".join(str(EDGES[e][1]) for e in range(12)) + "};",
        "",
        "// triangles per case",
        "__constant__ uint8_t c_mc_tri_count[256] = {",
    ]
    for r in range(0, 256, 32):
        lines.append("    " + ", ".join(str(int(v)) for v in count[r:r + 32]) + ",")
    lines += ["};", "", "// edges of each case's triangles, in emission order (-1: unused)",
              f"__constant__ int8_t c_mc_tris[256][{3 * mx}] = {{"]
    for c in range(256):
        lines.append(f"    {{{', '.join(str(int(v)) for v in tris[c].reshape(-1))}}},  // {c}")
    lines += ["};", ""]
    return "\n".join(lines)


if __name__ == "__main__":
    text = render()
    if "--check" in sys.argv:
        sys.exit(0 if open(HEADER).read() == text else 1)
    with open(HEADER, "w") as f:
        f.write(text)
    print(HEADER)
