"""Mesh extraction on the device: marching cubes over a density volume (C ABI Part 7, csrc/mesh.cu) and a PLY
writer — the replacement of torch-ngp's save_mesh, whose mcubes / trimesh dependencies this project does not have.

``marching_cubes`` is a drop-in for ``mcubes.marching_cubes(u, threshold)``: vertices in index space, triangles
as vertex indices, both on the device.  The contract (vertex order, interpolation, triangle table, winding) is
DESIGN.md §3.5.  NeRFNetwork.extract_geometry builds the volume from the field.  GPU tensors only; no CPU fallback.
"""
import numpy as np
import torch

from . import _lib
from ._lib import NvsfError, check, ptr, stream_ptr


@torch.no_grad()
@_lib.device_guard
def marching_cubes(volume, threshold):
    """volume [X,Y,Z] (CUDA, converted to contiguous fp32; each dimension in [2, 1024]), lattice point (i,j,k) =
    volume[i,j,k]; a point is inside when its value is > threshold.  Returns (vertices [V,3] fp32 in index space,
    triangles [T,3] int64), the normal (v1-v0)x(v2-v0) pointing out of the inside.  One host read (the two
    counts, to size the outputs)."""
    if not torch.is_tensor(volume) or not volume.is_cuda:
        raise NvsfError("marching_cubes: volume must be a CUDA tensor")
    if volume.dim() != 3:
        raise NvsfError(f"marching_cubes: volume must be [X, Y, Z], got {tuple(volume.shape)}")
    u = volume.detach().to(torch.float32).contiguous()
    X, Y, Z = (int(s) for s in u.shape)
    L = _lib.lib()
    wb = L.nvsf_marching_cubes_workspace_bytes(X, Y, Z)
    if wb == 0:
        raise NvsfError(f"marching_cubes: volume {X}x{Y}x{Z} out of range (each dimension in [2, 1024])")
    ws = torch.empty(wb, dtype=torch.uint8, device=u.device)
    counts = torch.empty(2, dtype=torch.int64, device=u.device)
    tau = float(threshold)
    check(L.nvsf_marching_cubes_count(ptr(u), X, Y, Z, tau, ptr(counts), ptr(ws), wb, stream_ptr()),
          "marching_cubes_count")
    V, T = counts.tolist()
    vertices = torch.empty(V, 3, dtype=torch.float32, device=u.device)
    triangles = torch.empty(T, 3, dtype=torch.int64, device=u.device)
    check(L.nvsf_marching_cubes_write(ptr(u), X, Y, Z, tau, ptr(vertices), V, ptr(triangles), T, ptr(ws), wb,
                                      stream_ptr()), "marching_cubes_write")
    return vertices, triangles


def write_ply(path, vertices, triangles):
    """Binary little-endian PLY: vertex (float x, y, z), face (list uchar int vertex_indices).  vertices [V,3],
    triangles [T,3] (tensors on any device, or arrays)."""
    v = np.ascontiguousarray(torch.as_tensor(vertices).detach().cpu().numpy(), dtype="<f4").reshape(-1, 3)
    t = torch.as_tensor(triangles).detach().cpu().numpy().reshape(-1, 3)
    if len(v) > 2 ** 31 - 1:
        raise NvsfError(f"write_ply: {len(v)} vertices do not fit the PLY int vertex indices")
    if len(t) and (t.min() < 0 or t.max() >= len(v)):
        raise NvsfError("write_ply: triangle index out of range")
    faces = np.empty(len(t), dtype=[("n", "u1"), ("i", "<i4", (3,))])
    faces["n"] = 3
    faces["i"] = t
    head = ("ply\nformat binary_little_endian 1.0\n"
            f"element vertex {len(v)}\nproperty float x\nproperty float y\nproperty float z\n"
            f"element face {len(t)}\nproperty list uchar int vertex_indices\nend_header\n")
    with open(path, "wb") as f:
        f.write(head.encode("ascii"))
        f.write(v.tobytes())
        f.write(faces.tobytes())
