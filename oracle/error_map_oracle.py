"""TEST INFRASTRUCTURE — numpy restatement of error-map guided ray sampling and its update.

torch-ngp's error-map branch of get_rays (the weighted coarse-cell draw and its jittered pixels) and the map update
of its train_step, the convention the reference's dataset and trainer derive from; their sources are not in this
tree: PARITY UNPINNED.  The contract is DESIGN.md §3.5.  Exact by construction (fp32 keys, a total order with
explicit tie rules), so the GPU is compared with it bit for bit.

Only tests/ and the tools/ benchmarks may import this module.
"""
import numpy as np

f32 = np.float32


def error_map_sample(w, E, jitter, res, N, H, W):
    """One map w [res*res] -> (inds_coarse [N], inds [N]) int64, the contract of DESIGN.md §3.5: the N
    smallest keys E / w (fp32) over the positive-weight cells (w > 0 and finite), ties to the lower cell,
    filled by the smallest E among the other cells when fewer than N are positive; cells in ascending
    order; pixel (row, col) of output j from jitter[j] = (u0, u1) by torch-ngp's expression."""
    w, E = np.asarray(w, f32), np.asarray(E, f32)
    jitter = np.asarray(jitter, f32).reshape(-1, 2)
    R = res * res
    assert w.shape == (R,) and E.shape == (R,) and 1 <= N <= R and jitter.shape[0] >= N
    pos = (w > 0) & np.isfinite(w)
    with np.errstate(over="ignore", divide="ignore", invalid="ignore"):
        key = np.where(pos, E / np.where(pos, w, f32(1)), E).astype(f32)
    order = np.lexsort((np.arange(R), key, ~pos))  # tier (positive first), then key, then cell index
    cells = np.sort(order[:N]).astype(np.int64)
    sx, sy = f32(H / res), f32(W / res)
    fr = (cells // res).astype(f32) * sx + jitter[:N, 0] * sx
    fc = (cells % res).astype(f32) * sy + jitter[:N, 1] * sy
    row = np.minimum(fr.astype(np.int64), H - 1)
    col = np.minimum(fc.astype(np.int64), W - 1)
    return cells, row * W + col


def error_map_update(m, inds_coarse, loss):
    """torch-ngp's train_step update of one map row: m[c] = 0.1 * m[c] + 0.9 * loss (fp32), returned as a
    new array; inds_coarse holds distinct cells."""
    m = np.array(m, dtype=f32)
    ic = np.asarray(inds_coarse, np.int64)
    m[ic] = f32(0.1) * m[ic] + f32(0.9) * np.asarray(loss, f32)
    return m
