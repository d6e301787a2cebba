"""Seeded input cases shared by the CPU (oracle vs golden) and GPU (CUDA vs oracle / reference
extension) parity tests and by oracle/make_golden_raymarching.py."""
import importlib

import numpy as np

S = importlib.import_module("selfsupervised-nvsf_b200.synth")

THRESH = 0.01  # renderer_dynamic.py:75 density_thresh default


def bitfield(fill, seed=0):
    return S.packbits_np(S.density_grid(fill, seed=seed), THRESH)


def march_inputs(kind, n, seed, perturb):
    """rays + near/far + noises for the marchers.  kind: 'lidar' | 'camera'."""
    rng = np.random.default_rng(1000 + seed)
    if kind == "lidar":
        o, d = S.lidar_rays(n, seed=seed)
        N = o.shape[0]
        nears = np.full(N, S.MIN_NEAR_LIDAR, np.float32)
        fars = np.full(N, S.LIDAR_MAX_DEPTH, np.float32)
    else:
        o, d = S.camera_rays(n, seed=seed)
        from oracle import raymarching_oracle as O
        nears, fars = O.near_far_from_aabb(o, d, S.AABB, S.MIN_NEAR)
        N = o.shape[0]
    noises = rng.random(N, dtype=np.float32) if perturb else np.zeros(N, np.float32)
    return o, d, nears, fars, noises


def field_values(M, seed):
    """Random per-sample sigmas / rgbs (what the field would return)."""
    rng = np.random.default_rng(2000 + seed)
    sigmas = np.exp(rng.normal(0.0, 2.0, size=M)).astype(np.float32)
    rgbs = rng.random((M, 3), dtype=np.float32)
    return sigmas, rgbs


COMPOSITE_COUNTS = (0, 1, 3, 4, 5, 15, 16, 17, 31, 32, 33, 48, 200, 768)
COMPOSITE_TERM_AT = (0, 3, 4, 15, 16, 17, 31, 32, -1)   # -1: the ray's last sample


def composite_table(N, seed):
    """A hand-built training ray table for the compositing kernels, with every hand-over on purpose.

    Per-ray counts from COMPOSITE_COUNTS (every count with every termination point of COMPOSITE_TERM_AT that
    fits it appears), early termination placed at sample k by a sigma that makes alpha 1 (sigma*delta >= 100)
    or 1 - 6e-6 (sigma*delta = 12).  Elsewhere sigma*delta is 2/c .. 8/c for a ray of c samples: T stays above
    e^-8 = 3.4e-4, three times T_thresh = 1e-4, so the termination point never depends on exp's last bit and is
    known here; and no alpha is so small that the ~2^-22 absolute difference between the GPU's and the oracle's
    exp breaks a 1e-5 relative comparison of the composited values.  Rows of the table are in
    shuffled order (index != i), rays sit in memory in another shuffled order with 0..3 gap rows between them,
    count-0 rays point anywhere, and the ray stored last runs past M.  Gap rows and the overflowing ray's rows
    hold NaN; so do the samples after a placed termination point, which a kernel may read but never use.

    Returns dict(rays [N,3] int32, sigmas [M], rgbs [M,3], deltas [M,2], written [M] bool: the samples whose
    gradients a backward writes, owned [M] bool: the rows of a ray that fits, dead [N] bool: rays that must
    produce zeros (count 0 or past M), term [N] int32: placed termination sample or -1)."""
    rng = np.random.default_rng(3000 + seed)
    counts = np.empty(N, np.int64)
    term = np.full(N, -1, np.int64)
    fixed = [(c, k) for c in COMPOSITE_COUNTS for k in (None,) + COMPOSITE_TERM_AT
             if c > 0 and (k is None or k < c)]
    nf = min(len(fixed), N - 1)
    for i, (c, k) in enumerate(fixed[:nf]):
        counts[i] = c
        term[i] = -1 if k is None else (c - 1 if k == -1 else k)
    p = np.array([4, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 4, 1, 0.25])
    counts[nf:] = rng.choice(COMPOSITE_COUNTS, size=N - nf, p=p / p.sum())
    placed = (rng.random(N - nf) < 0.5) & (counts[nf:] > 0)
    term[nf:] = np.where(placed, (rng.random(N - nf) * counts[nf:]).astype(np.int64), -1)
    # slot r is ray id ids[r]; slots are stored in memory in mem_order, the overflowing one (not a fixed case) last
    ids = rng.permutation(N)
    over = int(rng.integers(nf, N))
    mem_order = rng.permutation(np.delete(np.arange(N), over))
    mem_order = np.append(mem_order, over)
    counts[over] = 33
    term[over] = -1
    offsets = np.empty(N, np.int64)
    pos = 0
    for r in mem_order:
        pos += int(rng.integers(0, 4))
        if counts[r] == 0:
            offsets[r] = int(rng.integers(0, pos + 1))
            continue
        offsets[r] = pos
        pos += int(counts[r])
    M = int(offsets[over] + counts[over] - 5)          # the last ray runs 5 samples past the end
    nan = np.float32(np.nan)
    sig = np.full(M, nan, np.float32)
    rgb = np.full((M, 3), nan, np.float32)
    dl = np.full((M, 2), nan, np.float32)
    owned = np.zeros(M, bool)
    written = np.zeros(M, bool)
    dead = (counts == 0) | (offsets + counts > M)
    for r in range(N):
        c, o, k = int(counts[r]), int(offsets[r]), int(term[r])
        if dead[r]:
            continue
        s = slice(o, o + c)
        owned[s] = True
        dl[s] = (np.float32(1e-3) + rng.random((c, 2), dtype=np.float32) * np.float32(9e-3))
        sig[s] = (rng.uniform(2.0, 8.0, c) / c / dl[s, 0]).astype(np.float32)   # sigma*delta in [2, 8] / c
        rgb[s] = rng.random((c, 3), dtype=np.float32)
        if k >= 0:
            sig[o + k] = np.float32(1e5) if r % 2 else np.float32(12.0) / dl[o + k, 0]
            sig[o + k + 1:o + c] = nan
            rgb[o + k + 1:o + c] = nan
            dl[o + k + 1:o + c] = nan
            written[o:o + k + 1] = True
        else:
            written[s] = True
    row_order = rng.permutation(N)
    rays = np.empty((N, 3), np.int32)
    rays[:, 0] = ids[row_order]
    rays[:, 1] = offsets[row_order]
    rays[:, 2] = counts[row_order]
    # outputs are indexed by ray id: map per-ray flags from memory slot r to id ids[r]
    dead_by_id = np.zeros(N, bool)
    dead_by_id[ids] = dead
    term_by_id = np.full(N, -1, np.int32)
    term_by_id[ids] = term
    return dict(rays=rays, sigmas=sig, rgbs=rgb, deltas=dl, written=written, owned=owned,
                dead=dead_by_id, term=term_by_id, M=M)


def canonical_from_rays(rays, arrays):
    """Re-order the per-sample `arrays` of a marcher result into ray-id order.

    rays [N,3] rows (id, offset, count) in ANY order (the reference's order is scheduling
    dependent, raymarching.cu:445-454).  Returns (rays sorted by id with prefix-sum offsets,
    list of arrays concatenated in that order)."""
    rays = np.asarray(rays)
    order = np.argsort(rays[:, 0], kind="stable")
    r = rays[order]
    new_off = np.concatenate([[0], np.cumsum(r[:, 2])[:-1]]).astype(np.int32)
    total = int(r[:, 2].sum())
    idx = np.empty(total, np.int64)
    pos = 0
    for (rid, off, cnt) in r:
        idx[pos:pos + cnt] = np.arange(off, off + cnt)
        pos += cnt
    out_rays = np.stack([r[:, 0], new_off, r[:, 2]], 1).astype(np.int32)
    return out_rays, [np.asarray(a)[idx] for a in arrays]
