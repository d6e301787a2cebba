"""TEST INFRASTRUCTURE.  float64 restatement of the table-gradient half of the training backward
(csrc/train.cu: k_encode_bwd, k_flowgrid_bwd and the k_expand_* transposes of the time collapse),
fed the per-sample gradients the CUDA backward itself kept in its scratch buffer.

Every scatter of that path is linear in the per-sample gradient it is fed (for the planes: given
the texels of the product rule), so given the kernel's own `dfeat`, `dflowfeat`, `flow` and
fractions, the float64 transpose differs from the kernel only by fp32 rounding and the order of the
atomic adds.  The restatement returns, per entry of the master layouts, the float64 gradient, the
float64 sum A of the absolute values of the terms that land there (it sets the tolerance) and the
term count.

Semantics restated from oracle/field_oracle.py (the reference's NeRFNetwork.density encoders):
  static planes   product rule g*B*C, g*A*C, g*A*B of the three space planes, texels from the fp32
                  masters or their fp16 mirror (option enc_bwd_h16)
  time planes     queries t, (f+1)/F, (f-1)/F with weights 0.5 / 0.25 / 0.25; a missing neighbour frame
                  re-uses the un-warped query; rows blended over the two time rows of each query
  flow            coordinate gradient of the warped plane queries, grid_sample(align_corners=True,
                  padding_mode="border"): zero where the coordinate is clipped or on a border texel
  hashes          tcnn grid transpose; the dynamic 2-D hashes get gradient through the un-warped query
                  only, factor 0.5 + 0.25 per missing neighbour; time slices k1 / k2 blended and the
                  lagrange4 basis over the 4 features; the flow grid lagrange4 over its feature pairs
  liveness        a row whose scaled fp16 sigma-net output gradient is zero in all 16 columns adds
                  nothing (its dfeat may be unwritten and is never read); the flow grid applies the same
                  test to dflow with the flow scale

Index arithmetic (`exact=False`) is fp32 exactly as the kernels do it: the contractions below were
read from the SASS of the sm_100a library (cuobjdump -sass csrc/_obj/train.o and field.o):
  uniform_z   lin = k * step (k < S/2) or fma(S-1-k, -step, 1); z = fma(far - near, lin, near);
              z = fma(noise - 0.5, (far - near) / S, z)
  position    p = fma(d, z, o), clamped to +-bound; x = (p + bound) * (1 / (2 bound))
  grid_pos    fma(scale, x, 0.5), floor, frac
  collapse    time row = fma(1 - w, row_y0, w * row_y1)   (k_collapse_planes_dyn)
An FMA is emulated by forming the product exactly in float64 and rounding the sum once to float32.
`exact=True` takes float64 positions and forms the fractions in float64 (tests/test_encoder_bwd_oracle.py
compares that mode with torch.autograd of field_oracle's own encoder functions).
"""
import numpy as np

from .field_oracle import PLANE_COMBS, lagrange4

f32 = np.float32
_PRIMES = (1, 2654435761, 805459861)
_M32 = np.uint64(0xFFFFFFFF)
_TIME_COMBS = (2, 4, 5)   # (0,3), (1,3), (2,3)
_SPACE_COMBS = (0, 1, 3)  # (0,1), (0,2), (1,2)


def fma32(a, b, c):
    """fmaf(a, b, c) of float32 operands: the product is exact in float64, the sum is rounded to
    float32 (a second rounding differs only when float64 lands on a float32 tie, ~2^-29)."""
    return (np.asarray(a, np.float32).astype(np.float64) * np.asarray(b, np.float32).astype(np.float64)
            + np.asarray(c, np.float32).astype(np.float64)).astype(np.float32)


def uniform_z(nears, fars, S, noise=None):
    """z values [N, S] of the uniform sampler (field_common.cuh uniform_z), float32."""
    nears, fars = np.asarray(nears, f32), np.asarray(fars, f32)
    k = np.arange(S, dtype=np.int64)
    step = f32(1.0) / f32(max(S - 1, 1))
    lin = np.where(k < S // 2, k.astype(f32) * step, fma32((S - 1 - k).astype(f32), -step, f32(1.0)))
    span = fars - nears
    z = fma32(span[:, None], lin[None, :], nears[:, None])
    if noise is not None:
        z = fma32(np.asarray(noise, f32) - f32(0.5), (span / f32(S))[:, None], z)
    return z


def sample_positions(rays_o, rays_d, nears, fars, S, bound, noise=None):
    """Normalised sample positions [N*S, 3] (float32) and z [N, S] exactly as k_encode_bwd forms them."""
    z = uniform_z(nears, fars, S, noise)
    o, d = np.asarray(rays_o, f32).reshape(-1, 3), np.asarray(rays_d, f32).reshape(-1, 3)
    p = fma32(d[:, None, :], z[:, :, None], o[:, None, :])
    b = f32(bound)
    p = np.minimum(np.maximum(p, -b), b)
    inv2b = f32(1.0) / (b + b)
    return ((p + b) * inv2b).reshape(-1, 3), z


def _fp16(v):
    return np.asarray(v, np.float32).astype(np.float16).astype(np.float64)


def row_live(dout, scale):
    """The backward's zero test: the row is live iff fp16(scale * dout) is non-zero in some column."""
    return (np.asarray(dout, f32) * f32(scale)).astype(np.float16).astype(np.float32).any(axis=1)


class _Acc:
    """Per-entry float64 sum, absolute sum and term count of one flat master gradient tensor."""

    def __init__(self, n):
        self.g, self.a, self.k = np.zeros(n), np.zeros(n), np.zeros(n, np.int64)

    def add(self, offset, size, idx, val, absval):
        idx = np.asarray(idx, np.int64).reshape(-1)
        val, absval = np.asarray(val, np.float64).reshape(-1), np.asarray(absval, np.float64).reshape(-1)
        sl = slice(offset, offset + size)
        self.g[sl] += np.bincount(idx, weights=val, minlength=size)
        self.a[sl] += np.bincount(idx, weights=absval, minlength=size)
        self.k[sl] += np.bincount(idx, weights=(absval != 0).astype(np.float64), minlength=size).astype(np.int64)


class _Arith:
    """fp32 kernel arithmetic (exact=False) or float64 (exact=True) for positions and fractions."""

    def __init__(self, exact):
        self.exact = exact
        self.dt = np.float64 if exact else np.float32

    def grid_pos(self, scale, x):
        if self.exact:
            p = x * np.float64(f32(scale)) + 0.5
        else:
            p = fma32(f32(scale), x, f32(0.5))
        fl = np.floor(p)
        return fl.astype(np.int64), (p - fl).astype(np.float64)

    def plane_coord(self, p, R):
        """grid_sample(align_corners=True, border) along one axis: texels i0, i1, weight of i1 and
        d(texel coordinate)/dp (R-1 strictly inside, 0 where the coordinate is clipped or on a border)."""
        dt = self.dt
        p = np.asarray(p, dt)
        f = ((p * dt(2.0) - dt(1.0)) + dt(1.0)) * dt(0.5) * dt(R - 1)
        dcoord = np.where((f > 0) & (f < R - 1), float(R - 1), 0.0)
        f = np.minimum(np.maximum(f, dt(0.0)), dt(R - 1))
        fl = np.floor(f)
        i0 = fl.astype(np.int64)
        return i0, np.minimum(i0 + 1, R - 1), (f - fl).astype(np.float64), dcoord


def time_info(t, num_frames, tres, exact=False):
    """k_time_setup: per query q (t, (f+1)/F, (f-1)/F) validity, lagrange4 basis, hash slices and
    plane time rows; fp32 like the kernel unless exact (then float64 fractions, as field_oracle)."""
    t = f32(t)
    f = int(t * f32(num_frames - 1))
    ts = [t, f32((f + 1) / num_frames), f32((f - 1) / num_frames)]
    out = dict(valid=[True, f < num_frames - 1, f > 0], lag=[], k1=[], k2=[], wk=[], y0=[], y1=[], wy=[])
    for tq in ts:
        lag = lagrange4(float(tq))
        out["lag"].append(lag if exact else [float(f32(v)) for v in lag])
        idx = tq * f32(tres - 1)
        k1 = min(max(int(np.floor(idx)), 0), tres - 1)
        k2 = min(max(int(np.ceil(idx)), 0), tres - 1)
        out["k1"].append(k1)
        out["k2"].append(k2)
        out["wk"].append(0.0 if k1 == k2 else float(idx - f32(k1)))
        if exact:
            iy = ((float(tq) * 2.0 - 1.0) + 1.0) * 0.5 * (tres - 1)
        else:
            iy = ((tq * f32(2.0) - f32(1.0)) + f32(1.0)) * f32(0.5) * f32(tres - 1)
        iy = min(max(iy, 0.0), float(tres - 1))
        y0 = int(np.floor(iy))
        out["y0"].append(y0)
        out["y1"].append(min(y0 + 1, tres - 1))
        out["wy"].append(float(iy - np.floor(iy)))
    return out


def _hash_index(lv, cells):
    """tcnn corner index (uint32 arithmetic; dense levels wrap with % size)."""
    if lv["hashed"]:
        h = np.zeros(cells[0].shape, np.uint64)
        for d, c in enumerate(cells):
            h ^= (c.astype(np.uint64) * np.uint64(_PRIMES[d])) & _M32
        return (h & np.uint64(lv["size"] - 1)).astype(np.int64)
    lin, stride = np.zeros(cells[0].shape, np.uint64), 1
    for c in cells:
        lin = (lin + c.astype(np.uint64) * np.uint64(stride)) & _M32
        stride *= lv["res"]
    return (lin % np.uint64(lv["size"])).astype(np.int64)


def warp_heads(keys, live):
    """Run heads of k_encode_bwd / k_flowgrid_bwd per 32-sample warp: a lane starts a run when it is
    lane 0, it or its predecessor is not live, or its cell differs from its predecessor's.
    keys: [n] int cell keys; returns [n_warps] head counts (lanes past n are not live)."""
    n = keys.shape[0]
    nw = (n + 31) // 32
    k = np.full(nw * 32, -1, np.int64)
    lv = np.zeros(nw * 32, bool)
    k[:n], lv[:n] = keys, live
    head = np.ones(nw * 32, bool)
    head[1:] = (~lv[1:]) | (~lv[:-1]) | (k[1:] != k[:-1])
    head[::32] = True
    return head.reshape(nw, 32).sum(1)


def encoder_bwd(cfg, params, mod, x, t, flow, dfeat, dgeo16, dflow, dflowfeat, scale_sigma, scale_flow,
                h16, exact=False):
    """Gradients of the master tables hash_static, hash_dynamic, planes (of modality `mod`) and flow_grid.

    x [n,3] normalised positions (float32 from sample_positions, or float64 with exact=True);
    flow [n,>=6] the forward's flow; dfeat [n,>=120], dgeo16 [n,16], dflow [n,>=6], dflowfeat [n,32]:
    the backward's per-sample gradients; params: flat float tensors / arrays in the oracle layout.
    Returns dict(grads={name: (g, A, k)}, dflow=[n,6], dflow_abs=[n,6], live, flow_live, runs) where
    runs = {"hash_static": [levels, warps], "hash_dynamic": [3*levels, warps], "flow_grid": [...]} head counts."""
    ar = _Arith(exact)
    npy = lambda v: v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
    x = np.asarray(x, ar.dt)
    n = x.shape[0]
    flow = np.asarray(flow, ar.dt)[:, :6]
    sizes = cfg.sizes()
    live = row_live(dgeo16, scale_sigma)
    flive = row_live(np.asarray(dflow)[:, :6], scale_flow)
    g = np.asarray(dfeat)[live].astype(np.float64)          # only live rows are read
    F, Tn = cfg.n_features_hash, cfg.time_resolution
    ti = time_info(t, cfg.num_frames, Tn, exact)
    res = {}
    runs = {}

    # ---- planes -------------------------------------------------------------------------------
    planes = npy(params[mod]["planes"]).astype(np.float64)
    acc = _Acc(sizes["planes"])
    dfl = np.zeros((n, 6))
    dfl_abs = np.zeros((n, 6))
    xl = x[live]
    m = xl.shape[0]
    off = 0
    offs = []
    for r in cfg.plane_res:
        o = {}
        for ci, (a, b) in enumerate(PLANE_COMBS):
            o[ci] = off
            off += cfg.n_features_plane * r[a] * r[b]
        offs.append(o)
    qpos, qtab = [], []
    for q in range(3):
        if q == 0 or not ti["valid"][q]:
            qpos.append(xl)
            qtab.append(0)
        else:
            fq = flow[live][:, 3 * (q - 1):3 * q]
            qpos.append(xl + fq if exact else (xl + fq).astype(f32))
            qtab.append(q)
    for s, r in enumerate(cfg.plane_res):
        R, Tres, PF = r[0], r[3], cfg.n_features_plane
        # (a) space planes
        g8 = g[:, PF * s:PF * (s + 1)]
        samp, sabs, geo = [], [], []
        for ci, (a, b) in zip(_SPACE_COMBS, [PLANE_COMBS[c] for c in _SPACE_COMBS]):
            tab = planes[offs[s][ci]:offs[s][ci] + PF * R * R].reshape(PF, R, R)
            if h16:
                tab = _fp16(tab)
            i0, i1, wx, _ = ar.plane_coord(xl[:, a], R)
            j0, j1, wy, _ = ar.plane_coord(xl[:, b], R)
            corners = [(j0, i0, (1 - wx) * (1 - wy)), (j0, i1, wx * (1 - wy)), (j1, i0, (1 - wx) * wy),
                       (j1, i1, wx * wy)]
            v = sum(w[:, None] * tab[:, jj, ii].T for jj, ii, w in corners)
            va = sum(w[:, None] * np.abs(tab[:, jj, ii].T) for jj, ii, w in corners)
            samp.append(v)
            sabs.append(va)
            geo.append((ci, corners))
        for p3 in range(3):
            o1, o2 = [k for k in range(3) if k != p3]
            d = g8 * samp[o1] * samp[o2]
            da = np.abs(g8) * sabs[o1] * sabs[o2]
            ci, corners = geo[p3]
            for jj, ii, w in corners:
                idx = (np.arange(PF)[None, :] * R * R + (jj * R + ii)[:, None])
                acc.add(offs[s][ci], PF * R * R, idx, w[:, None] * d, w[:, None] * da)
        # (b) time planes
        g8 = g[:, 32 + PF * s:32 + PF * (s + 1)]
        for q in range(3):
            wq = 0.5 if q == 0 else 0.25
            qq = qtab[q]
            y0, y1, wy = ti["y0"][qq], ti["y1"][qq], ti["wy"][qq]
            rows, rabs, lin = [], [], []
            for axis, ci in enumerate(_TIME_COMBS):
                tab = planes[offs[s][ci]:offs[s][ci] + PF * Tres * R].reshape(PF, Tres, R)
                if exact:
                    row = (1.0 - wy) * tab[:, y0, :] + wy * tab[:, y1, :]
                else:
                    w32 = f32(wy)
                    row = fma32(f32(1.0) - w32, tab[:, y0, :].astype(f32),
                                w32 * tab[:, y1, :].astype(f32)).astype(np.float64)
                if h16:
                    row = _fp16(row)
                i0, i1, w, dc = ar.plane_coord(qpos[q][:, axis], R)
                a0, a1 = row[:, i0].T, row[:, i1].T
                rows.append((1 - w)[:, None] * a0 + w[:, None] * a1)
                rabs.append((1 - w)[:, None] * np.abs(a0) + w[:, None] * np.abs(a1))
                lin.append((ci, i0, i1, w, dc, a1 - a0, np.abs(a0) + np.abs(a1)))
            for axis in range(3):
                o1, o2 = [k for k in range(3) if k != axis]
                d = wq * g8 * rows[o1] * rows[o2]
                da = wq * np.abs(g8) * rabs[o1] * rabs[o2]
                ci, i0, i1, w, dc, slope, sa = lin[axis]
                # the collapsed [R][8] row of this query, then its two time rows (k_expand_planes_dyn)
                col = _Acc(R * PF)
                for ii, wx in ((i0, 1 - w), (i1, w)):
                    idx = ii[:, None] * PF + np.arange(PF)[None, :]
                    col.add(0, R * PF, idx, wx[:, None] * d, wx[:, None] * da)
                for yy, wt in ((y0, 1.0 - wy), (y1, wy)):
                    sl = (slice(None), yy, slice(None))
                    dst = [v[offs[s][ci]:offs[s][ci] + PF * Tres * R].reshape(PF, Tres, R) for v in (acc.g, acc.a, acc.k)]
                    dst[0][sl] += wt * col.g.reshape(R, PF).T
                    dst[1][sl] += abs(wt) * col.a.reshape(R, PF).T
                    dst[2][sl] += col.k.reshape(R, PF).T * (wt != 0)
                if q > 0 and ti["valid"][q]:
                    col = 3 * (q - 1) + axis
                    dfl[live, col] += (d * slope).sum(1) * dc
                    dfl_abs[live, col] += (da * sa).sum(1) * dc
    res["planes"] = acc

    # ---- static hash --------------------------------------------------------------------------
    acc = _Acc(sizes["hash_static"])
    keys_runs = []
    for l, lv in enumerate(cfg.static_levels):
        cw = [ar.grid_pos(lv["scale"], x[:, dd]) for dd in range(3)]
        key = cw[0][0] + (cw[1][0] << 21) + (cw[2][0] << 42)
        keys_runs.append(warp_heads(key, live))
        cells = [c[live] for c, _ in cw]
        ws = [w[live] for _, w in cw]
        g4 = g[:, 64 + F * l:64 + F * (l + 1)]
        idx, val = [], []
        for c in range(8):
            bits = [(c >> dd) & 1 for dd in range(3)]
            w = np.prod([ws[dd] if bits[dd] else 1 - ws[dd] for dd in range(3)], axis=0)
            e = _hash_index(lv, [cells[dd] + bits[dd] for dd in range(3)])
            idx.append(e[:, None] * F + np.arange(F)[None, :])
            val.append(w[:, None] * g4)
        val = np.concatenate([v.reshape(-1) for v in val])
        acc.add(lv["offset"] * F, lv["size"] * F, np.concatenate([i.reshape(-1) for i in idx]), val, np.abs(val))
    res["hash_static"] = acc
    runs["hash_static"] = np.stack(keys_runs)

    # ---- dynamic 2-D hashes (un-warped query only): collapsed table, then the time expansion ---------
    # (each master entry receives one collapsed entry times a fixed factor, so its A is that factor times
    #  the collapsed entry's)
    acc = _Acc(sizes["hash_dynamic"])
    fac = 0.5 + 0.25 * (not ti["valid"][1]) + 0.25 * (not ti["valid"][2])
    k1, k2, wk, lag = ti["k1"][0], ti["k2"][0], ti["wk"][0], ti["lag"][0]
    blend = [(k1, 1.0)] if k1 == k2 else [(k1, 1.0 - wk), (k2, wk)]
    base = 0
    keys_runs = []
    for pi, dims in enumerate(([0, 1], [0, 2], [1, 2])):
        E = cfg.dyn_entries[pi]
        col = _Acc(E)
        for l, lv in enumerate(cfg.dyn_levels[pi]):
            cw = [ar.grid_pos(lv["scale"], x[:, dd]) for dd in dims]
            keys_runs.append(warp_heads(cw[0][0] + (cw[1][0] << 21), live))
            cells = [c[live] for c, _ in cw]
            ws = [w[live] for _, w in cw]
            gs = fac * g[:, 96 + 8 * pi + l]
            for c in range(4):
                bits = [c & 1, c >> 1]
                w = np.prod([ws[dd] if bits[dd] else 1 - ws[dd] for dd in range(2)], axis=0)
                e = _hash_index(lv, [cells[dd] + bits[dd] for dd in range(2)])
                col.add(lv["offset"], lv["size"], e, w * gs, np.abs(w * gs))
        for k, wb in blend:
            for i in range(F):
                sl = slice(base + k * E * F + i, base + (k + 1) * E * F, F)
                acc.g[sl] += wb * lag[i] * col.g
                acc.a[sl] += abs(wb * lag[i]) * col.a
                acc.k[sl] += col.k * (wb * lag[i] != 0)
        base += Tn * E * F
    res["hash_dynamic"] = acc
    runs["hash_dynamic"] = np.stack(keys_runs)

    # ---- flow grid: collapsed [entries][nb] table, then lagrange4 over the feature groups ------------
    acc = _Acc(sizes["flow_grid"])
    FF = cfg.flow_features
    nb = FF // 4
    col = _Acc(cfg.flow_entries * nb)
    keys_runs = []
    gf = np.asarray(dflowfeat)[flive].astype(np.float64)
    for l, lv in enumerate(cfg.flow_grid_levels):
        cw = [ar.grid_pos(lv["scale"], x[:, dd]) for dd in range(3)]
        keys_runs.append(warp_heads(cw[0][0] + (cw[1][0] << 21) + (cw[2][0] << 42), flive))
        cells = [c[flive] for c, _ in cw]
        ws = [w[flive] for _, w in cw]
        g2 = gf[:, nb * l:nb * (l + 1)]
        idx, val = [], []
        for c in range(8):
            bits = [(c >> dd) & 1 for dd in range(3)]
            w = np.prod([ws[dd] if bits[dd] else 1 - ws[dd] for dd in range(3)], axis=0)
            e = _hash_index(lv, [cells[dd] + bits[dd] for dd in range(3)])
            idx.append(e[:, None] * nb + np.arange(nb)[None, :])
            val.append(w[:, None] * g2)
        val = np.concatenate([v.reshape(-1) for v in val])
        col.add(lv["offset"] * nb, lv["size"] * nb, np.concatenate([i.reshape(-1) for i in idx]), val, np.abs(val))
    cg, ca, ck = (v.reshape(-1, nb) for v in (col.g, col.a, col.k))
    for i, li in enumerate(ti["lag"][0]):
        sl = (slice(None), slice(i * nb, (i + 1) * nb))
        acc.g.reshape(-1, FF)[sl] += li * cg
        acc.a.reshape(-1, FF)[sl] += abs(li) * ca
        acc.k.reshape(-1, FF)[sl] += ck * (li != 0)
    res["flow_grid"] = acc
    runs["flow_grid"] = np.stack(keys_runs)

    return dict(grads={k: (a.g, a.a, a.k) for k, a in res.items()}, dflow=dfl, dflow_abs=dfl_abs, live=live,
                flow_live=flive, runs=runs)
