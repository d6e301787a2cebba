"""Every kernel variant of the ray-marching and compositing operators, on both sides of each size switch.

csrc/raymarching.cu picks among several kernels per operator, by batch size and by the options `march_mode`,
`composite_mode` and `composite_bwd_mode`.  The variants promise the same bits: the marchers bit-exact against the C
oracle, the compositing kernels bit-identical to each other (each lane runs the reference's per-sample operation
sequence in every regime) and within the exp-rounding tolerance of the oracle.  These tests hold every variant to that,
at the sizes where the dispatch switches and at the places where the kernels hand work over: the phase-1 stash
(kStash = 16 samples) and the marcher that resumes behind it, the scan's 1024-entry chunks, the direct walk's
kDirect = 16 samples and the tile's 16-sample chunks.

The entry points are called through the C ABI with output buffers pre-filled with a NaN sentinel, so that a row a
kernel should leave alone, or one it forgets to write, shows up."""
import functools

import numpy as np
import pytest

import cases
from conftest import assert_bits_equal

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

S = cases.S
C, H, BOUND = S.CASCADE, S.GRID_SIZE, S.BOUND
LIDAR_FRAME = S.LIDAR_H * S.LIDAR_W     # 67 980 rays
SENTINEL = 0x7FA5A5A5                   # a NaN no kernel computes
T_TRAIN = 1e-4


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def filled(*shape, bits=SENTINEL):
    return torch.full(shape, bits, dtype=torch.int32, device="cuda").view(torch.float32)


def sentinel_rows(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32) == np.uint32(SENTINEL)


def rel_close(a, b, rtol=1e-5, atol=1e-7, what=""):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    err = np.abs(a - b)
    tol = atol + rtol * np.maximum(np.abs(a), np.abs(b))
    assert (err <= tol).all(), f"{what}: max err {np.nanmax(err):.3e}, {int((~(err <= tol)).sum())} elements out"


def _oracle():
    from oracle import raymarching_oracle
    return raymarching_oracle


# ====================================================================== march_rays_train
# N: both sides of the count pass's 32-ray / kRayBlock switch (16 384), of the write pass's coop<32> / coop<128>
# switch (kSmallMarch = 75 776), the full LiDAR frame, and 131 073 rays = 1025 count CTAs, one past the scan's chunk.
MARCH_SIZES = (16384, 16385, LIDAR_FRAME, 75776, 75777, 131073)
# (kind, fill, perturb, dt_gamma, max_steps).  With max_steps 8 / 16 / 17 rays end below, exactly at and one past the
# kStash samples phase 1 keeps: dt_min > dt_max there, every step is dt_max and grazing camera rays hit the cap.
MARCH_SETTINGS = (
    ("lidar", "shell", True, S.DT_GAMMA, 1024),
    ("camera", "random5", False, 0.0, 1024),
    ("camera", "random5", True, S.DT_GAMMA, 8),
    ("camera", "shell", False, 0.0, 16),
    ("camera", "shell", True, S.DT_GAMMA, 17),
)
MARCH_PAD = 45      # rows past the last sample: zeroed when zero_tail_end covers them, left alone when it does not


def _march_id(N, si, mode):
    kind, fill, perturb, dt_gamma, max_steps = MARCH_SETTINGS[si]
    kind = "lidar" if N == LIDAR_FRAME else kind
    return (f"march_mode{mode}-N{N}-{kind}-{fill}-steps{max_steps}-{'perturb' if perturb else 'noperturb'}-"
            f"dtgamma{'0' if dt_gamma == 0 else 'S'}")


# the two modes of one case run back to back, so one oracle result is cached at a time
MARCH_CASES = [(N, si, mode) for N in MARCH_SIZES for si in range(len(MARCH_SETTINGS)) for mode in (1, 0)]


@functools.lru_cache(maxsize=1)
def _march_case(N, si):
    kind, fill, perturb, dt_gamma, max_steps = MARCH_SETTINGS[si]
    if N == LIDAR_FRAME:
        o, d, nears, fars, noises = cases.march_inputs("lidar", -1, seed=60 + si, perturb=perturb)
    else:
        o, d, nears, fars, noises = cases.march_inputs(kind, N, seed=60 + si, perturb=perturb)
    assert o.shape[0] == N
    bf = cases.bitfield(fill, seed=2)
    O = _oracle()
    args = (o, d, BOUND, bf, C, H, nears, fars, noises)
    m = int(O.march_rays_train(*args, dt_gamma=dt_gamma, max_steps=max_steps, M=1)[4][0])   # counts only
    ex, ed, el, er, ec = O.march_rays_train(*args, dt_gamma=dt_gamma, max_steps=max_steps, M=m)
    assert ec.tolist() == [m, N]
    return dict(o=o, d=d, nears=nears, fars=fars, noises=noises, bf=bf, m=m, xyzs=ex, dirs=ed, deltas=el, rays=er,
                dt_gamma=dt_gamma, max_steps=max_steps)


def _truncated(c, Mt):
    """The oracle's result for a buffer of Mt rows: rays that do not fit are dropped and their rows stay zero."""
    out = [c["xyzs"][:Mt].copy(), c["dirs"][:Mt].copy(), c["deltas"][:Mt].copy()]
    off, cnt = c["rays"][:, 1].astype(np.int64), c["rays"][:, 2].astype(np.int64)
    for r in np.nonzero((off < Mt) & (off + cnt > Mt))[0]:
        for a in out:
            a[off[r]:Mt] = 0
    return out


@pytest.mark.parametrize("N,si,mode", MARCH_CASES, ids=[_march_id(*c) for c in MARCH_CASES])
def test_march_rays_train_variants(pkg, N, si, mode):
    """Count pass, then the write pass through `_write_ws` (stash resume) and `_write` (full walk), with zeroed and
    with untouched tails, a `mean_count`-style truncated buffer, and the one-call `nvsf_march_rays_train`: every
    output bit for bit against the C oracle under march_mode 0 (serial) and 1 (warp-cooperative)."""
    L, check, ptr = pkg._lib.lib(), pkg._lib.check, pkg._lib.ptr
    c = _march_case(N, si)
    m = c["m"]
    o, d, bf, nears, fars, noises = (dev(c[k]) for k in ("o", "d", "bf", "nears", "fars", "noises"))
    ws_bytes = L.nvsf_march_rays_train_workspace_bytes(N)
    work = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    geom = (ptr(o), ptr(d), ptr(bf), BOUND, c["dt_gamma"], c["max_steps"], N, C, H)
    st = pkg._lib.stream_ptr()
    exp = (c["xyzs"], c["dirs"], c["deltas"])
    names = ("xyzs", "dirs", "deltas")

    with pkg._lib.option_scope({"march_mode": mode}):
        rays = torch.full((N, 3), -7, dtype=torch.int32, device="cuda")
        counter = torch.zeros(2, dtype=torch.int32, device="cuda")
        check(L.nvsf_march_rays_train_count(*geom, ptr(nears), ptr(fars), ptr(rays), ptr(counter), ptr(noises),
                                            ptr(work), ws_bytes, st), "count")
        assert host(counter).tolist() == [m, N]
        assert_bits_equal(host(rays), c["rays"], "rays")

        def write(M, with_stash, zero_tail_end):
            out = (filled(M, 3), filled(M, 3), filled(M, 2))
            tail = (ptr(nears), ptr(fars)) + tuple(ptr(t) for t in out) + (ptr(rays), ptr(counter), ptr(noises),
                                                                          zero_tail_end)
            if with_stash:
                check(L.nvsf_march_rays_train_write_ws(*geom, M, *tail, ptr(work), ws_bytes, st), "write_ws")
            else:
                check(L.nvsf_march_rays_train_write(*geom, M, *tail, st), "write")
            return [host(t) for t in out]

        # the whole buffer and MARCH_PAD rows more, zeroed up to zero_tail_end = M
        M = m + MARCH_PAD
        for with_stash in (True, False):
            got = write(M, with_stash, M)
            for g, e, name in zip(got, exp, names):
                assert_bits_equal(g[:m], e, f"{name} ({'stash resume' if with_stash else 'full walk'})")
                assert not g[m:].any(), f"{name}: tail rows not zeroed"
        # the same buffer without zero_tail_end: the rows behind the last sample keep what was there
        got = write(M, True, 0)
        for g, e, name in zip(got, exp, names):
            assert_bits_equal(g[:m], e, f"{name} (no tail zeroing)")
            assert sentinel_rows(g[m:]).all(), f"{name}: rows past the last sample were written"

        # mean_count-style truncation: the buffer ends one sample into a ray near the middle
        cnt = c["rays"][:, 2]
        long_rays = np.nonzero(cnt >= 2)[0]
        if long_rays.size:
            r = long_rays[long_rays.size // 2]
            Mt = int(c["rays"][r, 1]) + 1
            exp_t = _truncated(c, Mt)
            for with_stash in (True, False):
                got = write(Mt, with_stash, Mt)
                for g, e, name in zip(got, exp_t, names):
                    assert_bits_equal(g, e, f"{name} truncated to {Mt} of {m} rows "
                                            f"({'stash resume' if with_stash else 'full walk'})")

    # the one-call entry point (zero_tail_end = 0): caller-sized buffer, a fresh counter
    with pkg._lib.option_scope({"march_mode": mode}):
        rays2 = torch.full((N, 3), -7, dtype=torch.int32, device="cuda")
        counter2 = torch.zeros(2, dtype=torch.int32, device="cuda")
        out = (filled(M, 3), filled(M, 3), filled(M, 2))
        check(L.nvsf_march_rays_train(*geom, M, ptr(nears), ptr(fars), *(ptr(t) for t in out), ptr(rays2),
                                      ptr(counter2), ptr(noises), ptr(work), ws_bytes, st), "march_rays_train")
        assert host(counter2).tolist() == [m, N]
        assert_bits_equal(host(rays2), c["rays"], "rays (one call)")
        for t, e, name in zip(out, exp, names):
            g = host(t)
            assert_bits_equal(g[:m], e, f"{name} (one call)")
            assert sentinel_rows(g[m:]).all(), f"{name} (one call): rows past the last sample were written"


# ====================================================================== composite_rays_train
# around the 32 768-ray switch of both compositing entry points, and ray counts that are no multiple of 32 / 64 / 128
COMP_SIZES = (1000, 4096, 32768, 32769, 40000)


@functools.lru_cache(maxsize=2)
def _comp_case(N):
    c = cases.composite_table(N, seed=N)
    rng = np.random.default_rng(N)
    c["g_ws"] = rng.normal(size=N).astype(np.float32)
    c["g_img"] = rng.normal(size=(N, 3)).astype(np.float32)
    c["fwd"] = _oracle().composite_rays_train_forward(c["sigmas"], c["rgbs"], c["deltas"], c["rays"], T_TRAIN)
    return c


def _composite_forward(pkg, c, mode, t):
    L, ptr = pkg._lib.lib(), pkg._lib.ptr
    N, M = c["rays"].shape[0], c["M"]
    out = (filled(N), filled(N), filled(N, 3))
    with pkg._lib.option_scope({"composite_mode": mode}):
        pkg._lib.check(L.nvsf_composite_rays_train_forward(ptr(t["sigmas"]), ptr(t["rgbs"]), ptr(t["deltas"]),
                                                           ptr(t["rays"]), M, N, T_TRAIN, *(ptr(x) for x in out),
                                                           pkg._lib.stream_ptr()), "composite forward")
    return out


def _composite_backward(pkg, c, mode, t, fwd, fill):
    L, ptr = pkg._lib.lib(), pkg._lib.ptr
    N, M = c["rays"].shape[0], c["M"]
    gs = torch.zeros(M, device="cuda") if fill == 0 else filled(M)
    gr = torch.zeros(M, 3, device="cuda") if fill == 0 else filled(M, 3)
    ws, _, image = fwd
    with pkg._lib.option_scope({"composite_bwd_mode": mode}):
        pkg._lib.check(L.nvsf_composite_rays_train_backward(
            ptr(t["g_ws"]), ptr(t["g_img"]), ptr(t["sigmas"]), ptr(t["rgbs"]), ptr(t["deltas"]), ptr(t["rays"]),
            ptr(ws), ptr(image), M, N, T_TRAIN, ptr(gs), ptr(gr), pkg._lib.stream_ptr()), "composite backward")
    return host(gs), host(gr)


def _device(c):
    return {k: dev(c[k]) for k in ("sigmas", "rgbs", "deltas", "rays", "g_ws", "g_img")}


@pytest.mark.parametrize("mode", [0, 1, 2], ids=["composite_mode0", "composite_mode1", "composite_mode2"])
@pytest.mark.parametrize("N", COMP_SIZES)       # the modes of one table run back to back (cached)
def test_composite_rays_train_forward_variants(pkg, mode, N):
    """Tile (0), direct prologue + tile (1) and direct (2) forward: bit-identical to mode 2, within 1e-5 of the
    oracle, and exactly 0 for rays with no sample or past the end of the buffer."""
    c = _comp_case(N)
    t = _device(c)
    got = [host(x) for x in _composite_forward(pkg, c, mode, t)]
    ref = [host(x) for x in _composite_forward(pkg, c, 2, t)]
    for g, r, e, name in zip(got, ref, c["fwd"], ("weights_sum", "depth", "image")):
        assert_bits_equal(g, r, f"{name}: composite_mode {mode} vs 2")
        rel_close(g, e, what=f"{name} vs oracle")
        assert not g[c["dead"]].any(), f"{name}: a ray with no sample or past M composited something"
    # every ray terminated on purpose composited up to its termination point: T reached 0 or 6e-6 there
    placed = (c["term"] >= 0) & ~c["dead"]
    assert (got[0][placed] > 1 - 1e-5).all()


@pytest.mark.parametrize("mode", [0, 1, 2], ids=["composite_bwd_mode0", "composite_bwd_mode1", "composite_bwd_mode2"])
@pytest.mark.parametrize("N", COMP_SIZES)       # the modes of one table run back to back (cached)
def test_composite_rays_train_backward_variants(pkg, mode, N):
    """Tile (0), hybrid (1) and the size-picked default (2) backward: bit-identical to mode 2, from zeroed and from
    NaN-filled gradient buffers, against the oracle with the tolerances of test_composite_rays_train_forward_backward;
    exactly the samples up to each ray's termination point are written."""
    c = _comp_case(N)
    t = _device(c)
    fwd = _composite_forward(pkg, c, 2, t)
    zs, zr = _composite_backward(pkg, c, mode, t, fwd, 0)
    ns, nr = _composite_backward(pkg, c, mode, t, fwd, SENTINEL)
    rzs, rzr = _composite_backward(pkg, c, 2, t, fwd, 0)
    rns, rnr = _composite_backward(pkg, c, 2, t, fwd, SENTINEL)
    assert_bits_equal(zs, rzs, f"grad_sigmas: composite_bwd_mode {mode} vs 2")
    assert_bits_equal(zr, rzr, f"grad_rgbs: composite_bwd_mode {mode} vs 2")
    assert_bits_equal(ns, rns, f"grad_sigmas (NaN-filled): composite_bwd_mode {mode} vs 2")
    assert_bits_equal(nr, rnr, f"grad_rgbs (NaN-filled): composite_bwd_mode {mode} vs 2")
    # see test_composite_rays_train_forward_backward: alpha's exp differs by ~2^-22 absolute from the oracle's
    egs, egr = _oracle().composite_rays_train_backward(c["g_ws"], c["g_img"], c["sigmas"], c["rgbs"], c["deltas"],
                                                      c["rays"], host(fwd[0]), host(fwd[2]), T_TRAIN)
    rel_close(zs, egs, rtol=2e-5, atol=2e-5, what="grad_sigmas vs oracle")
    rel_close(zr, egr, rtol=1e-5, atol=5e-6, what="grad_rgbs vs oracle")
    w, owned = c["written"], c["owned"]
    after = owned & ~w
    assert after.any() and (~owned).any()
    assert not zs[after].any() and not zr[after].any(), "gradient written after a ray's termination point"
    assert sentinel_rows(ns[after]).all() and sentinel_rows(nr[after]).all(), "write after the termination point"
    assert sentinel_rows(ns[~owned]).all() and sentinel_rows(nr[~owned]).all(), \
        "write to a gap row, or to a ray with no sample or past M"
    assert not zs[~owned].any() and not zr[~owned].any()
    assert_bits_equal(ns[w], zs[w], "grad_sigmas: NaN-filled vs zeroed buffers")
    assert_bits_equal(nr[w], zr[w], "grad_rgbs: NaN-filled vs zeroed buffers")


# ====================================================================== inference pair
INF_ALIVE = (3000, 75777, 100003)
INF_STEPS = (1, 17, 33)
INF_CASES = [(n, s, mode) for n in INF_ALIVE for s in INF_STEPS for mode in (1, 0)]
INF_PAD = 77


@functools.lru_cache(maxsize=1)
def _inference_case(n_alive, n_step):
    R = n_alive + 4099                      # alive rays are a shuffled subset of R rays
    o, d, nears, fars, _ = cases.march_inputs("lidar", R, seed=70 + n_step, perturb=False)
    rng = np.random.default_rng(n_alive + n_step)
    alive = rng.permutation(R)[:n_alive].astype(np.int32)
    # half the rays start at near, the rest part-way along (later iterations of the run_cuda loop)
    rays_t = np.where(rng.random(R) < 0.5, nears, nears + rng.random(R, dtype=np.float32) * (fars - nears) * 0.6)
    rays_t = rays_t.astype(np.float32)
    noises = rng.random(n_alive, dtype=np.float32)
    bf = cases.bitfield("random5" if n_step == 17 else "shell", seed=4)
    M = n_alive * n_step + INF_PAD
    ex, ed, el = _oracle().march_rays(n_alive, n_step, alive, rays_t, o, d, BOUND, bf, C, H, nears, fars, noises,
                                     dt_gamma=S.DT_GAMMA, M=M)
    return dict(o=o, d=d, nears=nears, fars=fars, alive=alive, rays_t=rays_t, noises=noises, bf=bf, M=M,
                out=(ex, ed, el))


@pytest.mark.parametrize("n_alive,n_step,mode", INF_CASES,
                         ids=[f"march_mode{m}-n_alive{n}-n_step{s}" for n, s, m in INF_CASES])
def test_march_rays_variants(pkg, n_alive, n_step, mode):
    """Inference marcher, serial (march_mode 0) and warp-cooperative at 32- and 128-ray CTAs (1): every row of the
    M_padded buffer bit for bit against the oracle, unused slots and the padded tail included."""
    L, ptr = pkg._lib.lib(), pkg._lib.ptr
    c = _inference_case(n_alive, n_step)
    M = c["M"]
    t = {k: dev(c[k]) for k in ("o", "d", "nears", "fars", "alive", "rays_t", "noises", "bf")}
    out = (filled(M, 3), filled(M, 3), filled(M, 2))
    with pkg._lib.option_scope({"march_mode": mode}):
        pkg._lib.check(L.nvsf_march_rays(n_alive, n_step, ptr(t["alive"]), ptr(t["rays_t"]), ptr(t["o"]), ptr(t["d"]),
                                         BOUND, S.DT_GAMMA, 1024, C, H, ptr(t["bf"]), ptr(t["nears"]), ptr(t["fars"]),
                                         *(ptr(x) for x in out), ptr(t["noises"]), M, pkg._lib.stream_ptr()),
                       "march_rays")
    for x, e, name in zip(out, c["out"], ("xyzs", "dirs", "deltas")):
        assert_bits_equal(host(x), e, name)
    assert c["out"][2][:n_alive * n_step, 0].any() and not c["out"][2][:n_alive * n_step, 0].all()


@pytest.mark.parametrize("n_step", [17, 33])
def test_composite_rays_inference_vs_oracle(pkg, n_step):
    """In-place inference compositing over more samples than the kernel stages at once (16): rays stop at a zero
    delta or after a sample with alpha = 1 on both sides of the chunk boundaries; alive flags and rays_t exact, the
    accumulators within 1e-5 of the oracle, rays that are not alive untouched."""
    n_alive, R = 5001, 6007
    rng = np.random.default_rng(80 + n_step)
    alive = rng.permutation(R)[:n_alive].astype(np.int32)
    rays_t = rng.uniform(0.1, 1.0, R).astype(np.float32)
    # rays part-way through: accumulated values well above the ~1e-7 absolute exp difference against the oracle;
    # sigma*delta in [0.02, 0.06] keeps every weights_sum below 0.93, far from 1 - T_thresh, without a placed stop
    ws = rng.uniform(0.1, 0.5, R).astype(np.float32)
    depth = rng.uniform(0.2, 1.0, R).astype(np.float32)
    image = rng.uniform(0.1, 0.5, (R, 3)).astype(np.float32)
    rgb = rng.random((n_alive, n_step, 3), dtype=np.float32)
    dl = np.float32(1e-3) + rng.random((n_alive, n_step, 2), dtype=np.float32) * np.float32(9e-3)
    sig = (rng.uniform(0.02, 0.06, (n_alive, n_step)) / dl[..., 0]).astype(np.float32)
    edges = [k for k in (0, 1, 15, 16, 17, 31, 32) if k < n_step]
    for n in range(n_alive):
        k = edges[n % len(edges)]
        if n % 3 == 0:          # the marcher ran out of samples: zero deltas from slot k on
            dl[n, k:] = 0
            sig[n, k:] = np.nan
            rgb[n, k:] = np.nan
        elif n % 3 == 1:        # alpha = 1 at slot k: slot k + 1 is composited with T = 0, nothing after it
            sig[n, k] = 1e5
            sig[n, k + 2:] = np.nan
            rgb[n, k + 2:] = np.nan
            dl[n, k + 2:] = np.nan
    sig, rgb, dl = sig.reshape(-1), rgb.reshape(-1, 3), dl.reshape(-1, 2)
    e_alive, e_t, e_ws, e_depth, e_image = _oracle().composite_rays(n_alive, n_step, alive, rays_t, sig, rgb, dl, ws,
                                                                   depth, image, 1e-2)
    g = {k: dev(v) for k, v in dict(alive=alive, rays_t=rays_t, ws=ws, depth=depth, image=image).items()}
    pkg.raymarching.composite_rays(n_alive, n_step, g["alive"], g["rays_t"], dev(sig), dev(rgb), dev(dl), g["ws"],
                                   g["depth"], g["image"], 1e-2)
    assert np.array_equal(host(g["alive"]), e_alive)
    assert (e_alive < 0).sum() > n_alive // 2 and (e_alive >= 0).any()
    assert_bits_equal(host(g["rays_t"]), e_t, "rays_t")
    rel_close(host(g["ws"]), e_ws, what="weights_sum")
    rel_close(host(g["depth"]), e_depth, what="depth")
    rel_close(host(g["image"]), e_image, what="image")
    untouched = np.setdiff1d(np.arange(R), alive)
    assert_bits_equal(host(g["ws"])[untouched], ws[untouched], "weights_sum of rays that are not alive")
