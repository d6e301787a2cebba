// nvsf_b200 — Chamfer distance between two point clouds, forward and backward (sm_100a).
//
// Replaces the reference's second native extension (nvsf/nerf/chamfer3D/chamfer3D.cu:9-150
// NmDistanceKernel, :151-195 NmDistanceGradKernel; wrapper dist_chamfer_3D.py:42-95), which
// train_step calls on the predicted vs ground-truth LiDAR points (trainer.py:229-233) and on the
// flow-warped point clouds (:246-265).  Same results: dist[j] = min_k |p_j - q_k|^2 evaluated as
// the reference build evaluates it (x*x + y*y + z*z contracted to FMUL(y) + two FMAs), idx[j] = the first k
// that attains it (the reference scans k ascending with a strict `<`).
//
// The reference launches a fixed 32 x 16 grid of 512-thread CTAs in which blockIdx.x walks the
// batch: for the trainer's single batch of 4096 points 8 CTAs do all the work, each thread scanning
// the whole target cloud.  Here the (query block, target range) plane is tiled over all SMs:
// a CTA owns 512 queries (two per thread) and one range of targets, staged through shared memory
// in SoA tiles read as broadcasts; partial minima meet in one 64-bit atomicMin per query on the
// key (float bits of the distance << 32 | index) — distances are non-negative, so integer order is
// (distance, index) order and the result is the reference's first-minimum, deterministically.
#include <algorithm>
#include <cmath>
#include <string>

#include "common.cuh"

namespace {

constexpr int kChThreads = 256;
constexpr int kChQueries = 2 * kChThreads;   // per CTA
constexpr int kChTile = 1024;                // target points per shared-memory tile

// a point count kept in device memory, clamped to [0, capacity]
__device__ __forceinline__ uint32_t device_count(const int32_t* __restrict__ c, uint32_t cap) {
    return (uint32_t)min(max(__ldg(c), 0), (int32_t)cap);
}

// One CTA's share of the nearest-neighbour scan: queries q[blockIdx.x * kChQueries ...] against targets
// [blockIdx.y * per_split, +per_split) of t, folded into keys[j] with atomicMin.
__device__ __forceinline__ void chamfer_nn_tile(const float* __restrict__ q, uint32_t n, const float* __restrict__ t,
                                                uint32_t m, uint32_t per_split, unsigned long long* __restrict__ kb) {
    __shared__ float sx[kChTile], sy[kChTile], sz[kChTile];
    const uint32_t j0 = blockIdx.x * kChQueries + threadIdx.x, j1 = j0 + kChThreads;
    float x0 = 0.f, y0 = 0.f, z0 = 0.f, x1 = 0.f, y1 = 0.f, z1 = 0.f;
    if (j0 < n) { x0 = __ldg(q + 3 * (size_t)j0); y0 = __ldg(q + 3 * (size_t)j0 + 1); z0 = __ldg(q + 3 * (size_t)j0 + 2); }
    if (j1 < n) { x1 = __ldg(q + 3 * (size_t)j1); y1 = __ldg(q + 3 * (size_t)j1 + 1); z1 = __ldg(q + 3 * (size_t)j1 + 2); }
    float best0 = INFINITY, best1 = INFINITY;
    uint32_t bi0 = 0, bi1 = 0;
    const uint32_t k_begin = blockIdx.y * per_split, k_end = min(m, k_begin + per_split);
    for (uint32_t k2 = k_begin; k2 < k_end; k2 += kChTile) {
        const uint32_t cnt = min((uint32_t)kChTile, k_end - k2);
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < cnt; i += kChThreads) {
            sx[i] = __ldg(t + 3 * (size_t)(k2 + i));
            sy[i] = __ldg(t + 3 * (size_t)(k2 + i) + 1);
            sz[i] = __ldg(t + 3 * (size_t)(k2 + i) + 2);
        }
        __syncthreads();
#pragma unroll 4
        for (uint32_t k = 0; k < cnt; ++k) {
            const float tx = sx[k], ty = sy[k], tz = sz[k];
            // chamfer3D.cu:38-42: d = x2*x2 + y2*y2 + z2*z2 with x2 = buf - x1; nvcc contracts it to
            // fma(z2, z2, fma(x2, x2, y2*y2)) (sm_100a SASS of the reference kernel: FMUL on the y term,
            // then FFMA x, FFMA z; confirmed bit for bit against the extension's outputs)
            const float ax = tx - x0, ay = ty - y0, az = tz - z0;
            const float d0 = __fmaf_rn(az, az, __fmaf_rn(ax, ax, __fmul_rn(ay, ay)));
            const float bx = tx - x1, by = ty - y1, bz = tz - z1;
            const float d1 = __fmaf_rn(bz, bz, __fmaf_rn(bx, bx, __fmul_rn(by, by)));
            if (d0 < best0) { best0 = d0; bi0 = k2 + k; }
            if (d1 < best1) { best1 = d1; bi1 = k2 + k; }
        }
    }
    if (k_begin < k_end) {
        if (j0 < n) atomicMin(kb + j0, ((unsigned long long)__float_as_uint(best0) << 32) | bi0);
        if (j1 < n) atomicMin(kb + j1, ((unsigned long long)__float_as_uint(best1) << 32) | bi1);
    }
}

__global__ void __launch_bounds__(kChThreads)
k_chamfer_nn(const float* __restrict__ xyz, uint32_t n, const float* __restrict__ xyz2, uint32_t m,
             uint32_t per_split, unsigned long long* __restrict__ keys) {
    const uint32_t b = blockIdx.z;
    chamfer_nn_tile(xyz + (size_t)b * n * 3, n, xyz2 + (size_t)b * m * 3, m, per_split, keys + (size_t)b * n);
}

// The same scan with the cloud sizes read from device memory (clouds padded to a capacity; the grid is laid
// out for the capacities and CTAs past the counts return at once).
__global__ void __launch_bounds__(kChThreads)
k_chamfer_nn_counted(const float* __restrict__ xyz, uint32_t cap_n, const int32_t* __restrict__ n_dev,
                     const float* __restrict__ xyz2, uint32_t cap_m, const int32_t* __restrict__ m_dev,
                     uint32_t per_split, unsigned long long* __restrict__ keys) {
    const uint32_t n = device_count(n_dev, cap_n), m = device_count(m_dev, cap_m);
    if (blockIdx.x * kChQueries >= n || blockIdx.y * per_split >= m) return;
    chamfer_nn_tile(xyz, n, xyz2, m, per_split, keys);
}

// keys [c1 | c2] -> (dist1, idx1) and (dist2, idx2) in one launch
__global__ void k_chamfer_unpack(const unsigned long long* __restrict__ keys, size_t c1, size_t c2,
                                 float* __restrict__ dist1, int32_t* __restrict__ idx1,
                                 float* __restrict__ dist2, int32_t* __restrict__ idx2) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= c1 + c2) return;
    const unsigned long long k = keys[i];
    const float d = __uint_as_float((uint32_t)(k >> 32));
    const int32_t id = (int32_t)(uint32_t)k;
    if (i < c1) { dist1[i] = d; idx1[i] = id; }
    else { dist2[i - c1] = d; idx2[i - c1] = id; }
}

// keys [cap_n | cap_m] -> dist / idx of the counted forward.  A query whose target cloud is empty keeps the
// all-ones key and gets +inf / -1; rows past a count get 0 / -1.
__global__ void k_chamfer_unpack_counted(const unsigned long long* __restrict__ keys, uint32_t cap_n, uint32_t cap_m,
                                         const int32_t* __restrict__ n_dev, const int32_t* __restrict__ m_dev,
                                         float* __restrict__ dist1, int32_t* __restrict__ idx1,
                                         float* __restrict__ dist2, int32_t* __restrict__ idx2) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)cap_n + cap_m) return;
    const bool first = i < cap_n;
    const uint32_t r = first ? (uint32_t)i : (uint32_t)(i - cap_n);
    const uint32_t cnt = first ? device_count(n_dev, cap_n) : device_count(m_dev, cap_m);
    float d = 0.f;
    int32_t id = -1;
    if (r < cnt) {
        const unsigned long long k = keys[i];
        if (k == ~0ull) {
            d = INFINITY;
        } else {
            d = __uint_as_float((uint32_t)(k >> 32));
            id = (int32_t)(uint32_t)k;
        }
    }
    if (first) { dist1[r] = d; idx1[r] = id; }
    else { dist2[r] = d; idx2[r] = id; }
}

// chamfer3D.cu:151-178: g = 2 * grad_dist[j]; grad_a[j] += g (a_j - b_idx); grad_b[idx] -= g (a_j - b_idx)
__global__ void __launch_bounds__(256)
k_chamfer_grad(const float* __restrict__ a, uint32_t n, const float* __restrict__ bpts, uint32_t m,
               const float* __restrict__ gdist, const int32_t* __restrict__ idx,
               float* __restrict__ ga, float* __restrict__ gb) {
    const uint32_t b = blockIdx.y;
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const size_t ja = (size_t)b * n + j;
    const int32_t j2 = __ldg(idx + ja);
    const size_t jb = (size_t)b * m + (uint32_t)j2;
    const float g = __ldg(gdist + ja) * 2.f;
    const float dx = g * (__ldg(a + 3 * ja) - __ldg(bpts + 3 * jb));
    const float dy = g * (__ldg(a + 3 * ja + 1) - __ldg(bpts + 3 * jb + 1));
    const float dz = g * (__ldg(a + 3 * ja + 2) - __ldg(bpts + 3 * jb + 2));
    if (ga) {   // each (b, j) is visited once per direction: plain adds would do, but the two
                // directions of one backward run on the same stream into the same buffers
        atomicAdd(ga + 3 * ja, dx); atomicAdd(ga + 3 * ja + 1, dy); atomicAdd(ga + 3 * ja + 2, dz);
    }
    if (gb) {
        atomicAdd(gb + 3 * jb, -dx); atomicAdd(gb + 3 * jb + 1, -dy); atomicAdd(gb + 3 * jb + 2, -dz);
    }
}

// grid (query blocks, target ranges) of one scan direction
struct NnGrid {
    uint32_t qblocks, splits, per_split;
};

NnGrid nn_grid(uint32_t n, uint32_t m, uint32_t b, int sms) {
    const uint32_t qblocks = nvsf_div_up(n, (uint32_t)kChQueries);
    // enough target ranges to put ~2 CTAs on every SM; ranges are multiples of 128 targets (the trainer's single
    // batch of 4096 x 4096 points became 8 x 4 = 32 CTAs with whole 1024-target tiles: 0.33 ms against the
    // reference extension's 0.25 ms; 8 x 32 CTAs now)
    const uint32_t gran = 128;
    uint32_t splits = std::max(1u, std::min(nvsf_div_up(m, gran), (2u * (uint32_t)sms) / std::max(1u, qblocks * b)));
    const uint32_t per_split = nvsf_div_up(nvsf_div_up(m, splits), gran) * gran;
    splits = nvsf_div_up(m, per_split);
    return {qblocks, splits, per_split};
}

void launch_nn(const float* q, uint32_t n, const float* t, uint32_t m, uint32_t b,
               unsigned long long* keys, int sms, cudaStream_t s) {
    const NnGrid g = nn_grid(n, m, b, sms);
    k_chamfer_nn<<<dim3(g.qblocks, g.splits, b), kChThreads, 0, s>>>(q, n, t, m, g.per_split, keys);
}

int sm_count() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

// ============================================================================ uniform-grid nearest neighbours
// The same (distance, index) keys as the scan above, found by visiting a uniform grid over the target cloud ring
// by ring (Chebyshev shells around the query's home cell) until no unvisited target can reach the current best.
// Exactness argument and measurements: DESIGN.md §3.5.  Per cloud and batch element, with no host read:
//   k_grid_bbox    box of the finite points (order-preserving uint32 keys, integer atomicMin)
//   k_grid_setup   cell size and per-axis dimensions from the box (<= the cell budget from the host size)
//   k_grid_count   cell of every point (non-finite points: one bucket past the last cell) + slot in its cell
//   k_grid_tiles / k_grid_top / k_grid_starts   exclusive scan of the cell counts (tile sums, tile offsets, cells)
//   k_grid_scatter SoA coordinates + original index in cell order
// Then k_grid_nn runs one thread per query, the queries taken in their own cloud's cell order, so a warp's
// candidate loads come from neighbouring cells.  A query whose search outgrows max(kGridMinWork, m / 8) cells and
// candidates (one far outside a fine grid, where every target is about equally far) is listed for
// k_grid_nn_left, where a whole CTA scans every target for it.  A target cloud whose points crowd a few cells (sum of the
// squared cell counts above m^2 / kGridCrowd) is scanned by the brute-force tiles instead, gated on the device.
constexpr int kGridCellsPerPoint = 2;          // cell budget per point of the target cloud
constexpr uint32_t kGridMaxCells = 1u << 27;
constexpr double kGridCrowd = 32.0;
constexpr int kGridBlock = 256;
constexpr int kGridTile = 2048;                // cell counts per scan tile (8 per thread)
constexpr int kGridNnBlock = 128;
constexpr uint32_t kGridMinWork = 4096;        // per-query work (cells + candidates) before k_grid_nn_left takes over
constexpr int kGridLeftBlock = 256;
constexpr uint32_t kGridLeftCtas = 2 * 148;
constexpr unsigned long long kInfKey = 0x7f800000ull << 32;   // (+inf, 0): no finite distance

struct GridParams {
    double lo[3], hi[3];   // box of the finite points
    double mu[3];          // face margin (DESIGN.md §3.5)
    double h, inv_h;       // cell size
    uint32_t dims[3];
    uint32_t cells;        // dims[0] * dims[1] * dims[2]; bucket `cells` holds the non-finite points
    uint32_t count;        // points in the cloud
    uint32_t fallback;     // 1: searched by the brute-force scan
};

// one cloud's grid; arrays are [b][...] with the strides below
struct GridBufs {
    uint32_t* bbox;                  // [b][8]: min key x, y, z, ~max key x, y, z (all-ones = empty)
    unsigned long long* sumsq;       // [b]: sum of squared cell counts
    uint32_t* left_count;            // [b]: queries handed to k_grid_nn_left (this cloud's queries)
    uint32_t* left;                  // [b][cap]: their positions in cell order
    uint32_t* counts;                // [b][budget + 1]
    GridParams* params;              // [b]
    uint32_t* tiles;                 // [b][ntiles]
    uint32_t* start;                 // [b][budget + 2]
    uint32_t *cell, *slot;           // [b][cap]
    float4* sp;                      // [b][cap]: x, y, z, original index (bits) in cell order
    uint32_t cap, budget, ntiles;
    const int32_t* count_dev;        // counted form: device count (NULL: cap)
};

uint32_t grid_budget(uint32_t m) {
    return (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, (uint64_t)m * kGridCellsPerPoint), kGridMaxCells);
}

__device__ __forceinline__ uint32_t f2key(float f) {   // float order == uint32 order
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__device__ __forceinline__ uint32_t grid_count(const GridBufs& g) {
    return g.count_dev ? device_count(g.count_dev, g.cap) : g.cap;
}

__device__ __forceinline__ bool finite3(float x, float y, float z) {
    return isfinite(x) && isfinite(y) && isfinite(z);
}

__global__ void __launch_bounds__(kGridBlock)
k_grid_bbox(const float* __restrict__ xyz, GridBufs g) {
    const uint32_t b = blockIdx.y, n = grid_count(g);
    const float* p = xyz + (size_t)b * g.cap * 3;
    uint32_t k[6] = {~0u, ~0u, ~0u, ~0u, ~0u, ~0u};
    for (uint32_t i = blockIdx.x * kGridBlock + threadIdx.x; i < n; i += gridDim.x * kGridBlock) {
        const float x = __ldg(p + 3 * (size_t)i), y = __ldg(p + 3 * (size_t)i + 1), z = __ldg(p + 3 * (size_t)i + 2);
        if (!finite3(x, y, z)) continue;
        k[0] = min(k[0], f2key(x)); k[1] = min(k[1], f2key(y)); k[2] = min(k[2], f2key(z));
        k[3] = min(k[3], ~f2key(x)); k[4] = min(k[4], ~f2key(y)); k[5] = min(k[5], ~f2key(z));
    }
#pragma unroll
    for (int a = 0; a < 6; ++a) {
        const uint32_t v = __reduce_min_sync(0xffffffffu, k[a]);
        if ((threadIdx.x & 31) == 0 && v != ~0u) atomicMin(g.bbox + (size_t)b * 8 + a, v);
    }
}

// number of cells of size h over extents e (each axis at least one cell), saturating above `cap`
__device__ __forceinline__ double cells_for(const double e[3], double h, uint32_t d[3]) {
    double c = 1.0;
    for (int a = 0; a < 3; ++a) {
        const double n = fmax(1.0, ceil(e[a] / h));
        d[a] = n < 4294967295.0 ? (uint32_t)n : 4294967295u;
        c *= n;
    }
    return c;
}

__global__ void k_grid_setup(GridBufs g, uint32_t batch) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    const uint32_t n = grid_count(g);
    GridParams P;
    const uint32_t* k = g.bbox + (size_t)b * 8;
    const bool empty = k[0] == ~0u;   // no finite point
    double e[3], emax = 0.0;
    for (int a = 0; a < 3; ++a) {
        P.lo[a] = empty ? 0.0 : (double)key2f(k[a]);
        P.hi[a] = empty ? 0.0 : (double)key2f(~k[3 + a]);
        e[a] = P.hi[a] - P.lo[a];
        emax = fmax(emax, e[a]);
    }
    const double budget = fmin((double)g.budget, fmax(1.0, (double)n * kGridCellsPerPoint));
    double h = 1.0;
    if (emax > 0.0) {
        // smallest h (within 2^-40 relative) with at most `budget` cells: cells_for decreases with h; at h = emax
        // there is one cell per axis
        double lo = emax / budget, hi = emax;
        uint32_t d[3];
        for (int it = 0; it < 64 && hi > lo * (1.0 + 0x1p-40); ++it) {
            const double mid = sqrt(lo) * sqrt(hi);
            if (cells_for(e, mid, d) <= budget) hi = mid; else lo = mid;
        }
        h = hi;
    }
    P.h = h;
    P.inv_h = 1.0 / h;
    cells_for(e, h, P.dims);
    P.cells = P.dims[0] * P.dims[1] * P.dims[2];
    for (int a = 0; a < 3; ++a) P.mu[a] = 0x1p-40 * (fabs(P.lo[a]) + fabs(P.hi[a]) + h);
    P.count = n;
    P.fallback = 0;
    g.params[b] = P;
}

// home cell of a point: clamped into the grid, so points outside the box (queries) land in a boundary cell
__device__ __forceinline__ uint32_t axis_cell(float v, const GridParams& P, int a) {
    const double t = fmin(fmax(((double)v - P.lo[a]) * P.inv_h, 0.0), (double)(P.dims[a] - 1));
    return (uint32_t)t;
}

__global__ void __launch_bounds__(kGridBlock)
k_grid_count(const float* __restrict__ xyz, GridBufs g) {
    const uint32_t b = blockIdx.y, i = blockIdx.x * kGridBlock + threadIdx.x;
    const GridParams& P = g.params[b];
    if (i >= P.count) return;
    const float* p = xyz + ((size_t)b * g.cap + i) * 3;
    const float x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
    uint32_t c = P.cells;
    if (finite3(x, y, z))
        c = (axis_cell(z, P, 2) * P.dims[1] + axis_cell(y, P, 1)) * P.dims[0] + axis_cell(x, P, 0);
    const size_t o = (size_t)b * g.cap + i;
    g.cell[o] = c;
    g.slot[o] = atomicAdd(g.counts + (size_t)b * (g.budget + 1) + c, 1u);
}

// per tile of kGridTile counts: its sum, and the sum of squared cell counts into sumsq
__global__ void __launch_bounds__(kGridBlock)
k_grid_tiles(GridBufs g) {
    __shared__ uint32_t red[kGridBlock / 32];
    const uint32_t b = blockIdx.y, cells = g.params[b].cells;
    const uint32_t* cnt = g.counts + (size_t)b * (g.budget + 1);
    const uint32_t base = blockIdx.x * kGridTile, end = min(base + kGridTile, g.budget + 1);
    uint32_t s = 0;
    unsigned long long sq = 0;
    for (uint32_t i = base + threadIdx.x; i < end; i += kGridBlock) {
        const uint32_t c = cnt[i];
        s += c;
        if (i < cells) sq += (unsigned long long)c * c;
    }
    s = warp_reduce_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, d);
    if ((threadIdx.x & 31) == 0 && sq) atomicAdd(g.sumsq + b, sq);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < kGridBlock / 32; ++w) t += red[w];
        g.tiles[(size_t)b * g.ntiles + blockIdx.x] = t;
    }
}

// tile sums -> exclusive tile offsets (one CTA per batch element); the crowding test sets `fallback`
__global__ void __launch_bounds__(kGridBlock)
k_grid_top(GridBufs g) {
    __shared__ uint32_t warp_tot[kGridBlock / 32];
    __shared__ uint32_t carry;
    const uint32_t b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* t = g.tiles + (size_t)b * g.ntiles;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < g.ntiles; base += kGridBlock) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < g.ntiles ? t[i] : 0u;
        const uint32_t inc = warp_inclusive_scan(v, lane);
        if (lane == 31) warp_tot[warp] = inc;
        __syncthreads();
        uint32_t before = carry;
        for (uint32_t w = 0; w < warp; ++w) before += warp_tot[w];
        if (i < g.ntiles) t[i] = before + inc - v;
        __syncthreads();
        if (threadIdx.x == kGridBlock - 1) carry = before + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double n = (double)g.params[b].count;
        g.params[b].fallback = (double)g.sumsq[b] * kGridCrowd > n * n ? 1u : 0u;
    }
}

// start[i] = sum of counts[0, i) for i <= budget, start[budget + 1] = every point
__global__ void __launch_bounds__(kGridBlock)
k_grid_starts(GridBufs g) {
    __shared__ uint32_t warp_tot[kGridBlock / 32];
    constexpr int kPer = kGridTile / kGridBlock;
    const uint32_t b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t* cnt = g.counts + (size_t)b * (g.budget + 1);
    uint32_t* st = g.start + (size_t)b * (g.budget + 2);
    const uint32_t n = g.budget + 1, i0 = blockIdx.x * kGridTile + threadIdx.x * kPer;
    uint32_t c[kPer], s = 0;
#pragma unroll
    for (int j = 0; j < kPer; ++j) { c[j] = i0 + j < n ? cnt[i0 + j] : 0u; s += c[j]; }
    const uint32_t inc = warp_inclusive_scan(s, lane);
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    uint32_t run = g.tiles[(size_t)b * g.ntiles + blockIdx.x] + inc - s;
    for (uint32_t w = 0; w < warp; ++w) run += warp_tot[w];
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
        if (i0 + j < n) st[i0 + j] = run;
        run += c[j];
        if (i0 + j == n - 1) st[n] = run;
    }
}

__global__ void __launch_bounds__(kGridBlock)
k_grid_scatter(const float* __restrict__ xyz, GridBufs g) {
    const uint32_t b = blockIdx.y, i = blockIdx.x * kGridBlock + threadIdx.x;
    if (i >= g.params[b].count) return;
    const size_t o = (size_t)b * g.cap + i;
    const size_t pos = (size_t)b * g.cap + g.start[(size_t)b * (g.budget + 2) + g.cell[o]] + g.slot[o];
    const float* p = xyz + o * 3;
    g.sp[pos] = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __uint_as_float(i));
}

void build_grid(const float* xyz, const GridBufs& g, uint32_t b, cudaStream_t s) {
    const uint32_t pblocks = nvsf_div_up(g.cap, (uint32_t)kGridBlock);
    k_grid_bbox<<<dim3(std::min(pblocks, 256u), b), kGridBlock, 0, s>>>(xyz, g);
    k_grid_setup<<<nvsf_div_up(b, 32u), 32, 0, s>>>(g, b);
    k_grid_count<<<dim3(pblocks, b), kGridBlock, 0, s>>>(xyz, g);
    k_grid_tiles<<<dim3(g.ntiles, b), kGridBlock, 0, s>>>(g);
    k_grid_top<<<b, kGridBlock, 0, s>>>(g);
    k_grid_starts<<<dim3(g.ntiles, b), kGridBlock, 0, s>>>(g);
    k_grid_scatter<<<dim3(pblocks, b), kGridBlock, 0, s>>>(xyz, g);
}

// distance from v to [a, b] (0 inside)
__device__ __forceinline__ double gap(double v, double a, double b) { return fmax(fmax(a - v, v - b), 0.0); }

// squared distance from q to the box's slabs below cell b0 and above cell b1 of one axis (the sides not on the
// grid boundary), `others` = squared gaps on the other two axes; lowers `bound`
__device__ __forceinline__ void slab_bound(double q, double lo, double hi, double mu, double h, int b0, int b1,
                                           int dim, double others, double& bound, bool& open) {
    if (b0 > 0) {
        const double t = gap(q, lo, lo + b0 * h + mu);
        bound = fmin(bound, others + t * t);
        open = true;
    }
    if (b1 < dim - 1) {
        const double t = gap(q, lo + (b1 + 1) * h - mu, hi);
        bound = fmin(bound, others + t * t);
        open = true;
    }
}

// candidate keys of the sorted targets [s, e) against q, folded into best
__device__ __forceinline__ void grid_scan(const float4* __restrict__ sp, uint32_t s, uint32_t e, float qx, float qy,
                                          float qz, unsigned long long& best) {
    for (uint32_t k = s; k < e; ++k) {
        const float4 t = __ldg(sp + k);
        // the brute-force expression exactly (k_chamfer_nn): target minus query, fma(z, z, fma(x, x, y * y))
        const float ax = __fsub_rn(t.x, qx), ay = __fsub_rn(t.y, qy), az = __fsub_rn(t.z, qz);
        const float d = __fmaf_rn(az, az, __fmaf_rn(ax, ax, __fmul_rn(ay, ay)));
        const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | __float_as_uint(t.w);
        best = key < best ? key : best;   // +inf and NaN keys never beat the initial (+inf, 0)
    }
}

// One thread per query of cloud Q (in Q's cell order) against the grid of cloud T; writes keys[b][original index].
__global__ void __launch_bounds__(kGridNnBlock, 6)   // 80 registers, no spills
k_grid_nn(GridBufs Q, GridBufs T, uint32_t key_stride, unsigned long long* __restrict__ keys) {
    const uint32_t b = blockIdx.y, i = blockIdx.x * kGridNnBlock + threadIdx.x;
    const GridParams& P = T.params[b];
    if (P.fallback || P.count == 0 || i >= Q.params[b].count) return;   // brute-force scan / empty target (+inf, -1)
    const size_t qo = (size_t)b * Q.cap + i;
    const float4 qp = Q.sp[qo];
    const uint32_t orig = __float_as_uint(qp.w);
    if (i >= Q.start[(size_t)b * (Q.budget + 2) + Q.params[b].cells]) {   // non-finite query: no finite distance
        keys[(size_t)b * key_stride + orig] = kInfKey;
        return;
    }
    const float qx = qp.x, qy = qp.y, qz = qp.z;
    const float4* sp = T.sp + (size_t)b * T.cap;
    const uint32_t max_work = max(kGridMinWork, P.count / 8);
    uint32_t work = 0;
    const uint32_t* st = T.start + (size_t)b * (T.budget + 2);
    const int nx = (int)P.dims[0], ny = (int)P.dims[1], nz = (int)P.dims[2];
    const int cx = (int)axis_cell(qx, P, 0), cy = (int)axis_cell(qy, P, 1), cz = (int)axis_cell(qz, P, 2);
    unsigned long long best = kInfKey;
    for (int r = 0;; ++r) {
        const int x0 = max(cx - r, 0), x1 = min(cx + r, nx - 1), y0 = max(cy - r, 0), y1 = min(cy + r, ny - 1),
                  z0 = max(cz - r, 0), z1 = min(cz + r, nz - 1);
        for (int z = z0; z <= z1; ++z) {
            const bool zface = z == cz - r || z == cz + r;
            for (int y = y0; y <= y1; ++y) {
                const uint32_t row = ((uint32_t)z * ny + y) * nx;
                if (zface || y == cy - r || y == cy + r) {
                    const uint32_t s0 = st[row + x0], s1 = st[row + x1 + 1];
                    grid_scan(sp, s0, s1, qx, qy, qz, best);
                    work += (uint32_t)(x1 - x0 + 1) + (s1 - s0);
                } else {
                    work += 2;
                    if (cx - r >= 0) grid_scan(sp, st[row + cx - r], st[row + cx - r + 1], qx, qy, qz, best);
                    if (cx + r < nx) grid_scan(sp, st[row + cx + r], st[row + cx + r + 1], qx, qy, qz, best);
                }
            }
        }
        // lower bound on the true distance of every unvisited target: an unvisited target lies in one of the
        // slabs of the box beyond a face of the visited block that is not a grid boundary; each face is moved
        // outwards by mu (cell assignment rounding)
        // (the box parameters are re-read from L1 every ring rather than held in registers across the scans)
        const double gx = gap(qx, P.lo[0], P.hi[0]), gy = gap(qy, P.lo[1], P.hi[1]), gz = gap(qz, P.lo[2], P.hi[2]);
        double bound = INFINITY;
        bool open = false;
        slab_bound(qx, P.lo[0], P.hi[0], P.mu[0], P.h, x0, x1, nx, gy * gy + gz * gz, bound, open);
        slab_bound(qy, P.lo[1], P.hi[1], P.mu[1], P.h, y0, y1, ny, gx * gx + gz * gz, bound, open);
        slab_bound(qz, P.lo[2], P.hi[2], P.mu[2], P.h, z0, z1, nz, gx * gx + gy * gy, bound, open);
        if (!open) break;
        // the computed fp32 distance is at least (1 - 5 * 2^-24) of the true one, less ~5 * 2^-150 of underflow
        if (bound * (1.0 - 0x1p-20) - 0x1p-140 > (double)__uint_as_float((uint32_t)(best >> 32))) break;
        if (work > max_work) {   // far from where the targets are dense: an exhaustive scan by a whole CTA
            Q.left[(size_t)b * Q.cap + atomicAdd(Q.left_count + b, 1u)] = i;
            return;
        }
    }
    keys[(size_t)b * key_stride + orig] = best;
}

// The queries k_grid_nn listed: one CTA per query scans every finite target of T (the grid order holds them all).
__global__ void __launch_bounds__(kGridLeftBlock)
k_grid_nn_left(GridBufs Q, GridBufs T, uint32_t key_stride, unsigned long long* __restrict__ keys) {
    __shared__ unsigned long long red[kGridLeftBlock / 32];
    const uint32_t b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t nleft = Q.left_count[b];
    if (blockIdx.x >= nleft) return;
    const uint32_t nfin = T.start[(size_t)b * (T.budget + 2) + T.params[b].cells];
    const float4* sp = T.sp + (size_t)b * T.cap;
    for (uint32_t j = blockIdx.x; j < nleft; j += gridDim.x) {
        const float4 qp = Q.sp[(size_t)b * Q.cap + Q.left[(size_t)b * Q.cap + j]];
        unsigned long long best = kInfKey;
        for (uint32_t k = threadIdx.x; k < nfin; k += kGridLeftBlock) grid_scan(sp, k, k + 1, qp.x, qp.y, qp.z, best);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, d);
            best = o < best ? o : best;
        }
        if (lane == 0) red[warp] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kGridLeftBlock / 32; ++w) best = red[w] < best ? red[w] : best;
            keys[(size_t)b * key_stride + __float_as_uint(qp.w)] = best;
        }
        __syncthreads();
    }
}

// the brute-force scan for the batch elements whose target grid is crowded
__global__ void __launch_bounds__(kChThreads)
k_chamfer_nn_crowded(const float* __restrict__ xyz, uint32_t n, const float* __restrict__ xyz2, uint32_t m,
                     uint32_t per_split, unsigned long long* __restrict__ keys, const GridParams* __restrict__ tp) {
    const uint32_t b = blockIdx.z;
    if (!tp[b].fallback) return;
    chamfer_nn_tile(xyz + (size_t)b * n * 3, n, xyz2 + (size_t)b * m * 3, m, per_split, keys + (size_t)b * n);
}

__global__ void __launch_bounds__(kChThreads)
k_chamfer_nn_counted_crowded(const float* __restrict__ xyz, uint32_t cap_n, const int32_t* __restrict__ n_dev,
                             const float* __restrict__ xyz2, uint32_t cap_m, const int32_t* __restrict__ m_dev,
                             uint32_t per_split, unsigned long long* __restrict__ keys,
                             const GridParams* __restrict__ tp) {
    if (!tp->fallback) return;
    const uint32_t n = device_count(n_dev, cap_n), m = device_count(m_dev, cap_m);
    if (blockIdx.x * kChQueries >= n || blockIdx.y * per_split >= m) return;
    chamfer_nn_tile(xyz, n, xyz2, m, per_split, keys);
}

// ---- workspace: [keys | bbox 1 | bbox 2] (0xFF) [counts 1 | sumsq 1 | counts 2 | sumsq 2] (0) [the rest]
constexpr size_t kWsAlign = 16;

struct WsCarve {
    size_t off = 0;
    size_t take(size_t bytes) {
        const size_t at = off;
        off = nvsf_div_up(off + bytes, kWsAlign) * kWsAlign;
        return at;
    }
};

struct GridOffs {
    size_t bbox, counts, sumsq, left_count, left, params, tiles, start, cell, slot, sp;
};

struct ChamferWs {
    size_t keys_end, ff_end, zero_begin, zero_end, bytes;
    GridOffs g[2];
    uint32_t cap[2];
};

uint32_t grid_tiles(uint32_t cap) { return nvsf_div_up(grid_budget(cap) + 1, (uint32_t)kGridTile); }

ChamferWs chamfer_ws(uint32_t b, uint32_t n, uint32_t m) {
    WsCarve c;
    ChamferWs w;
    w.cap[0] = n;
    w.cap[1] = m;
    c.take((size_t)b * ((size_t)n + m) * sizeof(unsigned long long));
    w.keys_end = c.off;
    for (int k = 0; k < 2; ++k) w.g[k].bbox = c.take((size_t)b * 8 * sizeof(uint32_t));
    w.ff_end = c.off;
    w.zero_begin = c.off;
    for (int k = 0; k < 2; ++k) {
        w.g[k].counts = c.take((size_t)b * (grid_budget(w.cap[k]) + 1) * sizeof(uint32_t));
        w.g[k].sumsq = c.take((size_t)b * sizeof(unsigned long long));
        w.g[k].left_count = c.take((size_t)b * sizeof(uint32_t));
    }
    w.zero_end = c.off;
    for (int k = 0; k < 2; ++k) {
        const size_t pts = (size_t)b * w.cap[k];
        w.g[k].params = c.take((size_t)b * sizeof(GridParams));
        w.g[k].tiles = c.take((size_t)b * grid_tiles(w.cap[k]) * sizeof(uint32_t));
        w.g[k].start = c.take((size_t)b * (grid_budget(w.cap[k]) + 2) * sizeof(uint32_t));
        w.g[k].left = c.take(pts * sizeof(uint32_t));
        w.g[k].cell = c.take(pts * sizeof(uint32_t));
        w.g[k].slot = c.take(pts * sizeof(uint32_t));
        w.g[k].sp = c.take(pts * sizeof(float4));
    }
    w.bytes = c.off;
    return w;
}

GridBufs grid_bufs(const ChamferWs& w, int k, void* ws, const int32_t* count_dev) {
    char* base = reinterpret_cast<char*>(ws);
    const GridOffs& o = w.g[k];
    GridBufs g;
    g.bbox = reinterpret_cast<uint32_t*>(base + o.bbox);
    g.sumsq = reinterpret_cast<unsigned long long*>(base + o.sumsq);
    g.left_count = reinterpret_cast<uint32_t*>(base + o.left_count);
    g.left = reinterpret_cast<uint32_t*>(base + o.left);
    g.counts = reinterpret_cast<uint32_t*>(base + o.counts);
    g.params = reinterpret_cast<GridParams*>(base + o.params);
    g.tiles = reinterpret_cast<uint32_t*>(base + o.tiles);
    g.start = reinterpret_cast<uint32_t*>(base + o.start);
    g.cell = reinterpret_cast<uint32_t*>(base + o.cell);
    g.slot = reinterpret_cast<uint32_t*>(base + o.slot);
    g.sp = reinterpret_cast<float4*>(base + o.sp);
    g.cap = w.cap[k];
    g.budget = grid_budget(g.cap);
    g.ntiles = grid_tiles(g.cap);
    g.count_dev = count_dev;
    return g;
}

// ---- path selection
// "chamfer_grid": -1 automatic (grid from kGridMinPairs query-target pairs per batch element), 0 never, 1 always
constexpr uint64_t kGridMinPairs = 1ull << 28;
int g_chamfer_grid = -1;

// (the grid path reads float4 rows: it needs the 16-byte alignment every CUDA allocator gives)
bool use_grid(uint32_t b, uint64_t n, uint64_t m, const void* ws) {
    if (g_chamfer_grid == 0 || b > 65535u || (reinterpret_cast<uintptr_t>(ws) & (kWsAlign - 1))) return false;
    return g_chamfer_grid == 1 || n * m >= kGridMinPairs;
}

// Both directions through the grids: memsets, two grid builds, two searches, the gated brute-force scans.
int grid_forward(const float* xyz1, const float* xyz2, uint32_t b, uint32_t n, uint32_t m, const int32_t* n_dev,
                 const int32_t* m_dev, void* workspace, int sms, cudaStream_t s) {
    const ChamferWs w = chamfer_ws(b, n, m);
    char* base = reinterpret_cast<char*>(workspace);
    cudaError_t e = cudaMemsetAsync(base, 0xff, w.ff_end, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(base + w.zero_begin, 0, w.zero_end - w.zero_begin, s);
    if (e != cudaSuccess) return (int)e;
    unsigned long long* k1 = reinterpret_cast<unsigned long long*>(workspace);
    unsigned long long* k2 = k1 + (size_t)b * n;
    const GridBufs g1 = grid_bufs(w, 0, workspace, n_dev), g2 = grid_bufs(w, 1, workspace, m_dev);
    build_grid(xyz1, g1, b, s);
    build_grid(xyz2, g2, b, s);
    k_grid_nn<<<dim3(nvsf_div_up(n, (uint32_t)kGridNnBlock), b), kGridNnBlock, 0, s>>>(g1, g2, n, k1);
    k_grid_nn<<<dim3(nvsf_div_up(m, (uint32_t)kGridNnBlock), b), kGridNnBlock, 0, s>>>(g2, g1, m, k2);
    const uint32_t left_ctas = std::max(1u, kGridLeftCtas / b);
    k_grid_nn_left<<<dim3(left_ctas, b), kGridLeftBlock, 0, s>>>(g1, g2, n, k1);
    k_grid_nn_left<<<dim3(left_ctas, b), kGridLeftBlock, 0, s>>>(g2, g1, m, k2);
    const NnGrid a = nn_grid(n, m, b, sms), c = nn_grid(m, n, b, sms);
    if (n_dev) {
        k_chamfer_nn_counted_crowded<<<dim3(a.qblocks, a.splits), kChThreads, 0, s>>>(xyz1, n, n_dev, xyz2, m, m_dev,
                                                                                     a.per_split, k1, g2.params);
        k_chamfer_nn_counted_crowded<<<dim3(c.qblocks, c.splits), kChThreads, 0, s>>>(xyz2, m, m_dev, xyz1, n, n_dev,
                                                                                     c.per_split, k2, g1.params);
    } else {
        k_chamfer_nn_crowded<<<dim3(a.qblocks, a.splits, b), kChThreads, 0, s>>>(xyz1, n, xyz2, m, a.per_split, k1,
                                                                                g2.params);
        k_chamfer_nn_crowded<<<dim3(c.qblocks, c.splits, b), kChThreads, 0, s>>>(xyz2, m, xyz1, n, c.per_split, k2,
                                                                                g1.params);
    }
    return NVSF_OK;
}

}  // namespace

int nvsf_chamfer_set_option(const char* name, int value) {
    if (std::string(name) == "chamfer_grid") {
        if (value < -1 || value > 1) return NVSF_E_INVALID;
        g_chamfer_grid = value;
        return NVSF_OK;
    }
    return NVSF_E_INVALID;
}
int nvsf_chamfer_get_option(const char* name) {
    if (std::string(name) == "chamfer_grid") return g_chamfer_grid;
    return NVSF_E_INVALID;
}

extern "C" {

// enough for either path: the keys of the brute-force scan come first, the grids follow
size_t nvsf_chamfer_workspace_bytes(uint32_t b, uint32_t n, uint32_t m) { return chamfer_ws(b, n, m).bytes; }

int nvsf_chamfer_forward(const float* xyz1, const float* xyz2, uint32_t b, uint32_t n, uint32_t m,
                         float* dist1, float* dist2, int32_t* idx1, int32_t* idx2, void* workspace,
                         size_t workspace_bytes, void* stream) {
    if (b == 0 || (n == 0 && m == 0)) return NVSF_OK;
    if (n == 0 || m == 0) return NVSF_E_INVALID;   // a nearest neighbour needs a non-empty target
    if (!xyz1 || !xyz2 || !dist1 || !dist2 || !idx1 || !idx2 || !workspace) return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_chamfer_workspace_bytes(b, n, m)) return NVSF_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    const int sms = sm_count();
    unsigned long long* k1 = reinterpret_cast<unsigned long long*>(workspace);
    unsigned long long* k2 = k1 + (size_t)b * n;
    if (use_grid(b, n, m, workspace)) {
        const int st = grid_forward(xyz1, xyz2, b, n, m, nullptr, nullptr, workspace, sms, s);
        if (st != NVSF_OK) return st;
    } else {
        cudaMemsetAsync(workspace, 0xff, (size_t)b * ((size_t)n + m) * sizeof(unsigned long long), s);
        launch_nn(xyz1, n, xyz2, m, b, k1, sms, s);
        launch_nn(xyz2, m, xyz1, n, b, k2, sms, s);
    }
    const size_t c1 = (size_t)b * n, c2 = (size_t)b * m;
    k_chamfer_unpack<<<(unsigned)nvsf_div_up(c1 + c2, (size_t)256), 256, 0, s>>>(k1, c1, c2, dist1, idx1, dist2,
                                                                              idx2);
    return nvsf_launch_status();
}

int nvsf_chamfer_forward_counted(const float* xyz1, const float* xyz2, uint32_t cap_n, uint32_t cap_m,
                                 const int32_t* n, const int32_t* m, float* dist1, float* dist2, int32_t* idx1,
                                 int32_t* idx2, void* workspace, size_t workspace_bytes, void* stream) {
    if (cap_n == 0 || cap_m == 0 || cap_n > INT32_MAX || cap_m > INT32_MAX) return NVSF_E_INVALID;
    if (!xyz1 || !xyz2 || !n || !m || !dist1 || !dist2 || !idx1 || !idx2 || !workspace) return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_chamfer_workspace_bytes(1, cap_n, cap_m)) return NVSF_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    const int sms = sm_count();
    unsigned long long* k1 = reinterpret_cast<unsigned long long*>(workspace);
    unsigned long long* k2 = k1 + cap_n;
    if (use_grid(1, cap_n, cap_m, workspace)) {
        const int st = grid_forward(xyz1, xyz2, 1, cap_n, cap_m, n, m, workspace, sms, s);
        if (st != NVSF_OK) return st;
    } else {
        cudaMemsetAsync(workspace, 0xff, ((size_t)cap_n + cap_m) * sizeof(unsigned long long), s);
        const NnGrid g1 = nn_grid(cap_n, cap_m, 1, sms), g2 = nn_grid(cap_m, cap_n, 1, sms);
        k_chamfer_nn_counted<<<dim3(g1.qblocks, g1.splits), kChThreads, 0, s>>>(xyz1, cap_n, n, xyz2, cap_m, m,
                                                                               g1.per_split, k1);
        k_chamfer_nn_counted<<<dim3(g2.qblocks, g2.splits), kChThreads, 0, s>>>(xyz2, cap_m, m, xyz1, cap_n, n,
                                                                               g2.per_split, k2);
    }
    k_chamfer_unpack_counted<<<(unsigned)nvsf_div_up((size_t)cap_n + cap_m, (size_t)256), 256, 0, s>>>(
        k1, cap_n, cap_m, n, m, dist1, idx1, dist2, idx2);
    return nvsf_launch_status();
}

int nvsf_chamfer_backward(const float* xyz1, const float* xyz2, uint32_t b, uint32_t n, uint32_t m,
                          const float* grad_dist1, const float* grad_dist2, const int32_t* idx1,
                          const int32_t* idx2, float* grad_xyz1, float* grad_xyz2, void* stream) {
    if (b == 0 || n == 0 || m == 0) return NVSF_OK;
    if (!xyz1 || !xyz2 || !grad_dist1 || !grad_dist2 || !idx1 || !idx2 || (!grad_xyz1 && !grad_xyz2))
        return NVSF_E_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    k_chamfer_grad<<<dim3(nvsf_div_up(n, 256u), b), 256, 0, s>>>(xyz1, n, xyz2, m, grad_dist1, idx1, grad_xyz1,
                                                               grad_xyz2);
    k_chamfer_grad<<<dim3(nvsf_div_up(m, 256u), b), 256, 0, s>>>(xyz2, m, xyz1, n, grad_dist2, idx2, grad_xyz2,
                                                               grad_xyz1);
    return nvsf_launch_status();
}

}  // extern "C"
