// nvsf_b200 — the callers either side of the marcher (SURVEY.md §8f ranks 1 and 2), sm_100a:
//
//  * ray generation: get_lidar_rays / get_rays (reference nvsf/nerf/dataset/dataset_utils.py
//    :369-536 and :539-687) — origins and directions are pure functions of (pose, pixel id,
//    intrinsics), so a frame's rays are generated on the device instead of being built by ~20
//    ATen launches and copied;
//  * occupancy ("density") grid maintenance that produces the bitfield march_rays_train /
//    march_rays consume.  The reference ships only the primitives (morton3D, packbits,
//    raymarching.py:85-164) and no update loop; the semantics here are those of the
//    update_extra_state routine of torch-ngp, the code base the reference's raymarching
//    extension was taken from: jittered cell-centre samples per cascade, sigma * density_scale,
//    grid = max(grid * decay, new) on valid cells, threshold = min(mean(clamp(grid, 0)),
//    density_thresh), packbits.  Mean, threshold and packing stay on the device (no host sync).
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "lidar_dir.cuh"
#include "radix_select.cuh"

namespace {

// ---------------------------------------------------------------------------------- ray generation
struct Pose {
    float r[3][3];
    float t[3];
};

__device__ __forceinline__ Pose load_pose(const float* __restrict__ pose) {
    Pose P;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b = 0; b < 3; ++b) P.r[a][b] = __ldg(pose + a * 4 + b);
        P.t[a] = __ldg(pose + a * 4 + 3);
    }
    return P;
}

// rays_d = directions @ R^T, evaluated left to right without FMA contraction like a plain
// fp32 dot product; rays_o = translation column.
__device__ __forceinline__ void emit_ray(const Pose& P, float x, float y, float z, size_t k,
                                         float* __restrict__ rays_o, float* __restrict__ rays_d) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float v = __fadd_rn(__fadd_rn(__fmul_rn(x, P.r[a][0]), __fmul_rn(y, P.r[a][1])),
                                  __fmul_rn(z, P.r[a][2]));
        rays_d[k * 3 + a] = v;
        rays_o[k * 3 + a] = P.t[a];
    }
}

// direction of pixel id p = j*W + i: lidar_dir.cuh (dataset_utils.py:512-530)
__global__ void __launch_bounds__(256)
k_lidar_rays(const float* __restrict__ pose, const int64_t* __restrict__ inds, uint32_t n,
             uint32_t H, uint32_t W, float fov_up, float fov, float fov_hoz,
             float* __restrict__ rays_o, float* __restrict__ rays_d) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const Pose P = load_pose(pose);
    const int64_t p = inds ? inds[k] : (int64_t)k;
    float x, y, z;
    lidar_dir(p, H, W, fov_up, fov, fov_hoz, x, y, z);
    emit_ray(P, x, y, z, k, rays_o, rays_d);
}

// dataset_utils.py:563-681: xs = (i + 0.5 - cx)/fx, ys = (j + 0.5 - cy)/fy, zs = 1, normalised.
__global__ void __launch_bounds__(256)
k_camera_rays(const float* __restrict__ pose, const int64_t* __restrict__ inds, uint32_t n,
              uint32_t H, uint32_t W, float fx, float fy, float cx, float cy,
              float* __restrict__ rays_o, float* __restrict__ rays_d) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const Pose P = load_pose(pose);
    const int64_t p = inds ? inds[k] : (int64_t)k;
    const float i = (float)(p % W) + 0.5f, j = (float)(p / W) + 0.5f;
    const float xs = __fdiv_rn(__fsub_rn(i, cx), fx), ys = __fdiv_rn(__fsub_rn(j, cy), fy);
    const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(xs, xs), __fmul_rn(ys, ys)), 1.0f));
    emit_ray(P, __fdiv_rn(xs, nrm), __fdiv_rn(ys, nrm), __fdiv_rn(1.0f, nrm), k, rays_o, rays_d);
}

// ------------------------------------------------------------------------------- error-map sampling
// torch-ngp's error-map branch of get_rays: N distinct coarse cells of a res x res map drawn with
// probability proportional to the map (torch.multinomial without replacement), then one jittered pixel
// inside each cell.  Exponential race: the N smallest keys E_i / w_i are such a draw.  Cells with
// w <= 0 or non-finite w get the key E_i with the sign bit set, so as unsigned integers they order after
// every positive-weight key: the N smallest keys are then the positive cells' draw, filled when there are
// fewer than N positive cells by the smallest E among the rest.  One CTA per map holds the R = res^2 keys
// in shared memory, radix-selects the N-th smallest and compacts the selected cells in ascending cell
// order (ties at the N-th key go to the lower cells).
constexpr int kEmBlock = 1024;

// Exclusive count of `flag` over the CTA in thread order; *total = the CTA's count.  `warp_off` holds
// kEmBlock / 32 + 1 words of shared memory.
__device__ __forceinline__ uint32_t block_exclusive_count(bool flag, uint32_t* warp_off, uint32_t& total) {
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t bal = __ballot_sync(0xffffffffu, flag);
    __syncthreads();  // `warp_off` may still be read from the previous call
    if (lane == 0) warp_off[warp] = __popc(bal);
    __syncthreads();
    if (tid < 32) {
        const uint32_t c = warp_off[tid];
        const uint32_t inc = warp_inclusive_scan(c, lane);
        warp_off[tid] = inc - c;
        if (tid == 31) warp_off[kEmBlock / 32] = inc;
    }
    __syncthreads();
    total = warp_off[kEmBlock / 32];
    return warp_off[warp] + __popc(bal & ((1u << lane) - 1u));
}

__global__ void __launch_bounds__(kEmBlock)
k_error_map_sample(const float* __restrict__ error_map, const float* __restrict__ expo,
                   const float* __restrict__ jitter, uint32_t res, uint32_t N, uint32_t H, uint32_t W,
                   int64_t* __restrict__ inds_coarse, int64_t* __restrict__ inds) {
    extern __shared__ uint32_t keys[];
    __shared__ uint32_t hist[256];
    __shared__ uint32_t warp_off[kEmBlock / 32 + 1];
    const uint32_t R = res * res, tid = threadIdx.x;
    for (uint32_t i = tid; i < R; i += kEmBlock) {
        const float w = __ldg(error_map + i), e = __ldg(expo + i);
        keys[i] = w > 0.f && w < INFINITY ? __float_as_uint(__fdiv_rn(e, w)) : 0x80000000u | __float_as_uint(e);
    }
    __syncthreads();
    uint32_t ties;
    const uint32_t T = radix_select<kEmBlock>([](uint32_t i) { return keys[i]; }, R, N - 1, hist, ties);
    // torch-ngp: row = (cr * sx + u0 * sx).long().clamp(max=H-1), sx = H / res in fp32; cols with W
    const float sx = (float)((double)H / (double)res), sy = (float)((double)W / (double)res);
    uint32_t tie_base = 0, out_base = 0;
    for (uint32_t c0 = 0; c0 < R && out_base < N; c0 += kEmBlock) {
        const uint32_t i = c0 + tid;
        const uint32_t u = i < R ? keys[i] : 0u;
        const bool tie = i < R && u == T;
        uint32_t n_tie, n_take;
        const uint32_t tie_rank = tie_base + block_exclusive_count(tie, warp_off, n_tie);
        const bool take = i < R && (u < T || (tie && tie_rank <= ties));
        const uint32_t j = out_base + block_exclusive_count(take, warp_off, n_take);
        if (take) {
            const float u0 = __ldg(jitter + 2 * (size_t)j), u1 = __ldg(jitter + 2 * (size_t)j + 1);
            const float r = __fadd_rn(__fmul_rn((float)(i / res), sx), __fmul_rn(u0, sx));
            const float c = __fadd_rn(__fmul_rn((float)(i % res), sy), __fmul_rn(u1, sy));
            const int64_t row = min((int64_t)r, (int64_t)H - 1), col = min((int64_t)c, (int64_t)W - 1);
            inds_coarse[j] = (int64_t)i;
            inds[j] = row * W + col;
        }
        tie_base += n_tie;
        out_base += n_take;
    }
}

// torch-ngp train_step: map[c_j] = 0.1 * map[c_j] + 0.9 * loss[j] over one batch row's distinct cells.
__global__ void __launch_bounds__(256)
k_error_map_update(float* __restrict__ error_map, uint32_t R, const int64_t* __restrict__ inds_coarse,
                   uint32_t N, const float* __restrict__ loss) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    const int64_t c = __ldg(inds_coarse + j);
    if (c < 0 || c >= (int64_t)R) return;  // never write outside the map
    error_map[c] = __fadd_rn(__fmul_rn(0.1f, error_map[c]), __fmul_rn(0.9f, __ldg(loss + j)));
}

// ---------------------------------------------------------------------------------- occupancy grid
__device__ __forceinline__ uint32_t compact_by3(uint32_t x) {  // raymarching.cu:83-90 inverse spread
    x &= 0x09249249u;
    x = (x ^ (x >> 2)) & 0x030c30c3u;
    x = (x ^ (x >> 4)) & 0x0300f00fu;
    x = (x ^ (x >> 8)) & 0xff0000ffu;
    x = (x ^ (x >> 16)) & 0x000003ffu;
    return x;
}

// Sample point of Morton cell m of cascade c: xyz = 2*coords/(H-1) - 1 in [-1,1], scaled to the
// cascade box shrunk by half a cell, plus a (noise*2-1)*half_cell jitter.  Output row c*H^3 + m,
// i.e. already in the [C, H^3] Morton layout of the density grid.
// `first` / `count` select a slice of the C*H^3 cells (multi-GPU update: each rank owns one slice);
// noise and xyz rows are relative to the slice.
// Sample point of cell g = c*H^3 + m; `noise` points at the cell's 3 jitter values or is NULL.
__device__ __forceinline__ void cell_point(size_t g, uint32_t H, float bound, const float* __restrict__ noise,
                                           float v[3]) {
    const uint32_t H3 = H * H * H;
    const uint32_t c = (uint32_t)(g / H3), m = (uint32_t)(g % H3);
    const float bc = fminf(exp2f((float)c), bound);
    const float half = __fdiv_rn(bc, (float)H);
    const float ext = __fsub_rn(bc, half);
    const uint32_t co[3] = {compact_by3(m), compact_by3(m >> 1), compact_by3(m >> 2)};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float u = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, (float)co[a]), (float)(H - 1)), 1.0f);
        v[a] = __fmul_rn(u, ext);
        if (noise) {
            const float j = __fsub_rn(__fmul_rn(__ldg(noise + a), 2.0f), 1.0f);
            v[a] = __fadd_rn(v[a], __fmul_rn(j, half));
        }
    }
}

__global__ void __launch_bounds__(256)
k_grid_cell_points(uint32_t C, uint32_t H, float bound, const float* __restrict__ noise,
                   float* __restrict__ xyz, size_t first, size_t count) {
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= count) return;
    float v[3];
    cell_point(first + r, H, bound, noise ? noise + r * 3 : nullptr, v);
#pragma unroll
    for (int a = 0; a < 3; ++a) xyz[r * 3 + a] = v[a];
}

// Sample points of the cells listed in cells[0, count) (ids c*H^3 + m; a negative id yields the origin).
// The jitter row of entry r is noise[cells[r]] when noise_by_cell, else noise[r].
__global__ void __launch_bounds__(256)
k_grid_cell_points_list(uint32_t H, float bound, const int32_t* __restrict__ cells, uint32_t count,
                        const float* __restrict__ noise, uint32_t noise_by_cell, float* __restrict__ xyz) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= count) return;
    const int32_t g = __ldg(cells + r);
    float v[3] = {0.f, 0.f, 0.f};
    if (g >= 0) cell_point((size_t)g, H, bound, noise ? noise + (size_t)(noise_by_cell ? (uint32_t)g : r) * 3 : nullptr,
                           v);
#pragma unroll
    for (int a = 0; a < 3; ++a) xyz[(size_t)r * 3 + a] = v[a];
}

// --------------------------------------------------------------------------- untrained-cell marking
// torch-ngp's mark_untrained_grid with the tests of DESIGN.md §3.5: a cell is covered by a pose when its
// un-jittered centre lies inside the sensor's field of view widened by the margin m = 2 b_c / H.  Every
// slope and edge normal is prepared on the host in float64 and rounded to fp32 once; the kernel only
// multiplies, adds and compares, each operation rounded on its own, so a numpy fp32 restatement gives
// the same bits.
constexpr uint32_t kCovPoses = 128;  // poses per launch, kept in shared memory (12 floats each)

struct Coverage {
    uint32_t lidar;  // 0: camera frustum, 1: LiDAR shell
    // camera: x-slopes (sl, sr), y-slopes (st, sb); LiDAR: range [near, far], elevation slopes (s_lo, s_up)
    float a0, a1, a2, a3;
    uint32_t wedge;  // LiDAR azimuth: 0 none (360 degrees), 1 intersection of the two half-planes, 2 union
    float n1x, n1y, n2x, n2y;
};

__device__ __forceinline__ bool covers(const Coverage& S, const float* P, const float x[3], float m) {
    // p = R^T (x - t): d_b = fl(x_b - t_b), p_a = fl(fl(fl(R[0][a] d_0) + fl(R[1][a] d_1)) + fl(R[2][a] d_2))
    const float d0 = __fsub_rn(x[0], P[3]), d1 = __fsub_rn(x[1], P[7]), d2 = __fsub_rn(x[2], P[11]);
    float p[3];
#pragma unroll
    for (int a = 0; a < 3; ++a)
        p[a] = __fadd_rn(__fadd_rn(__fmul_rn(P[a], d0), __fmul_rn(P[4 + a], d1)), __fmul_rn(P[8 + a], d2));
    if (!S.lidar) {
        if (!(p[2] > 0.f)) return false;
        if (!(p[0] > __fsub_rn(__fmul_rn(S.a0, p[2]), m) && p[0] < __fadd_rn(__fmul_rn(S.a1, p[2]), m))) return false;
        return p[1] > __fsub_rn(__fmul_rn(S.a2, p[2]), m) && p[1] < __fadd_rn(__fmul_rn(S.a3, p[2]), m);
    }
    const float xy = __fadd_rn(__fmul_rn(p[0], p[0]), __fmul_rn(p[1], p[1]));
    const float r = __fsqrt_rn(__fadd_rn(xy, __fmul_rn(p[2], p[2])));
    const float rho = __fsqrt_rn(xy);
    if (!(r > __fsub_rn(S.a0, m) && r < __fadd_rn(S.a1, m))) return false;
    if (!(p[2] > __fsub_rn(__fmul_rn(S.a2, rho), m) && p[2] < __fadd_rn(__fmul_rn(S.a3, rho), m))) return false;
    if (S.wedge == 0) return true;
    const bool in1 = __fadd_rn(__fmul_rn(S.n1x, p[0]), __fmul_rn(S.n1y, p[1])) > -m;
    const bool in2 = __fadd_rn(__fmul_rn(S.n2x, p[0]), __fmul_rn(S.n2y, p[1])) > -m;
    return S.wedge == 1 ? (in1 && in2) : (in1 || in2);
}

// One thread per cell; a warp owns one 32-bit word of the covered mask (bit i of byte k = cell 8k + i) and
// ORs its ballot into it.  Cells already covered skip the poses; a cell stops at its first covering pose.
__global__ void __launch_bounds__(256)
k_grid_coverage(uint32_t n, uint32_t H, float bound, const float* __restrict__ poses, uint32_t B, Coverage S,
                uint32_t* __restrict__ covered) {
    __shared__ float P[kCovPoses * 12];
    for (uint32_t i = threadIdx.x; i < B * 12; i += blockDim.x) P[i] = __ldg(poses + (i / 12) * 16 + i % 12);
    __syncthreads();
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;  // n is a multiple of 32: whole warps
    if (g >= n) return;
    const uint32_t lane = threadIdx.x & 31, word = covered[g >> 5];
    bool cov = (word >> lane) & 1u;
    if (!cov) {
        const uint32_t H3 = H * H * H;
        const float bc = fminf(exp2f((float)(g / H3)), bound);
        const float m = __fdiv_rn(__fmul_rn(2.0f, bc), (float)H);
        float x[3];
        cell_point(g, H, bound, nullptr, x);
        for (uint32_t b = 0; b < B && !cov; ++b) cov = covers(S, P + b * 12, x, m);
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, cov);
    if (lane == 0 && bal != word) covered[g >> 5] = bal;
}

// Applies the covered mask, one thread per mask byte (8 cells): uncovered cells get grid = -1 and their
// bitfield bit cleared; a covered cell that holds a mark from an earlier call is restored to 0.
// *n_marked (zeroed by the caller) receives the number of uncovered cells.
__global__ void __launch_bounds__(256)
k_grid_apply_marks(float* __restrict__ grid, uint8_t* __restrict__ bitfield, const uint8_t* __restrict__ covered,
                   uint32_t n_bytes, int32_t* __restrict__ n_marked) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t marked = 0;
    if (b < n_bytes) {
        const uint32_t cov = covered[b];
        marked = 8u - __popc(cov);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float* g = grid + (size_t)b * 8 + i;
            if (!((cov >> i) & 1u)) *g = -1.f;
            else if (*g < 0.f) *g = 0.f;
        }
        bitfield[b] &= (uint8_t)cov;
    }
    marked = warp_reduce_sum(marked);
    if ((threadIdx.x & 31) == 0 && marked) atomicAdd(n_marked, (int32_t)marked);
}

// Order-preserving list of the cells with grid >= 0 (above = 0) or grid > 0 (above = 1), as int32 cell ids,
// by per-CTA counts then a scatter (like the alive-list compaction).  offsets[c] (c < C) receives the list
// position of the first listed cell of cascade c and offsets[C] the length: the list is cascade-major.
constexpr int kCellBlock = 1024;
__device__ __forceinline__ bool cell_listed(const float* grid, uint32_t i, uint32_t n, uint32_t above) {
    if (i >= n) return false;
    const float g = grid[i];
    return above ? g > 0.f : g >= 0.f;
}

__global__ void __launch_bounds__(kCellBlock)
k_cell_count(const float* __restrict__ grid, uint32_t n, uint32_t above, uint32_t* __restrict__ counts) {
    const uint32_t c = __syncthreads_count(cell_listed(grid, blockIdx.x * kCellBlock + threadIdx.x, n, above));
    if (threadIdx.x == 0) counts[blockIdx.x] = c;
}

__global__ void __launch_bounds__(kCellBlock)
k_cell_scatter(const float* __restrict__ grid, uint32_t n, uint32_t H3, uint32_t above,
               const uint32_t* __restrict__ counts, int32_t* __restrict__ out, int32_t* __restrict__ offsets) {
    __shared__ uint32_t warp_off[kCellBlock / 32 + 1];
    __shared__ uint32_t base_s;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 32) {  // exclusive prefix of the CTA counts before this CTA
        uint32_t s = 0;
        for (uint32_t b = lane; b < blockIdx.x; b += 32) s += counts[b];
        s = warp_reduce_sum(s);
        if (lane == 0) base_s = s;
    }
    const uint32_t i = blockIdx.x * kCellBlock + tid;
    const bool keep = cell_listed(grid, i, n, above);
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_off[warp] = __popc(bal);
    __syncthreads();
    if (tid < 32) {
        const uint32_t c = warp_off[tid];
        const uint32_t inc = warp_inclusive_scan(c, lane);
        warp_off[tid] = inc - c;
        if (tid == 31) warp_off[kCellBlock / 32] = inc;
    }
    __syncthreads();
    const uint32_t pos = base_s + warp_off[warp] + __popc(bal & ((1u << lane) - 1u));
    if (keep) out[pos] = (int32_t)i;
    if (i < n && i % H3 == 0) offsets[i / H3] = (int32_t)pos;
    if (tid == 0 && blockIdx.x == gridDim.x - 1) offsets[n / H3] = (int32_t)(base_s + warp_off[kCellBlock / 32]);
}

// ------------------------------------------------------------------------------ partial update draws
// torch-ngp's partial update: per cascade c, slots s < Q = H^3/4 draw a uniformly random cell of the cascade,
// slots Q <= s < 2Q draw uniformly from the cascade's ascending list of cells with grid > 0 (slot -> -1 when
// that list is empty).  The draw of (seed, iter, c, s) is the high 32 bits of
// h = splitmix64(splitmix64(splitmix64(seed) ^ iter) ^ (c << 32 | s)) reduced to [0, range) as (hi * range) >> 32.
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__global__ void __launch_bounds__(256)
k_grid_draws(uint32_t C, uint32_t H3, uint64_t key, const int32_t* __restrict__ occupied,
             const int32_t* __restrict__ offsets, int32_t* __restrict__ cells) {
    const uint32_t Q = H3 / 4, D = 2 * Q;
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= C * D) return;
    const uint32_t c = k / D, s = k % D;
    const uint64_t h = splitmix64(key ^ ((uint64_t)c << 32 | s));
    const uint64_t hi = h >> 32;
    int32_t cell;
    if (s < Q) {
        cell = (int32_t)(c * H3 + (uint32_t)((hi * H3) >> 32));
    } else {
        const int32_t lo = __ldg(offsets + c), cnt = __ldg(offsets + c + 1) - lo;
        cell = cnt > 0 ? __ldg(occupied + lo + (uint32_t)((hi * (uint32_t)cnt) >> 32)) : -1;
    }
    cells[k] = cell;
}

// tmp[cells[r]] = max(tmp[cells[r]], vals[r]) for cells[r] >= 0.  tmp starts at -1 and the values are
// sigma * density_scale >= 0, whose order is that of their bit patterns as signed integers: an integer
// atomicMax keeps the maximum whatever the order of the writes (a negative value leaves the cell alone).
__global__ void __launch_bounds__(256)
k_grid_scatter_max(float* __restrict__ tmp, const int32_t* __restrict__ cells, const float* __restrict__ vals,
                   uint32_t count, uint32_t n) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= count) return;
    const int32_t g = __ldg(cells + r);
    if (g < 0 || (uint32_t)g >= n) return;
    atomicMax(reinterpret_cast<int*>(tmp) + g, __float_as_int(__ldg(vals + r)));
}

// tmp = sigma * density_scale (first pass) or max(tmp, sigma * density_scale) (further times)
__global__ void __launch_bounds__(256)
k_grid_accumulate(float* __restrict__ tmp, const float* __restrict__ sigma, uint32_t n, float scale,
                  uint32_t first) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float s = __fmul_rn(__ldg(sigma + i), scale);
    tmp[i] = first ? s : fmaxf(tmp[i], s);
}

constexpr int kUpdBlock = 256;

// grid = max(grid*decay, tmp) where both are >= 0; per-CTA sum of clamp(grid, 0) in double.
__global__ void __launch_bounds__(kUpdBlock)
k_grid_update(float* __restrict__ grid, const float* __restrict__ tmp, uint32_t n, float decay,
              double* __restrict__ partial) {
    __shared__ double red[kUpdBlock / 32];
    double acc = 0.0;
    for (uint32_t i = blockIdx.x * kUpdBlock + threadIdx.x; i < n; i += gridDim.x * kUpdBlock) {
        float g = grid[i];
        const float t = __ldg(tmp + i);
        if (g >= 0.f && t >= 0.f) {
            g = fmaxf(__fmul_rn(g, decay), t);
            grid[i] = g;
        }
        acc += (double)fmaxf(g, 0.f);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < kUpdBlock / 32; ++w) s += red[w];
        partial[blockIdx.x] = s;
    }
}

// stats[0] = mean density, stats[1] = min(mean, density_thresh) (fixed summation order)
__global__ void k_grid_stats(const double* __restrict__ partial, uint32_t nblk, uint32_t n,
                             float density_thresh, float* __restrict__ stats) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double s = 0.0;
    for (uint32_t b = 0; b < nblk; ++b) s += partial[b];
    const float mean = (float)(s / (double)n);
    stats[0] = mean;
    stats[1] = fminf(mean, density_thresh);
}

// packbits (raymarching.cu:287-320) with the threshold read from device memory: one warp turns
// 256 densities (2 x float4 per lane) into 8 words.
__global__ void __launch_bounds__(256)
k_packbits_dev(const float* __restrict__ grid, uint32_t n_bytes, const float* __restrict__ stats,
               uint8_t* __restrict__ bitfield) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_bytes) return;
    const float thresh = __ldg(stats + 1);
    const float4 lo = __ldg(reinterpret_cast<const float4*>(grid) + (size_t)b * 2);
    const float4 hi = __ldg(reinterpret_cast<const float4*>(grid) + (size_t)b * 2 + 1);
    const uint32_t bits = (lo.x > thresh ? 1u : 0u) | (lo.y > thresh ? 2u : 0u) |
                          (lo.z > thresh ? 4u : 0u) | (lo.w > thresh ? 8u : 0u) |
                          (hi.x > thresh ? 16u : 0u) | (hi.y > thresh ? 32u : 0u) |
                          (hi.z > thresh ? 64u : 0u) | (hi.w > thresh ? 128u : 0u);
    bitfield[b] = (uint8_t)bits;
}

// Order-preserving compaction of the inference loop's alive list (rays_alive[rays_alive >= 0] in
// the torch-ngp driver): per-CTA counts, then every CTA sums the counts before it and scatters.
// No atomics, so the surviving rays keep their order and the result is deterministic.
constexpr int kCmpBlock = 1024;
__global__ void __launch_bounds__(kCmpBlock)
k_alive_count(const int32_t* __restrict__ alive, uint32_t n, uint32_t* __restrict__ counts) {
    const uint32_t i = blockIdx.x * kCmpBlock + threadIdx.x;
    const bool keep = i < n && alive[i] >= 0;
    const uint32_t c = __syncthreads_count(keep);
    if (threadIdx.x == 0) counts[blockIdx.x] = c;
}
__global__ void __launch_bounds__(kCmpBlock)
k_alive_scatter(const int32_t* __restrict__ alive, uint32_t n, const uint32_t* __restrict__ counts,
                int32_t* __restrict__ out, int32_t* __restrict__ n_out) {
    __shared__ uint32_t warp_off[kCmpBlock / 32];
    __shared__ uint32_t base_s;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 32) {  // exclusive prefix of the CTA counts before this CTA (<= a few hundred CTAs)
        uint32_t s = 0;
        for (uint32_t b = lane; b < blockIdx.x; b += 32) s += counts[b];
        s = warp_reduce_sum(s);
        if (lane == 0) base_s = s;
    }
    const uint32_t i = blockIdx.x * kCmpBlock + tid;
    const int32_t v = i < n ? alive[i] : -1;
    const bool keep = v >= 0;
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_off[warp] = __popc(bal);
    __syncthreads();
    if (tid < 32) {
        const uint32_t c = warp_off[tid];
        const uint32_t inc = warp_inclusive_scan(c, lane);
        warp_off[tid] = inc - c;
        if (tid == 31 && blockIdx.x == gridDim.x - 1) *n_out = (int32_t)(base_s + inc);
    }
    __syncthreads();
    if (keep) out[base_s + warp_off[warp] + __popc(bal & ((1u << lane) - 1u))] = v;
}

}  // namespace

extern "C" {

int nvsf_get_lidar_rays(const float* pose, const int64_t* inds, uint32_t n, uint32_t H, uint32_t W,
                        float fov_up, float fov, float fov_hoz, float* rays_o, float* rays_d,
                        void* stream) {
    if (n == 0) return NVSF_OK;
    if (!pose || !rays_o || !rays_d || H == 0 || W == 0) return NVSF_E_INVALID;
    k_lidar_rays<<<nvsf_div_up(n, 256u), 256, 0, (cudaStream_t)stream>>>(
        pose, inds, n, H, W, fov_up, fov, fov_hoz, rays_o, rays_d);
    return nvsf_launch_status();
}

int nvsf_get_rays(const float* pose, const int64_t* inds, uint32_t n, uint32_t H, uint32_t W,
                  float fx, float fy, float cx, float cy, float* rays_o, float* rays_d,
                  void* stream) {
    if (n == 0) return NVSF_OK;
    if (!pose || !rays_o || !rays_d || H == 0 || W == 0 || fx == 0.f || fy == 0.f)
        return NVSF_E_INVALID;
    k_camera_rays<<<nvsf_div_up(n, 256u), 256, 0, (cudaStream_t)stream>>>(
        pose, inds, n, H, W, fx, fy, cx, cy, rays_o, rays_d);
    return nvsf_launch_status();
}

int nvsf_error_map_sample(const float* error_map, const float* expo, const float* jitter, uint32_t res,
                          uint32_t N, uint32_t H, uint32_t W, int64_t* inds_coarse, int64_t* inds, void* stream) {
    if (!error_map || !expo || !jitter || !inds_coarse || !inds || res == 0 || res > NVSF_ERROR_MAP_MAX_RES ||
        H == 0 || W == 0 || N == 0 || N > res * res)
        return NVSF_E_INVALID;
    const size_t smem = (size_t)res * res * sizeof(uint32_t);
    const cudaError_t e =
        cudaFuncSetAttribute(k_error_map_sample, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    k_error_map_sample<<<1, kEmBlock, smem, (cudaStream_t)stream>>>(error_map, expo, jitter, res, N, H, W,
                                                                    inds_coarse, inds);
    return nvsf_launch_status();
}

int nvsf_error_map_update(float* error_map, uint32_t R, const int64_t* inds_coarse, uint32_t N, const float* loss,
                          void* stream) {
    if (N == 0) return NVSF_OK;
    if (!error_map || !inds_coarse || !loss || R == 0) return NVSF_E_INVALID;
    k_error_map_update<<<nvsf_div_up(N, 256u), 256, 0, (cudaStream_t)stream>>>(error_map, R, inds_coarse, N, loss);
    return nvsf_launch_status();
}

int nvsf_grid_cell_points(uint32_t C, uint32_t H, float bound, const float* noise, float* xyz,
                          void* stream) {
    if (!xyz || C == 0 || H < 2 || H > 1024 || !(bound > 0.f)) return NVSF_E_INVALID;
    const size_t n = (size_t)C * H * H * H;
    k_grid_cell_points<<<(unsigned)nvsf_div_up(n, (size_t)256), 256, 0, (cudaStream_t)stream>>>(
        C, H, bound, noise, xyz, 0, n);
    return nvsf_launch_status();
}

int nvsf_grid_cell_points_range(uint32_t C, uint32_t H, float bound, const float* noise, uint64_t first,
                                uint64_t count, float* xyz, void* stream) {
    if (!xyz || C == 0 || H < 2 || H > 1024 || !(bound > 0.f)) return NVSF_E_INVALID;
    const size_t n = (size_t)C * H * H * H;
    if (first > n || count > n - first) return NVSF_E_INVALID;
    if (count == 0) return NVSF_OK;
    k_grid_cell_points<<<(unsigned)nvsf_div_up((size_t)count, (size_t)256), 256, 0, (cudaStream_t)stream>>>(
        C, H, bound, noise, xyz, (size_t)first, (size_t)count);
    return nvsf_launch_status();
}

int nvsf_grid_accumulate(float* tmp_grid, const float* sigma, uint32_t n, float density_scale,
                         uint32_t first, void* stream) {
    if (n == 0) return NVSF_OK;
    if (!tmp_grid || !sigma) return NVSF_E_INVALID;
    k_grid_accumulate<<<nvsf_div_up(n, 256u), 256, 0, (cudaStream_t)stream>>>(
        tmp_grid, sigma, n, density_scale, first);
    return nvsf_launch_status();
}

static uint32_t grid_update_blocks(uint32_t n) {
    return std::min<uint32_t>(nvsf_div_up(n, (uint32_t)kUpdBlock), 148u * 8u);
}

size_t nvsf_grid_update_workspace_bytes(uint32_t n) {
    return (size_t)grid_update_blocks(n) * sizeof(double);
}

int nvsf_grid_update(float* density_grid, const float* tmp_grid, uint32_t n, float decay,
                     float density_thresh, uint8_t* bitfield, float* stats, void* workspace,
                     size_t workspace_bytes, void* stream) {
    if (!density_grid || !tmp_grid || !bitfield || !stats || !workspace || n == 0 || n % 8 != 0)
        return NVSF_E_INVALID;
    if ((reinterpret_cast<uintptr_t>(density_grid) & 15) != 0) return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_grid_update_workspace_bytes(n)) return NVSF_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    const uint32_t nblk = grid_update_blocks(n);
    double* partial = reinterpret_cast<double*>(workspace);
    k_grid_update<<<nblk, kUpdBlock, 0, s>>>(density_grid, tmp_grid, n, decay, partial);
    k_grid_stats<<<1, 32, 0, s>>>(partial, nblk, n, density_thresh, stats);
    k_packbits_dev<<<nvsf_div_up(n / 8, 256u), 256, 0, s>>>(density_grid, n / 8, stats, bitfield);
    return nvsf_launch_status();
}

int nvsf_grid_cell_points_list(uint32_t C, uint32_t H, float bound, const int32_t* cells, uint32_t count,
                               const float* noise, uint32_t noise_by_cell, float* xyz, void* stream) {
    if (C == 0 || H < 2 || H > 1024 || !(bound > 0.f) || (uint64_t)C * H * H * H > INT32_MAX) return NVSF_E_INVALID;
    if (count == 0) return NVSF_OK;
    if (!cells || !xyz) return NVSF_E_INVALID;
    k_grid_cell_points_list<<<nvsf_div_up(count, 256u), 256, 0, (cudaStream_t)stream>>>(H, bound, cells, count,
                                                                                        noise, noise_by_cell, xyz);
    return nvsf_launch_status();
}

// Checks shared by the coverage entry points; n = C*H^3 must fill whole 32-bit mask words.
static bool coverage_args_ok(uint32_t C, uint32_t H, float bound, const float* poses, uint8_t* covered) {
    if (!poses || !covered || C == 0 || H < 2 || H > 1024 || !(bound > 0.f)) return false;
    const uint64_t n = (uint64_t)C * H * H * H;
    return n % 32 == 0 && n <= INT32_MAX && (reinterpret_cast<uintptr_t>(covered) & 3) == 0;
}

static int launch_coverage(uint32_t C, uint32_t H, float bound, const float* poses, uint32_t B, const Coverage& S,
                           uint8_t* covered, cudaStream_t s) {
    const uint32_t n = C * H * H * H;
    for (uint32_t b0 = 0; b0 < B; b0 += kCovPoses) {
        k_grid_coverage<<<nvsf_div_up(n, 256u), 256, 0, s>>>(n, H, bound, poses + (size_t)b0 * 16,
                                                             std::min(kCovPoses, B - b0), S,
                                                             reinterpret_cast<uint32_t*>(covered));
        const int e = nvsf_launch_status();
        if (e != NVSF_OK) return e;
    }
    return NVSF_OK;
}

int nvsf_grid_coverage_camera(uint32_t C, uint32_t H, float bound, const float* poses, uint32_t B, float fx,
                              float fy, float cx, float cy, uint32_t img_H, uint32_t img_W, uint8_t* covered,
                              void* stream) {
    if (B == 0) return NVSF_OK;
    if (!coverage_args_ok(C, H, bound, poses, covered) || img_H == 0 || img_W == 0) return NVSF_E_INVALID;
    if (!(fx > 0.f) || !(fy > 0.f) || !std::isfinite(fx) || !std::isfinite(fy) || !std::isfinite(cx) ||
        !std::isfinite(cy))
        return NVSF_E_INVALID;
    Coverage S{};
    S.lidar = 0;
    S.a0 = (float)(-(double)cx / (double)fx);
    S.a1 = (float)(((double)img_W - (double)cx) / (double)fx);
    S.a2 = (float)(-(double)cy / (double)fy);
    S.a3 = (float)(((double)img_H - (double)cy) / (double)fy);
    return launch_coverage(C, H, bound, poses, B, S, covered, (cudaStream_t)stream);
}

int nvsf_grid_coverage_lidar(uint32_t C, uint32_t H, float bound, const float* poses, uint32_t B, float fov_up,
                             float fov, float fov_hoz, float near, float far, uint8_t* covered, void* stream) {
    if (B == 0) return NVSF_OK;
    if (!coverage_args_ok(C, H, bound, poses, covered)) return NVSF_E_INVALID;
    const double up = fov_up, lo = (double)fov_up - (double)fov, hoz = fov_hoz;
    if (!(up < 90.0) || !(lo > -90.0) || !(fov > 0.f) || !(hoz > 0.0 && hoz <= 360.0)) return NVSF_E_INVALID;
    if (!(near >= 0.f) || !(far > near) || !std::isfinite(far)) return NVSF_E_INVALID;
    const double deg = 3.14159265358979323846 / 180.0;
    Coverage S{};
    S.lidar = 1;
    S.a0 = near;
    S.a1 = far;
    S.a2 = (float)std::tan(lo * deg);
    S.a3 = (float)std::tan(up * deg);
    if (hoz < 360.0) {  // wedge [-h, h] of azimuth: inner normals of its edges at -h and +h
        const double h = 0.5 * hoz * deg, sh = std::sin(h), ch = std::cos(h);
        S.wedge = hoz <= 180.0 ? 1u : 2u;
        S.n1x = (float)sh;
        S.n1y = (float)ch;
        S.n2x = (float)sh;
        S.n2y = (float)-ch;
    }
    return launch_coverage(C, H, bound, poses, B, S, covered, (cudaStream_t)stream);
}

int nvsf_grid_apply_marks(float* density_grid, uint8_t* bitfield, const uint8_t* covered, uint32_t n,
                          int32_t* n_marked, void* stream) {
    if (!density_grid || !bitfield || !covered || !n_marked || n == 0 || n % 8 != 0) return NVSF_E_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    const cudaError_t e = cudaMemsetAsync(n_marked, 0, sizeof(int32_t), s);
    if (e != cudaSuccess) return (int)e;
    k_grid_apply_marks<<<nvsf_div_up(n / 8, 256u), 256, 0, s>>>(density_grid, bitfield, covered, n / 8, n_marked);
    return nvsf_launch_status();
}

size_t nvsf_grid_cell_list_workspace_bytes(uint32_t n) {
    return (size_t)nvsf_div_up(n, (uint32_t)kCellBlock) * sizeof(uint32_t);
}

int nvsf_grid_cell_list(const float* density_grid, uint32_t C, uint32_t H3, uint32_t above, int32_t* cells,
                        int32_t* offsets, void* workspace, size_t workspace_bytes, void* stream) {
    if (!density_grid || !cells || !offsets || !workspace || C == 0 || H3 == 0 || above > 1) return NVSF_E_INVALID;
    const uint64_t n64 = (uint64_t)C * H3;
    if (n64 > INT32_MAX) return NVSF_E_INVALID;
    const uint32_t n = (uint32_t)n64;
    if (workspace_bytes < nvsf_grid_cell_list_workspace_bytes(n)) return NVSF_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    const uint32_t nblk = nvsf_div_up(n, (uint32_t)kCellBlock);
    uint32_t* counts = reinterpret_cast<uint32_t*>(workspace);
    k_cell_count<<<nblk, kCellBlock, 0, s>>>(density_grid, n, above, counts);
    k_cell_scatter<<<nblk, kCellBlock, 0, s>>>(density_grid, n, H3, above, counts, cells, offsets);
    return nvsf_launch_status();
}

int nvsf_grid_draws(uint32_t C, uint32_t H3, uint64_t seed, uint64_t iter, const int32_t* occupied,
                    const int32_t* offsets, int32_t* cells, void* stream) {
    if (!occupied || !offsets || !cells || C == 0 || H3 < 4 || H3 % 4 != 0 || (uint64_t)C * H3 > INT32_MAX)
        return NVSF_E_INVALID;
    const uint32_t draws = C * (H3 / 2);
    k_grid_draws<<<nvsf_div_up(draws, 256u), 256, 0, (cudaStream_t)stream>>>(
        C, H3, splitmix64(splitmix64(seed) ^ iter), occupied, offsets, cells);
    return nvsf_launch_status();
}

int nvsf_grid_scatter_max(float* tmp_grid, uint32_t n, const int32_t* cells, const float* vals, uint32_t count,
                          void* stream) {
    if (count == 0) return NVSF_OK;
    if (!tmp_grid || !cells || !vals || n == 0) return NVSF_E_INVALID;
    k_grid_scatter_max<<<nvsf_div_up(count, 256u), 256, 0, (cudaStream_t)stream>>>(tmp_grid, cells, vals, count, n);
    return nvsf_launch_status();
}

size_t nvsf_compact_alive_workspace_bytes(uint32_t n) {
    return (size_t)nvsf_div_up(n, (uint32_t)kCmpBlock) * sizeof(uint32_t);
}

int nvsf_compact_alive(const int32_t* rays_alive, uint32_t n, int32_t* out, int32_t* n_out,
                       void* workspace, size_t workspace_bytes, void* stream) {
    if (!n_out) return NVSF_E_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0) return (int)cudaMemsetAsync(n_out, 0, sizeof(int32_t), s);
    if (!rays_alive || !out || !workspace) return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_compact_alive_workspace_bytes(n)) return NVSF_E_WORKSPACE;
    const uint32_t nblk = nvsf_div_up(n, (uint32_t)kCmpBlock);
    uint32_t* counts = reinterpret_cast<uint32_t*>(workspace);
    k_alive_count<<<nblk, kCmpBlock, 0, s>>>(rays_alive, n, counts);
    k_alive_scatter<<<nblk, kCmpBlock, 0, s>>>(rays_alive, n, counts, out, n_out);
    return nvsf_launch_status();
}

}  // extern "C"
