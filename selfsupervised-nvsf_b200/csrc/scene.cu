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
__global__ void __launch_bounds__(256)
k_grid_cell_points(uint32_t C, uint32_t H, float bound, const float* __restrict__ noise,
                   float* __restrict__ xyz, size_t first, size_t count) {
    const uint32_t H3 = H * H * H;
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= count) return;
    const size_t g = first + r;
    const uint32_t c = (uint32_t)(g / H3), m = (uint32_t)(g % H3);
    const float bc = fminf(exp2f((float)c), bound);
    const float half = __fdiv_rn(bc, (float)H);
    const float ext = __fsub_rn(bc, half);
    const uint32_t co[3] = {compact_by3(m), compact_by3(m >> 1), compact_by3(m >> 2)};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float u = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, (float)co[a]), (float)(H - 1)), 1.0f);
        float v = __fmul_rn(u, ext);
        if (noise) {
            const float j = __fsub_rn(__fmul_rn(__ldg(noise + r * 3 + a), 2.0f), 1.0f);
            v = __fadd_rn(v, __fmul_rn(j, half));
        }
        xyz[r * 3 + a] = v;
    }
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
