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

}  // namespace

extern "C" {

size_t nvsf_chamfer_workspace_bytes(uint32_t b, uint32_t n, uint32_t m) {
    return (size_t)b * ((size_t)n + m) * sizeof(unsigned long long);
}

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
    cudaMemsetAsync(workspace, 0xff, nvsf_chamfer_workspace_bytes(b, n, m), s);
    launch_nn(xyz1, n, xyz2, m, b, k1, sms, s);
    launch_nn(xyz2, m, xyz1, n, b, k2, sms, s);
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
    cudaMemsetAsync(workspace, 0xff, nvsf_chamfer_workspace_bytes(1, cap_n, cap_m), s);
    const NnGrid g1 = nn_grid(cap_n, cap_m, 1, sms), g2 = nn_grid(cap_m, cap_n, 1, sms);
    k_chamfer_nn_counted<<<dim3(g1.qblocks, g1.splits), kChThreads, 0, s>>>(xyz1, cap_n, n, xyz2, cap_m, m,
                                                                           g1.per_split, k1);
    k_chamfer_nn_counted<<<dim3(g2.qblocks, g2.splits), kChThreads, 0, s>>>(xyz2, cap_m, m, xyz1, cap_n, n,
                                                                           g2.per_split, k2);
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
