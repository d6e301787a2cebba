// nvsf_b200 — evaluation of rendered frames on the device (sm_100a): range image -> point cloud, and the
// per-frame metrics of the reference's evaluation (Trainer.evaluate_one_epoch / test_step, trainer.py:817-903,
// 1458-1846; meters nvsf/lib/error_matrices.py, range image -> points nvsf/lib/convert.py).  The metric
// definitions are restated in DESIGN.md §3.5 ("parity unpinned": the reference's nvsf/lib is not in the tree).
//
// Every reduction has a fixed order (per-CTA trees, then one CTA over the CTA partials): the same inputs give
// a bit-identical metric row.  Nothing is read back to the host; the row is written to device memory.
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "lidar_dir.cuh"
#include "radix_select.cuh"

namespace {

// ------------------------------------------------------------------------------------------- block reductions
enum class Op { Sum, Min, Max };

template <Op op>
__device__ __forceinline__ double combine(double a, double b) {
    if (op == Op::Sum) return a + b;
    if (op == Op::Min) return fmin(a, b);
    return fmax(a, b);
}

// Fixed-order reduction over the CTA (butterfly in each warp, then warp 0 over the warp results in order);
// the result is valid in thread 0.  `red` holds one double per warp.
template <Op op>
__device__ __forceinline__ double block_reduce(double v, double* red) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = combine<op>(v, __shfl_xor_sync(0xffffffffu, v, d));
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    __syncthreads();  // `red` may still be read from a previous call
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0)
        for (uint32_t w = 1; w < nwarps; ++w) v = combine<op>(v, red[w]);
    return v;
}

// --------------------------------------------------------------------------------- range image -> point cloud
// Order-preserving compaction as nvsf_compact_alive: per-CTA counts, then every CTA sums the counts before it
// (and all of them, for the total) and scatters.  No atomics: rows are in row-major pixel order.
constexpr int kPtBlock = 1024;

__device__ __forceinline__ float masked_depth(const float* __restrict__ depth, const float* __restrict__ raydrop,
                                              float thr, uint32_t p) {
    const float d = __ldg(depth + p);
    return raydrop ? __fmul_rn(d, __ldg(raydrop + p) > thr ? 1.f : 0.f) : d;
}

__global__ void __launch_bounds__(kPtBlock)
k_points_count(const float* __restrict__ depth, const float* __restrict__ raydrop, float thr, uint32_t n,
               uint32_t* __restrict__ counts) {
    const uint32_t p = blockIdx.x * kPtBlock + threadIdx.x;
    const bool keep = p < n && masked_depth(depth, raydrop, thr, p) != 0.f;
    const uint32_t c = __syncthreads_count(keep);
    if (threadIdx.x == 0) counts[blockIdx.x] = c;
}

// row r of `points` ([n, 3] or [n, 4] with intensity) = lidar_dir(pixel) * (masked depth / scale) of the r-th
// kept pixel; rows [count, n) are zero; *count = number kept.
__global__ void __launch_bounds__(kPtBlock)
k_points_scatter(const float* __restrict__ depth, const float* __restrict__ raydrop, float thr,
                 const float* __restrict__ intensity, uint32_t H, uint32_t W, float fov_up, float fov, float fov_hoz,
                 float scale, const uint32_t* __restrict__ counts, float* __restrict__ points,
                 int32_t* __restrict__ count) {
    __shared__ uint32_t warp_off[kPtBlock / 32];
    __shared__ uint32_t base_s, total_s;
    const uint32_t n = H * W, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 32) {
        uint32_t before = 0, all = 0;
        for (uint32_t b = lane; b < gridDim.x; b += 32) {
            const uint32_t c = counts[b];
            all += c;
            if (b < blockIdx.x) before += c;
        }
        before = warp_reduce_sum(before);
        all = warp_reduce_sum(all);
        if (lane == 0) { base_s = before; total_s = all; }
    }
    const uint32_t p = blockIdx.x * kPtBlock + tid;
    const float md = p < n ? masked_depth(depth, raydrop, thr, p) : 0.f;
    const bool keep = p < n && md != 0.f;
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_off[warp] = __popc(bal);
    __syncthreads();
    if (tid < 32) {
        const uint32_t c = warp_off[tid];
        warp_off[tid] = warp_inclusive_scan(c, lane) - c;
    }
    __syncthreads();
    const uint32_t cols = intensity ? 4u : 3u;
    if (keep) {
        const size_t row = base_s + warp_off[warp] + __popc(bal & ((1u << lane) - 1u));
        float x, y, z;
        lidar_dir(p, H, W, fov_up, fov, fov_hoz, x, y, z);
        const float r = __fdiv_rn(md, scale);
        float* o = points + row * cols;
        o[0] = __fmul_rn(x, r);
        o[1] = __fmul_rn(y, r);
        o[2] = __fmul_rn(z, r);
        if (intensity) o[3] = __ldg(intensity + p);
    }
    // row p past the count is zeroed whether or not pixel p is kept: a kept pixel's own row is always below
    // the count, so the two stores never meet
    if (p < n && p >= total_s)
        for (uint32_t c = 0; c < cols; ++c) points[(size_t)p * cols + c] = 0.f;
    if (blockIdx.x == 0 && tid == 0) *count = (int32_t)total_s;
}

uint32_t points_blocks(uint32_t n) { return nvsf_div_up(n, (uint32_t)kPtBlock); }

void launch_points(const float* depth, const float* raydrop, float thr, const float* intensity, uint32_t H,
                   uint32_t W, float fov_up, float fov, float fov_hoz, float scale, float* points, int32_t* count,
                   uint32_t* counts, cudaStream_t s) {
    const uint32_t nblk = points_blocks(H * W);
    k_points_count<<<nblk, kPtBlock, 0, s>>>(depth, raydrop, thr, H * W, counts);
    k_points_scatter<<<nblk, kPtBlock, 0, s>>>(depth, raydrop, thr, intensity, H, W, fov_up, fov, fov_hoz, scale,
                                               counts, points, count);
}

// --------------------------------------------------------------------------------- point cloud -> range image
// The nearest return of each pixel, ties to the lowest point index: one 64-bit key per pixel, (depth32 bits << 32 |
// index within the scan), lowered by atomicMin (depth32 > 0, so its fp32 bits order as integers); 0xFF..FF = empty.
// Float64 arithmetic in the contract's order (DESIGN.md §3.5), every operation rounded on its own.
constexpr int kRiBlock = 256;
constexpr unsigned long long kRiEmpty = ~0ull;
constexpr uint32_t kRiNoPixel = 0xFFFFFFFFu;  // above every pixel id (H*W <= 2^26)

__device__ __forceinline__ double ri_col_or_row(double num, double den, uint32_t n) {
    return rint(__dmul_rn(__ddiv_rn(num, den), (double)n));
}

// Grid (point blocks, scans), blockIdx.x fastest: the blocks in flight cover one or two scans, whose keys stay in L2.
__global__ void __launch_bounds__(kRiBlock)
k_range_scatter(const float* __restrict__ points, uint32_t channels, const int64_t* __restrict__ offsets,
                const float* __restrict__ poses, uint32_t H, uint32_t W, float fov_up, float fov, float fov_hoz,
                float max_depth, unsigned long long* __restrict__ keys) {
    __shared__ double pose_s[12];  // rows 0..2 of lidar2world: R | t
    const uint32_t b = blockIdx.y;
    const int64_t begin = offsets[b], count = offsets[b + 1] - begin;
    if ((int64_t)blockIdx.x * kRiBlock >= count) return;
    if (poses && threadIdx.x < 12) pose_s[threadIdx.x] = (double)poses[(size_t)b * 16 + threadIdx.x];
    __syncthreads();
    const uint32_t i = blockIdx.x * kRiBlock + threadIdx.x;
    uint32_t pix = kRiNoPixel;
    float depth32 = 0.f;
    if ((int64_t)i < count) {
        const float* p = points + (size_t)(begin + i) * channels;
        double qx = (double)__ldg(p), qy = (double)__ldg(p + 1), qz = (double)__ldg(p + 2);
        if (poses) {  // R^T (p - t)
            const double dx = __dsub_rn(qx, pose_s[3]), dy = __dsub_rn(qy, pose_s[7]), dz = __dsub_rn(qz, pose_s[11]);
            qx = __dadd_rn(__dadd_rn(__dmul_rn(pose_s[0], dx), __dmul_rn(pose_s[4], dy)), __dmul_rn(pose_s[8], dz));
            qy = __dadd_rn(__dadd_rn(__dmul_rn(pose_s[1], dx), __dmul_rn(pose_s[5], dy)), __dmul_rn(pose_s[9], dz));
            qz = __dadd_rn(__dadd_rn(__dmul_rn(pose_s[2], dx), __dmul_rn(pose_s[6], dy)), __dmul_rn(pose_s[10], dz));
        }
        const double xy2 = __dadd_rn(__dmul_rn(qx, qx), __dmul_rn(qy, qy));
        depth32 = __double2float_rn(__dsqrt_rn(__dadd_rn(xy2, __dmul_rn(qz, qz))));
        if (depth32 > 0.f && depth32 < max_depth) {  // false for NaN; inf is never below max_depth
            const double kDeg = 180.0 / 3.14159265358979323846;
            const double beta = __dmul_rn(atan2(qy, qx), kDeg), alpha = __dmul_rn(atan2(qz, __dsqrt_rn(xy2)), kDeg);
            const double fh = (double)fov_hoz;
            const double c = ri_col_or_row(__dsub_rn(__dmul_rn(0.5, fh), beta), fh, W);
            const double r = ri_col_or_row(__dsub_rn((double)fov_up, alpha), (double)fov, H);
            // the seam half-column that rounds to c = W is dropped, as the reference loop drops it
            if (c >= 0.0 && c < (double)W && r >= 0.0 && r < (double)H) pix = (uint32_t)r * W + (uint32_t)c;
        }
    }
    const unsigned long long key = ((unsigned long long)__float_as_uint(depth32) << 32) | i;
    // Same-address reductions serialise; lanes of a warp that share a pixel (an accumulated cloud, a point
    // repeated, a scan in firing order) first take their minimum by pointer jumping along the lanes of their group,
    // and the lowest lane issues the one reduction.  The grouping (MATCH.ANY) costs ~10 % on a scan of distinct
    // pixels, so it only runs in a warp where two neighbouring lanes share a pixel.
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t prev = __shfl_up_sync(0xffffffffu, pix, 1);
    unsigned long long kmin = key;
    bool lead = true;
    if (__any_sync(0xffffffffu, lane > 0 && prev == pix && pix != kRiNoPixel)) {
        const uint32_t peers = __match_any_sync(0xffffffffu, pix);
        lead = (peers & ((1u << lane) - 1u)) == 0;
        const uint32_t above = peers & ~((2u << lane) - 1u);
        int next = above ? __ffs(above) - 1 : -1;
#pragma unroll
        for (int step = 0; step < 5; ++step) {
            const int src = next >= 0 ? next : (int)lane;
            const unsigned long long k2 = __shfl_sync(0xffffffffu, kmin, src);
            const int n2 = __shfl_sync(0xffffffffu, next, src);
            if (next >= 0) {
                kmin = k2 < kmin ? k2 : kmin;
                next = n2;
            }
        }
    }
    if (pix != kRiNoPixel && lead)
        atomicMin(keys + (size_t)b * H * W + pix, kmin);  // result unused: a RED, not an ATOM
}

// One thread per pixel: the winner's row (1, intensity or 0, depth32 * scale) and its global point row, or
// (0, 0, 0) and -1 for an empty pixel.
__global__ void __launch_bounds__(kRiBlock)
k_range_resolve(const unsigned long long* __restrict__ keys, const float* __restrict__ points, uint32_t channels,
                const int64_t* __restrict__ offsets, uint32_t n, float scale, float* __restrict__ images,
                int64_t* __restrict__ index) {
    const uint32_t p = blockIdx.x * kRiBlock + threadIdx.x;
    if (p >= n) return;
    const size_t g = (size_t)blockIdx.y * n + p;
    const unsigned long long k = keys[g];
    float m = 0.f, it = 0.f, d = 0.f;
    int64_t row = -1;
    if (k != kRiEmpty) {
        row = offsets[blockIdx.y] + (int64_t)(uint32_t)k;
        m = 1.f;
        if (channels == 4) it = __ldg(points + (size_t)row * 4 + 3);
        d = __fmul_rn(__uint_as_float((uint32_t)(k >> 32)), scale);
    }
    images[3 * g] = m;
    images[3 * g + 1] = it;
    images[3 * g + 2] = d;
    if (index) index[g] = row;
}

// ------------------------------------------------------------------------------------------ LiDAR pixel pass
// Per pixel, with m^ = (raydrop^ > 0.5): P = D^ m^ / scale, G = D r / scale (unclamped: the point clouds),
// clamped copies for depth [1e-3, max_depth] and intensity I^ = i^ m^, I = i r in [1e-6, 1] (the SSIM images),
// |G - P| and |I - I^| of the clamped values (the medians), and per-CTA partials of the accumulators below.
enum Acc : int {
    kSqDepth, kSqInt, kSqDrop, kAgree, kTp, kFp, kFn,  // sums
    kGMinDepth, kGMinInt,                              // minima
    kGMaxDepth, kGMaxInt,                              // maxima
    kNAcc
};
constexpr int kFirstMin = kGMinDepth, kFirstMax = kGMaxDepth;
constexpr int kPixBlock = 256;
constexpr uint32_t kPixMaxBlocks = 148u * 4u;

uint32_t pixel_blocks(uint32_t n) { return std::min<uint32_t>(nvsf_div_up(n, (uint32_t)kPixBlock), kPixMaxBlocks); }

__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

struct LidarImages {  // [n] each
    float *pc, *gc, *ip, *ig, *pu, *gu, *ad, *ai;
};

__global__ void __launch_bounds__(kPixBlock)
k_lidar_pixels(const float* __restrict__ depth, const float* __restrict__ image, const float* __restrict__ gt,
               uint32_t n, float scale, float max_depth, LidarImages im, double* __restrict__ partial) {
    __shared__ double red[kPixBlock / 32];
    double acc[kNAcc];
#pragma unroll
    for (int a = 0; a < kNAcc; ++a) acc[a] = a < kFirstMin ? 0.0 : (a < kFirstMax ? INFINITY : -INFINITY);
    for (uint32_t p = blockIdx.x * kPixBlock + threadIdx.x; p < n; p += gridDim.x * kPixBlock) {
        const float dh = __ldg(depth + p), rh = __ldg(image + 2 * (size_t)p), ih = __ldg(image + 2 * (size_t)p + 1);
        const float r = __ldg(gt + 3 * (size_t)p), it = __ldg(gt + 3 * (size_t)p + 1),
                    dt = __ldg(gt + 3 * (size_t)p + 2);
        const float mh = rh > 0.5f ? 1.f : 0.f;
        const float pu = __fdiv_rn(__fmul_rn(dh, mh), scale), gu = __fdiv_rn(__fmul_rn(dt, r), scale);
        const float pc = clampf(pu, 1e-3f, max_depth), gc = clampf(gu, 1e-3f, max_depth);
        const float ip = clampf(__fmul_rn(ih, mh), 1e-6f, 1.f), ig = clampf(__fmul_rn(it, r), 1e-6f, 1.f);
        const float ed = __fsub_rn(gc, pc), ei = __fsub_rn(ig, ip);
        im.pu[p] = pu; im.gu[p] = gu;
        im.pc[p] = pc; im.gc[p] = gc;
        im.ip[p] = ip; im.ig[p] = ig;
        im.ad[p] = fabsf(ed); im.ai[p] = fabsf(ei);
        const double dr = (double)r - (double)mh;
        const bool pos = mh != 0.f, tpos = r > 0.5f;
        acc[kSqDepth] += (double)ed * (double)ed;
        acc[kSqInt] += (double)ei * (double)ei;
        acc[kSqDrop] += dr * dr;
        acc[kAgree] += pos == tpos ? 1.0 : 0.0;
        acc[kTp] += pos && tpos ? 1.0 : 0.0;
        acc[kFp] += pos && !tpos ? 1.0 : 0.0;
        acc[kFn] += !pos && tpos ? 1.0 : 0.0;
        acc[kGMinDepth] = fmin(acc[kGMinDepth], (double)gc);
        acc[kGMinInt] = fmin(acc[kGMinInt], (double)ig);
        acc[kGMaxDepth] = fmax(acc[kGMaxDepth], (double)gc);
        acc[kGMaxInt] = fmax(acc[kGMaxInt], (double)ig);
    }
#pragma unroll
    for (int a = 0; a < kNAcc; ++a) {
        const double v = a < kFirstMin ? block_reduce<Op::Sum>(acc[a], red)
                         : a < kFirstMax ? block_reduce<Op::Min>(acc[a], red)
                                         : block_reduce<Op::Max>(acc[a], red);
        if (threadIdx.x == 0) partial[(size_t)blockIdx.x * kNAcc + a] = v;
    }
}

// stats[a] = the accumulators over all CTAs (CTA order); stats[kNAcc + 0 / 1] = SSIM data range of depth /
// intensity = max G - min G.
__global__ void k_lidar_stats(const double* __restrict__ partial, uint32_t nblk, double* __restrict__ stats) {
    const int a = threadIdx.x;
    if (a < kNAcc) {
        double v = partial[a];
        for (uint32_t b = 1; b < nblk; ++b) {
            const double x = partial[(size_t)b * kNAcc + a];
            v = a < kFirstMin ? v + x : (a < kFirstMax ? fmin(v, x) : fmax(v, x));
        }
        stats[a] = v;
    }
    __syncthreads();
    if (a == 0) {
        stats[kNAcc + 0] = stats[kGMaxDepth] - stats[kGMinDepth];
        stats[kNAcc + 1] = stats[kGMaxInt] - stats[kGMinInt];
    }
}

// ------------------------------------------------------------------------------------------------------ SSIM
// skimage.metrics.structural_similarity with its defaults: 7x7 uniform window, K1 = 0.01, K2 = 0.03, sample
// covariance (/48), mean over the windows that lie entirely inside the image (skimage's 3-pixel crop).  One
// thread per window over a shared-memory tile; the moments are two-pass (mean, then centred sums) so depths up
// to 80 m lose nothing to E[x^2] - E[x]^2 cancellation.  Per-CTA partial sums of S in double.
constexpr int kSsWin = 7, kSsTX = 32, kSsTY = 8;
constexpr int kSsInX = kSsTX + kSsWin - 1, kSsInY = kSsTY + kSsWin - 1;

__global__ void __launch_bounds__(kSsTX * kSsTY)
k_ssim(const float* __restrict__ x, const float* __restrict__ y, uint32_t H, uint32_t W, uint32_t channels,
       const double* __restrict__ range_dev, double range, double* __restrict__ partial) {
    __shared__ float sx[kSsInY][kSsInX], sy[kSsInY][kSsInX];
    __shared__ double red[kSsTX * kSsTY / 32];
    const uint32_t c = blockIdx.z, ox0 = blockIdx.x * kSsTX, oy0 = blockIdx.y * kSsTY;
    for (uint32_t k = threadIdx.x; k < kSsInX * kSsInY; k += kSsTX * kSsTY) {
        const uint32_t ty = k / kSsInX, tx = k % kSsInX, gy = oy0 + ty, gx = ox0 + tx;
        const bool in = gy < H && gx < W;
        const size_t g = ((size_t)gy * W + gx) * channels + c;
        sx[ty][tx] = in ? __ldg(x + g) : 0.f;
        sy[ty][tx] = in ? __ldg(y + g) : 0.f;
    }
    __syncthreads();
    const uint32_t tx = threadIdx.x % kSsTX, ty = threadIdx.x / kSsTX;
    double S = 0.0;
    if (oy0 + ty + kSsWin <= H && ox0 + tx + kSsWin <= W) {
        float mx = 0.f, my = 0.f;
#pragma unroll
        for (int a = 0; a < kSsWin; ++a)
#pragma unroll
            for (int b = 0; b < kSsWin; ++b) { mx += sx[ty + a][tx + b]; my += sy[ty + a][tx + b]; }
        mx /= 49.f;
        my /= 49.f;
        float vx = 0.f, vy = 0.f, vxy = 0.f;
#pragma unroll
        for (int a = 0; a < kSsWin; ++a)
#pragma unroll
            for (int b = 0; b < kSsWin; ++b) {
                const float dx = sx[ty + a][tx + b] - mx, dy = sy[ty + a][tx + b] - my;
                vx = fmaf(dx, dx, vx);
                vy = fmaf(dy, dy, vy);
                vxy = fmaf(dx, dy, vxy);
            }
        const double R = range_dev ? *range_dev : range;
        const double C1 = (0.01 * R) * (0.01 * R), C2 = (0.03 * R) * (0.03 * R);
        const double ux = mx, uy = my, sxx = vx / 48.0, syy = vy / 48.0, sxy = vxy / 48.0;
        S = ((2.0 * ux * uy + C1) * (2.0 * sxy + C2)) / ((ux * ux + uy * uy + C1) * (sxx + syy + C2));
    }
    S = block_reduce<Op::Sum>(S, red);
    if (threadIdx.x == 0) partial[((size_t)c * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = S;
}

struct SsimGrid {
    dim3 grid;
    uint32_t per_channel;  // CTAs (= partials) per channel
    uint32_t windows;      // windows per channel; 0 when the image is smaller than 7x7 (SSIM = NaN)
};

SsimGrid ssim_grid(uint32_t H, uint32_t W, uint32_t channels) {
    if (H < (uint32_t)kSsWin || W < (uint32_t)kSsWin) return {dim3(1, 1, channels), 0, 0};
    const uint32_t wy = H - kSsWin + 1, wx = W - kSsWin + 1;
    const dim3 g(nvsf_div_up(wx, (uint32_t)kSsTX), nvsf_div_up(wy, (uint32_t)kSsTY), channels);
    return {g, g.x * g.y, wy * wx};
}

// ------------------------------------------------------------------------------------------------ medians
// Exact order statistics of non-negative floats (their bits order as unsigned integers): one CTA per (rank,
// array) runs a 4-pass, 8-bit radix select.  For an odd count both CTAs of an array select rank n/2, for an
// even count ranks n/2 - 1 and n/2 (np.median's two middle values).
constexpr int kSelBlock = 1024;

__global__ void __launch_bounds__(kSelBlock)
k_select(const float* __restrict__ arrays, uint32_t n, float* __restrict__ sel) {
    __shared__ uint32_t hist[256];
    const float* a = arrays + (size_t)blockIdx.y * n;
    const uint32_t k = (n & 1u) ? n / 2 : n / 2 - 1 + blockIdx.x;
    uint32_t ties;
    const uint32_t v = radix_select<kSelBlock>([a](uint32_t i) { return __float_as_uint(__ldg(a + i)); }, n, k,
                                               hist, ties);
    if (threadIdx.x == 0) sel[blockIdx.y * 2 + blockIdx.x] = __uint_as_float(v);
}

__device__ __forceinline__ float median_of(const float* sel, uint32_t n) {
    return (n & 1u) ? sel[0] : __fmul_rn(__fadd_rn(sel[0], sel[1]), 0.5f);
}

// ------------------------------------------------------------------------------------------------ finalize
constexpr int kFinBlock = 256;

// sum of v[0..n) in a fixed order (strided per thread, then block_reduce); valid in thread 0
__device__ double block_sum(const double* __restrict__ v, uint32_t n, double* red) {
    double s = 0.0;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s += v[i];
    return block_reduce<Op::Sum>(s, red);
}

__device__ __forceinline__ double ssim_mean(const double* partial, const SsimGrid& g, uint32_t c, double* red) {
    const double s = block_sum(partial + (size_t)c * g.per_channel, g.per_channel, red);
    return g.windows ? s / (double)g.windows : NAN;
}

__device__ __forceinline__ double f1_of(double p, double r) { return p + r > 0.0 ? 2.0 * p * r / (p + r) : 0.0; }

// The point metrics of both meters, from the squared nearest-neighbour distances of the np_ predicted and ng
// ground-truth points: chamfer = mean dist1 + mean dist2, fscore = F1 of the shares below the threshold; +inf / 0
// when a cloud is empty.  Called by the whole CTA; the results are valid in thread 0.
__device__ void points_metrics(const float* __restrict__ dist1, const float* __restrict__ dist2, uint32_t np_,
                               uint32_t ng, float fscore_threshold, double* red, double& chamfer, double& fscore) {
    double s1 = 0.0, s2 = 0.0, c1 = 0.0, c2 = 0.0;
    if (np_ && ng) {
        for (uint32_t i = threadIdx.x; i < np_; i += kFinBlock) {
            s1 += dist1[i];
            c1 += dist1[i] < fscore_threshold ? 1.0 : 0.0;
        }
        for (uint32_t i = threadIdx.x; i < ng; i += kFinBlock) {
            s2 += dist2[i];
            c2 += dist2[i] < fscore_threshold ? 1.0 : 0.0;
        }
    }
    s1 = block_reduce<Op::Sum>(s1, red);
    s2 = block_reduce<Op::Sum>(s2, red);
    c1 = block_reduce<Op::Sum>(c1, red);
    c2 = block_reduce<Op::Sum>(c2, red);
    chamfer = INFINITY;
    fscore = 0.0;
    if (np_ && ng) {
        chamfer = s1 / (double)np_ + s2 / (double)ng;
        fscore = f1_of(c1 / (double)np_, c2 / (double)ng);
    }
}

__global__ void __launch_bounds__(kFinBlock)
k_lidar_finalize(const double* __restrict__ stats, const double* __restrict__ ssim_part, SsimGrid sg,
                 const float* __restrict__ sel, uint32_t n, float max_depth, float fscore_threshold,
                 const float* __restrict__ dist1, const float* __restrict__ dist2, const int32_t* __restrict__ counts,
                 float* __restrict__ row) {
    __shared__ double red[kFinBlock / 32];
    const double ssim_d = ssim_mean(ssim_part, sg, 0, red);
    const double ssim_i = ssim_mean(ssim_part, sg, 1, red);
    const uint32_t np_ = (uint32_t)max(counts[0], 0), ng = (uint32_t)max(counts[1], 0);
    double chamfer, fscore;
    points_metrics(dist1, dist2, np_, ng, fscore_threshold, red, chamfer, fscore);
    if (threadIdx.x != 0) return;
    const double N = (double)n, md = (double)max_depth;
    const double mse_d = stats[kSqDepth] / N, mse_i = stats[kSqInt] / N;
    const double tp = stats[kTp], fp = stats[kFp], fn = stats[kFn];
    const double prec = tp + fp > 0.0 ? tp / (tp + fp) : 0.0, rec = tp + fn > 0.0 ? tp / (tp + fn) : 0.0;
    const double out[NVSF_EVAL_LIDAR_K] = {
        sqrt(mse_d), (double)median_of(sel, n), 10.0 * log10(md * md / mse_d), ssim_d,
        sqrt(mse_i), (double)median_of(sel + 2, n), 10.0 * log10(1.0 / mse_i), ssim_i,
        sqrt(stats[kSqDrop] / N), stats[kAgree] / N, f1_of(prec, rec),
        chamfer, fscore, (double)np_, (double)ng};
    for (int k = 0; k < NVSF_EVAL_LIDAR_K; ++k) row[k] = (float)out[k];
}

// row = (chamfer, fscore, points_pred, points_gt) of two clouds with device counts (clamped to the capacities)
__global__ void __launch_bounds__(kFinBlock)
k_points_finalize(const float* __restrict__ dist1, const float* __restrict__ dist2, const int32_t* __restrict__ n_pred,
                  uint32_t cap_p, const int32_t* __restrict__ n_gt, uint32_t cap_g, float fscore_threshold,
                  float* __restrict__ row) {
    __shared__ double red[kFinBlock / 32];
    const uint32_t np_ = (uint32_t)min(max(*n_pred, 0), (int32_t)cap_p), ng = (uint32_t)min(max(*n_gt, 0), (int32_t)cap_g);
    double chamfer, fscore;
    points_metrics(dist1, dist2, np_, ng, fscore_threshold, red, chamfer, fscore);
    if (threadIdx.x != 0) return;
    row[0] = (float)chamfer;
    row[1] = (float)fscore;
    row[2] = (float)np_;
    row[3] = (float)ng;
}

// ------------------------------------------------------------------------------------------------- camera
__global__ void __launch_bounds__(kPixBlock)
k_sq_err(const float* __restrict__ a, const float* __restrict__ b, size_t n, double* __restrict__ partial) {
    __shared__ double red[kPixBlock / 32];
    double s = 0.0;
    for (size_t i = (size_t)blockIdx.x * kPixBlock + threadIdx.x; i < n; i += (size_t)gridDim.x * kPixBlock) {
        const float e = __fsub_rn(__ldg(a + i), __ldg(b + i));
        s += (double)e * (double)e;
    }
    s = block_reduce<Op::Sum>(s, red);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kFinBlock)
k_camera_finalize(const double* __restrict__ sq_part, uint32_t nsq, size_t n, const double* __restrict__ ssim_part,
                  SsimGrid sg, float* __restrict__ row) {
    __shared__ double red[kFinBlock / 32];
    const double sq = block_sum(sq_part, nsq, red);
    double ssim = 0.0;
    for (uint32_t c = 0; c < 3; ++c) ssim += ssim_mean(ssim_part, sg, c, red);
    if (threadIdx.x != 0) return;
    row[0] = (float)(-10.0 * log10(sq / (double)n));
    row[1] = (float)(ssim / 3.0);
}

// --------------------------------------------------------------------------------------------- workspaces
constexpr size_t kAlign = 256;

struct Carve {
    size_t off = 0;
    template <typename T>
    size_t take(size_t count) {
        const size_t at = off;
        off = nvsf_div_up(off + count * sizeof(T), kAlign) * kAlign;
        return at;
    }
};

struct LidarWs {
    size_t images, partial, stats, ssim, sel, pts_p, pts_g, counts, cmp, ch_ws, d1, d2, i1, i2, bytes;
};

LidarWs lidar_ws(uint32_t n, uint32_t H, uint32_t W) {
    Carve c;
    LidarWs w;
    w.images = c.take<float>((size_t)8 * n);
    w.partial = c.take<double>((size_t)pixel_blocks(n) * kNAcc);
    w.stats = c.take<double>(kNAcc + 2);
    w.ssim = c.take<double>((size_t)2 * ssim_grid(H, W, 1).per_channel);
    w.sel = c.take<float>(4);
    w.pts_p = c.take<float>((size_t)3 * n);
    w.pts_g = c.take<float>((size_t)3 * n);
    w.counts = c.take<int32_t>(2);
    w.cmp = c.take<uint32_t>((size_t)2 * points_blocks(n));
    w.ch_ws = c.take<unsigned char>(nvsf_chamfer_workspace_bytes(1, n, n));
    w.d1 = c.take<float>(n);
    w.d2 = c.take<float>(n);
    w.i1 = c.take<int32_t>(n);
    w.i2 = c.take<int32_t>(n);
    w.bytes = c.off;
    return w;
}

struct CameraWs {
    size_t partial, ssim, bytes;
};

CameraWs camera_ws(uint32_t H, uint32_t W) {
    Carve c;
    CameraWs w;
    w.partial = c.take<double>(pixel_blocks(H * W));
    w.ssim = c.take<double>((size_t)3 * ssim_grid(H, W, 1).per_channel);
    w.bytes = c.off;
    return w;
}

// frames up to 2^26 pixels (a 66 x 1030 LiDAR frame has 67 980, a 376 x 1408 camera frame 529 408)
bool frame_ok(uint32_t H, uint32_t W) { return H > 0 && W > 0 && (uint64_t)H * W <= (1ull << 26); }

struct PointsWs {
    size_t ch_ws, d1, d2, i1, i2, bytes;
};

PointsWs points_ws(uint32_t cap_p, uint32_t cap_g) {
    Carve c;
    PointsWs w;
    w.ch_ws = c.take<unsigned char>(nvsf_chamfer_workspace_bytes(1, cap_p, cap_g));
    w.d1 = c.take<float>(cap_p);
    w.d2 = c.take<float>(cap_g);
    w.i1 = c.take<int32_t>(cap_p);
    w.i2 = c.take<int32_t>(cap_g);
    w.bytes = c.off;
    return w;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

extern "C" {

size_t nvsf_lidar_points_workspace_bytes(uint32_t H, uint32_t W) {
    return frame_ok(H, W) ? (size_t)points_blocks(H * W) * sizeof(uint32_t) : 0;
}

int nvsf_lidar_points(const float* depth, const float* raydrop, float raydrop_threshold, const float* intensity,
                      uint32_t H, uint32_t W, float fov_up, float fov, float fov_hoz, float scale, float* points,
                      int32_t* count, void* workspace, size_t workspace_bytes, void* stream) {
    if (!depth || !points || !count || !workspace || !frame_ok(H, W)) return NVSF_E_INVALID;
    if (!(scale > 0.f) || !std::isfinite(scale)) return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_lidar_points_workspace_bytes(H, W)) return NVSF_E_WORKSPACE;
    launch_points(depth, raydrop, raydrop_threshold, intensity, H, W, fov_up, fov, fov_hoz, scale, points, count,
                  reinterpret_cast<uint32_t*>(workspace), (cudaStream_t)stream);
    return nvsf_launch_status();
}

size_t nvsf_range_image_workspace_bytes(uint32_t B, uint32_t H, uint32_t W) {
    return frame_ok(H, W) ? (size_t)B * H * W * sizeof(unsigned long long) : 0;
}

int nvsf_range_image(const float* points, uint32_t channels, const int64_t* offsets, uint32_t B, uint32_t max_count,
                     const float* poses, uint32_t H, uint32_t W, float fov_up, float fov, float fov_hoz, float scale,
                     float max_depth, float* images, int64_t* index, void* workspace, size_t workspace_bytes,
                     void* stream) {
    if ((channels != 3 && channels != 4) || !frame_ok(H, W) || B > 65535u) return NVSF_E_INVALID;
    if (B == 0) return NVSF_OK;
    if (!offsets || !images || !workspace || (max_count && !points)) return NVSF_E_INVALID;
    if (reinterpret_cast<uintptr_t>(workspace) & 7u) return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_range_image_workspace_bytes(B, H, W)) return NVSF_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    auto* keys = reinterpret_cast<unsigned long long*>(workspace);
    const uint32_t n = H * W;
    cudaError_t e = cudaMemsetAsync(keys, 0xFF, (size_t)B * n * sizeof(unsigned long long), s);
    if (e != cudaSuccess) return (int)e;
    if (max_count)
        k_range_scatter<<<dim3((uint32_t)nvsf_div_up<uint64_t>(max_count, kRiBlock), B), kRiBlock, 0, s>>>(
            points, channels, offsets, poses, H, W, fov_up, fov, fov_hoz, max_depth, keys);
    k_range_resolve<<<dim3(nvsf_div_up(n, (uint32_t)kRiBlock), B), kRiBlock, 0, s>>>(keys, points, channels, offsets, n,
                                                                                      scale, images, index);
    return nvsf_launch_status();
}

size_t nvsf_eval_lidar_workspace_bytes(uint32_t H, uint32_t W) {
    return frame_ok(H, W) ? lidar_ws(H * W, H, W).bytes : 0;
}

int nvsf_eval_lidar(const float* depth, const float* image, const float* gt, uint32_t H, uint32_t W, float fov_up,
                    float fov, float fov_hoz, float scale, float max_depth, float fscore_threshold, float* row,
                    void* workspace, size_t workspace_bytes, void* stream) {
    if (!depth || !image || !gt || !row || !workspace || !frame_ok(H, W) || !aligned16(workspace))
        return NVSF_E_INVALID;
    if (!(scale > 0.f) || !std::isfinite(scale) || !(max_depth > 1e-3f) || !std::isfinite(max_depth) ||
        !(fscore_threshold >= 0.f))
        return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_eval_lidar_workspace_bytes(H, W)) return NVSF_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    const uint32_t n = H * W;
    const LidarWs w = lidar_ws(n, H, W);
    char* base = reinterpret_cast<char*>(workspace);
    float* img = reinterpret_cast<float*>(base + w.images);
    const LidarImages im{img, img + n, img + 2 * (size_t)n, img + 3 * (size_t)n,
                         img + 4 * (size_t)n, img + 5 * (size_t)n, img + 6 * (size_t)n, img + 7 * (size_t)n};
    double* partial = reinterpret_cast<double*>(base + w.partial);
    double* stats = reinterpret_cast<double*>(base + w.stats);
    double* ssim_part = reinterpret_cast<double*>(base + w.ssim);
    float* sel = reinterpret_cast<float*>(base + w.sel);
    float* pts_p = reinterpret_cast<float*>(base + w.pts_p);
    float* pts_g = reinterpret_cast<float*>(base + w.pts_g);
    int32_t* counts = reinterpret_cast<int32_t*>(base + w.counts);
    uint32_t* cmp = reinterpret_cast<uint32_t*>(base + w.cmp);
    float* d1 = reinterpret_cast<float*>(base + w.d1);
    float* d2 = reinterpret_cast<float*>(base + w.d2);

    const uint32_t nblk = pixel_blocks(n);
    k_lidar_pixels<<<nblk, kPixBlock, 0, s>>>(depth, image, gt, n, scale, max_depth, im, partial);
    k_lidar_stats<<<1, 32, 0, s>>>(partial, nblk, stats);
    const SsimGrid sg = ssim_grid(H, W, 1);
    if (sg.windows) {
        k_ssim<<<sg.grid, kSsTX * kSsTY, 0, s>>>(im.pc, im.gc, H, W, 1, stats + kNAcc, 0.0, ssim_part);
        k_ssim<<<sg.grid, kSsTX * kSsTY, 0, s>>>(im.ip, im.ig, H, W, 1, stats + kNAcc + 1, 0.0,
                                                 ssim_part + sg.per_channel);
    }
    k_select<<<dim3(2, 2), kSelBlock, 0, s>>>(im.ad, n, sel);  // im.ad and im.ai are adjacent
    launch_points(im.pu, nullptr, 0.f, nullptr, H, W, fov_up, fov, fov_hoz, 1.f, pts_p, counts, cmp, s);
    launch_points(im.gu, nullptr, 0.f, nullptr, H, W, fov_up, fov, fov_hoz, 1.f, pts_g, counts + 1,
                  cmp + points_blocks(n), s);
    const int st = nvsf_chamfer_forward_counted(pts_p, pts_g, n, n, counts, counts + 1, d1, d2,
                                                reinterpret_cast<int32_t*>(base + w.i1),
                                                reinterpret_cast<int32_t*>(base + w.i2), base + w.ch_ws,
                                                nvsf_chamfer_workspace_bytes(1, n, n), stream);
    if (st != NVSF_OK) return st;
    k_lidar_finalize<<<1, kFinBlock, 0, s>>>(stats, ssim_part, sg, sel, n, max_depth, fscore_threshold, d1, d2,
                                             counts, row);
    return nvsf_launch_status();
}

size_t nvsf_eval_points_workspace_bytes(uint32_t cap_p, uint32_t cap_g) {
    if (cap_p == 0 || cap_g == 0 || cap_p > INT32_MAX || cap_g > INT32_MAX) return 0;
    return points_ws(cap_p, cap_g).bytes;
}

int nvsf_eval_points(const float* pred, uint32_t cap_p, const int32_t* n_pred, const float* gt, uint32_t cap_g,
                     const int32_t* n_gt, float fscore_threshold, float* row, void* workspace, size_t workspace_bytes,
                     void* stream) {
    if (!pred || !n_pred || !gt || !n_gt || !row || !workspace || !aligned16(workspace)) return NVSF_E_INVALID;
    if (cap_p == 0 || cap_g == 0 || cap_p > INT32_MAX || cap_g > INT32_MAX || !(fscore_threshold >= 0.f))
        return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_eval_points_workspace_bytes(cap_p, cap_g)) return NVSF_E_WORKSPACE;
    const PointsWs w = points_ws(cap_p, cap_g);
    char* base = reinterpret_cast<char*>(workspace);
    float* d1 = reinterpret_cast<float*>(base + w.d1);
    float* d2 = reinterpret_cast<float*>(base + w.d2);
    const int st = nvsf_chamfer_forward_counted(pred, gt, cap_p, cap_g, n_pred, n_gt, d1, d2,
                                                reinterpret_cast<int32_t*>(base + w.i1),
                                                reinterpret_cast<int32_t*>(base + w.i2), base + w.ch_ws,
                                                nvsf_chamfer_workspace_bytes(1, cap_p, cap_g), stream);
    if (st != NVSF_OK) return st;
    k_points_finalize<<<1, kFinBlock, 0, (cudaStream_t)stream>>>(d1, d2, n_pred, cap_p, n_gt, cap_g, fscore_threshold,
                                                                 row);
    return nvsf_launch_status();
}

size_t nvsf_eval_camera_workspace_bytes(uint32_t H, uint32_t W) { return frame_ok(H, W) ? camera_ws(H, W).bytes : 0; }

int nvsf_eval_camera(const float* pred, const float* gt, uint32_t H, uint32_t W, float* row, void* workspace,
                     size_t workspace_bytes, void* stream) {
    if (!pred || !gt || !row || !workspace || !frame_ok(H, W) || !aligned16(workspace)) return NVSF_E_INVALID;
    if (workspace_bytes < nvsf_eval_camera_workspace_bytes(H, W)) return NVSF_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    const CameraWs w = camera_ws(H, W);
    char* base = reinterpret_cast<char*>(workspace);
    double* partial = reinterpret_cast<double*>(base + w.partial);
    double* ssim_part = reinterpret_cast<double*>(base + w.ssim);
    const size_t n = (size_t)H * W * 3;
    const uint32_t nblk = pixel_blocks(H * W);
    k_sq_err<<<nblk, kPixBlock, 0, s>>>(pred, gt, n, partial);
    const SsimGrid sg = ssim_grid(H, W, 3);
    if (sg.windows) k_ssim<<<sg.grid, kSsTX * kSsTY, 0, s>>>(pred, gt, H, W, 3, nullptr, 1.0, ssim_part);
    k_camera_finalize<<<1, kFinBlock, 0, s>>>(partial, nblk, n, ssim_part, sg, row);
    return nvsf_launch_status();
}

}  // extern "C"
