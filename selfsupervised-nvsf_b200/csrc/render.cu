// nvsf_b200 — uniform-sample renderer: alpha compositing fused with the colour heads (sm_100a).
//
// Replaces the tail of NeRFRenderer.run (reference nvsf/nerf/models/renderer_dynamic.py:181-237:
// deltas, alphas, cumprod weights, w > 1e-4 mask, masked colour query, weights_sum / depth / image
// accumulation, background) and NeRFNetwork.color (network_dynamic.py:290-332: Frequency / SH
// direction encoding, intensity + raydrop nets or colour net, sigmoid).
//
// One warp owns one ray.  The direction encoding is constant along a ray, so its contribution to
// the first layer of the head MLPs is computed once per ray (u = W1[:, dir] * enc(d)) and used to
// initialise the tensor-core accumulators; per sample only the 15 geometry features go through
// layer 1.  Transmittance is an exclusive product scan over 32-sample chunks (warp shuffles) with
// a running carry; chunks in which no sample passes the w > 1e-4 mask skip the heads entirely.
#include <algorithm>
#include <string>

#include "umma.cuh"

namespace {

constexpr int kRWarps = 4;
// resident CTAs per SM the register allocation is tuned for: 4 -> <= 128 registers (16 warps/SM,
// 24 bytes of spills) instead of 150 registers / 12 warps; the kernel is latency bound (ncu: stall
// `wait` + long_scoreboard at 14 % occupancy, profiles/r01_composite_v1_ncu_full.txt)
#ifndef NVSF_RENDER_MIN_CTAS
#define NVSF_RENDER_MIN_CTAS 4
#endif
constexpr int kGeoLd = kLdK16;  // 24 halves per staged geo row
constexpr int kWarpScratchBytes = 32 * kGeoLd * 2 + 2 * kHidden * 4 + kHeadDirMax * 4;

template <bool LIDAR>
constexpr size_t render_smem() {
    return (size_t)(LIDAR ? 2 : 1) * kHeadHalves * sizeof(__half) +
           (size_t)kRWarps * kWarpScratchBytes;
}

__device__ __forceinline__ float uniform_z2(float near, float far, uint32_t k, uint32_t S,
                                            const float* __restrict__ noise, size_t g) {
    const float step = 1.0f / (float)(S > 1 ? S - 1 : 1);
    const float lin = (k < S / 2) ? step * (float)k : 1.0f - step * (float)(S - 1 - k);
    float z = near + (far - near) * lin;
    if (noise) z = z + (__ldg(noise + g) - 0.5f) * ((far - near) / (float)S);
    return z;
}

__device__ __forceinline__ float sigmoidf_(float h) { return 1.0f / (1.0f + expf(-h)); }

template <bool LIDAR>
__global__ void __launch_bounds__(kRWarps * 32, NVSF_RENDER_MIN_CTAS)
k_render_composite(const __grid_constant__ nvsf_field_config_t cfg, const __half* __restrict__ mlp,
                   const float* __restrict__ rays_d, const float* __restrict__ nears,
                   const float* __restrict__ fars, const float* __restrict__ noise,
                   const float* __restrict__ sigma, const __half* __restrict__ geo, uint32_t N,
                   uint32_t S, float bg_color, float* __restrict__ depth_out,
                   float* __restrict__ image_out, float* __restrict__ ws_out,
                   float* __restrict__ weights_out, float* __restrict__ z_out,
                   float* __restrict__ rgbs_out /* [N*S,4] kept for the backward pass, or NULL */) {
    constexpr int NETS = LIDAR ? 2 : 1;
    constexpr int NDIR = LIDAR ? 72 : 16;
    constexpr int NCH = LIDAR ? 2 : 3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __half* Wsm = reinterpret_cast<__half*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned char* wscr = smem_raw + (size_t)NETS * kHeadHalves * sizeof(__half) +
                          (size_t)warp * kWarpScratchBytes;
    __half* geo_s = reinterpret_cast<__half*>(wscr);
    float* u_s = reinterpret_cast<float*>(wscr + 32 * kGeoLd * 2);
    float* enc_s = u_s + 2 * kHidden;

    block_copy16(Wsm, mlp + kHeadBase, NETS * kHeadHalves * (int)sizeof(__half) / 16, tid,
                 kRWarps * 32);
    __syncthreads();

    const int gq = lane >> 2, tq = lane & 3;
    const float kexp = cfg.active_sensor ? 2.0f : 1.0f;

    for (uint32_t r = blockIdx.x * kRWarps + warp; r < N; r += gridDim.x * kRWarps) {
        const float near = __ldg(nears + r), far = __ldg(fars + r);
        const float dx = __ldg(rays_d + (size_t)r * 3), dy = __ldg(rays_d + (size_t)r * 3 + 1),
                    dz = __ldg(rays_d + (size_t)r * 3 + 2);
        // ---- direction encoding (network_dynamic.py:310-311 / 319-320) ----
        __syncwarp();
        if (LIDAR) {
            // tcnn Frequency, 12 octaves: sin(2^k pi x + (j&1) pi/2), x = (d+1)/2
            for (int j = lane; j < NDIR; j += 32) {
                const int dim = j / 24, oct = (j >> 1) % 12;
                const float v = ((dim == 0 ? dx : (dim == 1 ? dy : dz)) + 1.0f) * 0.5f;
                enc_s[j] = sinpif(scalbnf(v, oct) + 0.5f * (float)(j & 1));
            }
        } else if (lane < 16) {
            // tcnn SphericalHarmonics degree 4 of 2*((d+1)/2)-1
            const float x = ((dx + 1.0f) * 0.5f) * 2.0f - 1.0f, y = ((dy + 1.0f) * 0.5f) * 2.0f - 1.0f,
                        z = ((dz + 1.0f) * 0.5f) * 2.0f - 1.0f;
            const float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
            float v;
            switch (lane) {
                case 0: v = 0.28209479177387814f; break;
                case 1: v = -0.48860251190291987f * y; break;
                case 2: v = 0.48860251190291987f * z; break;
                case 3: v = -0.48860251190291987f * x; break;
                case 4: v = 1.0925484305920792f * xy; break;
                case 5: v = -1.0925484305920792f * yz; break;
                case 6: v = 0.94617469575755997f * z2 - 0.31539156525251999f; break;
                case 7: v = -1.0925484305920792f * xz; break;
                case 8: v = 0.54627421529603959f * x2 - 0.54627421529603959f * y2; break;
                case 9: v = 0.59004358992664352f * y * (-3.0f * x2 + y2); break;
                case 10: v = 2.8906114426405538f * xy * z; break;
                case 11: v = 0.45704579946446572f * y * (1.0f - 5.0f * z2); break;
                case 12: v = 0.3731763325901154f * z * (5.0f * z2 - 3.0f); break;
                case 13: v = 0.45704579946446572f * x * (1.0f - 5.0f * z2); break;
                case 14: v = 1.4453057213202769f * z * (x2 - y2); break;
                default: v = 0.59004358992664352f * x * (-x2 + 3.0f * y2); break;
            }
            enc_s[lane] = v;
        }
        __syncwarp();
        // ---- per-ray part of layer 1: u[net][n] = sum_j W1[n][j] * enc[j] ----
#pragma unroll
        for (int net = 0; net < NETS; ++net) {
            const __half* W1d = Wsm + net * kHeadHalves + kHeadW1d;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int nrow = lane + 32 * h;
                float acc = 0.f;
                for (int j = 0; j < NDIR; j += 2) {
                    const float2 w = __half22float2(
                        *reinterpret_cast<const __half2*>(W1d + nrow * kHeadDirMax + j));
                    acc = fmaf(w.x, enc_s[j], acc);
                    acc = fmaf(w.y, enc_s[j + 1], acc);
                }
                u_s[net * kHidden + nrow] = acc;
            }
        }
        __syncwarp();

        float carry = 1.0f, ws = 0.f, dep = 0.f, img[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) img[c] = 0.f;

        for (uint32_t c0 = 0; c0 < S; c0 += 32) {
            const uint32_t i = c0 + lane;
            const bool in = i < S;
            const size_t g = (size_t)r * S + (in ? i : S - 1);
            const float z = uniform_z2(near, far, in ? i : S - 1, S, noise, g);
            float delta;
            if (i + 1 < S) delta = uniform_z2(near, far, i + 1, S, noise, g + 1) - z;
            else delta = (far - near) / (float)S;  // renderer_dynamic.py:160,182
            const float sg = in ? __ldg(sigma + g) : 0.f;
            const float alpha = in ? 1.0f - expf(((-kexp * delta) * cfg.density_scale) * sg) : 0.f;
            const float v = (1.0f - alpha) + 1e-15f;
            float incl = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float o = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl *= o;
            }
            float excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = 1.0f;
            const float T = carry * excl;
            carry *= __shfl_sync(0xffffffffu, incl, 31);
            const float w = in ? alpha * T : 0.f;
            ws += w;
            dep = fmaf(w, z, dep);
            if (weights_out && in) { weights_out[g] = w; z_out[g] = z; }
            const bool m = w > 1e-4f;  // renderer_dynamic.py:202
            if (__ballot_sync(0xffffffffu, m) == 0) {
                if (rgbs_out && in) *reinterpret_cast<float4*>(rgbs_out + g * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                continue;
            }

            // ---- heads on this 32-sample chunk ----
            {
                uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0;
                if (in) {
                    const uint4* src = reinterpret_cast<const uint4*>(geo + g * kGeo);
                    a0 = __ldg(src); a1 = __ldg(src + 1);
                    a0.x = (a0.x & 0xffff0000u) | kOneH;  // col 0: sigma logit -> the constant-1 padding input
                }
                uint4* dst = reinterpret_cast<uint4*>(geo_s + lane * kGeoLd);
                dst[0] = a0; dst[1] = a1;
            }
            __syncwarp();
            uint32_t a[2][1][4];
            load_a_frags<1>(geo_s, kGeoLd, a, lane);
            if (rgbs_out) {  // the staged geo rows are in registers now: reuse them to stage colours
                __syncwarp();
                reinterpret_cast<float4*>(geo_s)[lane] = make_float4(0.f, 0.f, 0.f, 0.f);
                __syncwarp();
            }
            const float wm = m ? w : 0.f;
            const float w0 = __shfl_sync(0xffffffffu, wm, gq), w1 = __shfl_sync(0xffffffffu, wm, gq + 8),
                        w2 = __shfl_sync(0xffffffffu, wm, gq + 16), w3 = __shfl_sync(0xffffffffu, wm, gq + 24);
#pragma unroll
            for (int net = 0; net < NETS; ++net) {
                const __half* Wn = Wsm + net * kHeadHalves;
                float acc[2][8][4];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float2 u = *reinterpret_cast<const float2*>(u_s + net * kHidden + 8 * j + 2 * tq);
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        acc[mt][j][0] = u.x; acc[mt][j][1] = u.y;
                        acc[mt][j][2] = u.x; acc[mt][j][3] = u.y;
                    }
                }
                warp_gemm_regA<1, 8>(a, Wn + kHeadW1g, kLdK16, acc, lane);
                uint32_t a2[2][4][4];
                relu_to_a<8>(acc, a2);
                zero_acc<8>(acc);
                warp_gemm_regA<4, 8>(a2, Wn + kHeadW2, kLdK64, acc, lane);
                relu_to_a<8>(acc, a2);
                float o[2][1][4];
                zero_acc<1>(o);
                warp_gemm_regA<4, 1>(a2, Wn + kHeadW3, kLdK64, o, lane);
                // colours of rows gq, gq+8, gq+16, gq+24; columns 2tq, 2tq+1 of the output layer
                const float s00 = sigmoidf_(o[0][0][0]), s01 = sigmoidf_(o[0][0][1]),
                            s10 = sigmoidf_(o[0][0][2]), s11 = sigmoidf_(o[0][0][3]),
                            s20 = sigmoidf_(o[1][0][0]), s21 = sigmoidf_(o[1][0][1]),
                            s30 = sigmoidf_(o[1][0][2]), s31 = sigmoidf_(o[1][0][3]);
                if (LIDAR) {
                    // h = [raydrop, intensity] (network_dynamic.py:317): slot 0 = intensity, 1 = raydrop
                    if (tq == 0) {
                        const float s = w0 * s00 + w1 * s10 + w2 * s20 + w3 * s30;
                        if (net == 0) img[1] += s; else img[0] += s;
                        if (rgbs_out) {
                            const int ch = net == 0 ? 1 : 0;
                            float* cs = reinterpret_cast<float*>(geo_s);  // [32][4] colour staging
                            cs[gq * 4 + ch] = w0 > 0.f ? s00 : 0.f;
                            cs[(gq + 8) * 4 + ch] = w1 > 0.f ? s10 : 0.f;
                            cs[(gq + 16) * 4 + ch] = w2 > 0.f ? s20 : 0.f;
                            cs[(gq + 24) * 4 + ch] = w3 > 0.f ? s30 : 0.f;
                        }
                    }
                } else {
                    if (tq == 0) {
                        img[0] += w0 * s00 + w1 * s10 + w2 * s20 + w3 * s30;
                        img[1] += w0 * s01 + w1 * s11 + w2 * s21 + w3 * s31;
                    } else if (tq == 1) {
                        img[2] += w0 * s00 + w1 * s10 + w2 * s20 + w3 * s30;
                    }
                    if (rgbs_out && tq < 2) {
                        const float z1 = tq == 0 ? 1.f : 0.f;  // output column 3 is padding
                        float2* cs = reinterpret_cast<float2*>(geo_s);  // [32][2 x float2] colour staging
                        cs[gq * 2 + tq] = make_float2(w0 > 0.f ? s00 : 0.f, w0 > 0.f ? s01 * z1 : 0.f);
                        cs[(gq + 8) * 2 + tq] = make_float2(w1 > 0.f ? s10 : 0.f, w1 > 0.f ? s11 * z1 : 0.f);
                        cs[(gq + 16) * 2 + tq] = make_float2(w2 > 0.f ? s20 : 0.f, w2 > 0.f ? s21 * z1 : 0.f);
                        cs[(gq + 24) * 2 + tq] = make_float2(w3 > 0.f ? s30 : 0.f, w3 > 0.f ? s31 * z1 : 0.f);
                    }
                }
            }
            __syncwarp();
            if (rgbs_out) {
                if (in) *reinterpret_cast<float4*>(rgbs_out + g * 4) = reinterpret_cast<const float4*>(geo_s)[lane];
                __syncwarp();
            }
        }
        // ---- reduce over the warp and write the ray ----
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            ws += __shfl_xor_sync(0xffffffffu, ws, d);
            dep += __shfl_xor_sync(0xffffffffu, dep, d);
#pragma unroll
            for (int c = 0; c < NCH; ++c) img[c] += __shfl_xor_sync(0xffffffffu, img[c], d);
        }
        if (lane == 0) {
            ws_out[r] = ws;
            depth_out[r] = dep;
#pragma unroll
            for (int c = 0; c < NCH; ++c)
                image_out[(size_t)r * NCH + c] = LIDAR ? img[c] : img[c] + (1.0f - ws) * bg_color;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// The same renderer with the head MLPs on the 5th-generation tensor cores (tcgen05.mma, TMEM).
//
// One CTA per SM, four independent warpgroups; a warpgroup owns a ray and walks it in tiles of 128
// samples (thread = sample = UMMA row = TMEM lane).  Per tile: transmittance by a 128-wide product
// scan (shuffles + one exchange through shared memory) with a carry; if any sample passes the
// w > 1e-4 mask (bar.red.or), the geo rows go into the swizzled K-major operand tile and the heads
// of BOTH LiDAR nets run as three MMA batches, the hidden activations going TMEM -> tcgen05.ld ->
// registers (+ per-ray direction term, relu, fp16) -> the operand tile:
//   D1 [128 x 64 NETS] = geo [128 x 16] W1g^T      1 x tcgen05.mma (N = 128 for LiDAR)
//   D2[net] [128 x 64] = H1[net] W2[net]^T         4 x tcgen05.mma per net
//   D3[net] [128 x 16] = H2[net] W3[net]^T         4 x tcgen05.mma per net
// The next tile's sigma / geo rows are loaded before the first wait, so they travel during the chain.
// ------------------------------------------------------------------------------------------------
using namespace umma;

constexpr int kCWG = 4;
constexpr int kCThreads = kCWG * kRows;
constexpr uint32_t kHOffW1 = 0;                            // [128 rows][128 B]: rows 64.. = net 1, K = 16
constexpr uint32_t kHOffW2 = kHOffW1 + 128 * 128;          // 2 x [64 rows][128 B]
constexpr uint32_t kHOffW3 = kHOffW2 + 2 * kHidden * 128;  // 2 x [16 rows][128 B] (rows >= n_out zero)
constexpr uint32_t kHImgBytes = kHOffW3 + 2 * 16 * 128;
constexpr uint32_t kCOffW1d = kHImgBytes;                  // fp16 [2][64][72]: direction columns of layer 1
constexpr uint32_t kCW1dBytes = 2 * kHidden * kHeadDirMax * 2;
constexpr uint32_t kCOffTiles = kCOffW1d + kCW1dBytes;
constexpr uint32_t kCTile = kRows * 128;                   // one [128 rows][128 B] operand tile
constexpr uint32_t kCScratchFloats = 256;                  // per warpgroup: enc[72] u[128] ptot[4] red[4][8]
static_assert(kHImgBytes % 1024 == 0 && kCOffTiles % 1024 == 0, "swizzled tiles start on 1024-byte boundaries");

template <bool LIDAR>
constexpr size_t composite_tc_smem() {
    return kCOffTiles + (size_t)kCWG * (LIDAR ? 2 : 1) * kCTile + kCWG * kCScratchFloats * 4 + 16 * kCWG + 16 + 1024;
}

// head weights (fp16 image of field.cu) -> swizzled K-major operand images
__global__ void k_pack_heads_tc(const __half* __restrict__ mlp, unsigned char* __restrict__ dst, int nets) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;  // one 16-byte chunk each
    const uint32_t per_net = kHidden * 2 + kHidden * 8 + 8 * 8;
    if (nets == 1 && i >= per_net && i < per_net + (uint32_t)kHidden * 4) {
        // camera workspaces: rows 64..127 of the layer-1 image (net 1 does not exist) hold the WHOLE
        // first layer of color_net, K = 32 = [SH-4 direction columns | geo columns], for k_color_tc
        const uint32_t k = i - per_net, r = k >> 2, c = k & 3;
        const __half* hm = mlp + kHeadBase;
        const uint4 v = c < 2 ? *reinterpret_cast<const uint4*>(hm + kHeadW1d + r * kHeadDirMax + c * 8)
                              : *reinterpret_cast<const uint4*>(hm + kHeadW1g + r * kLdK16 + (c - 2) * 8);
        *reinterpret_cast<uint4*>(dst + kHOffW1 + swz(kHidden + r, c)) = v;
        return;
    }
    if (i >= per_net * (uint32_t)nets) return;
    const uint32_t net = i / per_net, j = i - net * per_net;
    const __half* hm = mlp + kHeadBase + net * kHeadHalves;
    if (j < (uint32_t)kHidden * 2) {                       // W1g [64][16 of 24]
        const uint32_t r = j >> 1, c = j & 1;
        *reinterpret_cast<uint4*>(dst + kHOffW1 + swz(net * kHidden + r, c)) =
            *reinterpret_cast<const uint4*>(hm + kHeadW1g + r * kLdK16 + c * 8);
    } else if (j < (uint32_t)kHidden * 10) {               // W2 [64][64]
        const uint32_t k = j - kHidden * 2, r = k >> 3, c = k & 7;
        *reinterpret_cast<uint4*>(dst + kHOffW2 + net * (kHidden * 128) + swz(r, c)) =
            *reinterpret_cast<const uint4*>(hm + kHeadW2 + r * kLdK64 + c * 8);
    } else {                                               // W3 [8][64]
        const uint32_t k = j - kHidden * 10, r = k >> 3, c = k & 7;
        *reinterpret_cast<uint4*>(dst + kHOffW3 + net * (16 * 128) + swz(r, c)) =
            *reinterpret_cast<const uint4*>(hm + kHeadW3 + r * kLdK64 + c * 8);
    }
}

__device__ __forceinline__ float sh4_term(int k, float dx, float dy, float dz) {
    // tcnn SphericalHarmonics degree 4 of 2*((d+1)/2)-1 (same expressions as k_render_composite)
    const float x = ((dx + 1.0f) * 0.5f) * 2.0f - 1.0f, y = ((dy + 1.0f) * 0.5f) * 2.0f - 1.0f,
                z = ((dz + 1.0f) * 0.5f) * 2.0f - 1.0f;
    const float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
    switch (k) {
        case 0: return 0.28209479177387814f;
        case 1: return -0.48860251190291987f * y;
        case 2: return 0.48860251190291987f * z;
        case 3: return -0.48860251190291987f * x;
        case 4: return 1.0925484305920792f * xy;
        case 5: return -1.0925484305920792f * yz;
        case 6: return 0.94617469575755997f * z2 - 0.31539156525251999f;
        case 7: return -1.0925484305920792f * xz;
        case 8: return 0.54627421529603959f * x2 - 0.54627421529603959f * y2;
        case 9: return 0.59004358992664352f * y * (-3.0f * x2 + y2);
        case 10: return 2.8906114426405538f * xy * z;
        case 11: return 0.45704579946446572f * y * (1.0f - 5.0f * z2);
        case 12: return 0.3731763325901154f * z * (5.0f * z2 - 3.0f);
        case 13: return 0.45704579946446572f * x * (1.0f - 5.0f * z2);
        case 14: return 1.4453057213202769f * z * (x2 - y2);
        default: return 0.59004358992664352f * x * (-x2 + 3.0f * y2);
    }
}

// H[net] row `t` = fp16(relu(D[:, 0..63] (+ u))) from this thread's TMEM lane into the operand tile
template <bool ADD_U>
__device__ __forceinline__ void hidden_to_tile(uint32_t taddr, const float* __restrict__ u,
                                               unsigned char* tile, uint32_t t) {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        uint32_t v[32];
        tmem_ld32(taddr + q * 32, v);          // 32 columns per load
        tmem_ld_wait();
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[8 * h + i]);
            if (ADD_U) {
                const float4 ua = *reinterpret_cast<const float4*>(u + q * 32 + 8 * h);
                const float4 ub = *reinterpret_cast<const float4*>(u + q * 32 + 8 * h + 4);
                f[0] += ua.x; f[1] += ua.y; f[2] += ua.z; f[3] += ua.w;
                f[4] += ub.x; f[5] += ub.y; f[6] += ub.z; f[7] += ub.w;
            }
            uint4 o;   // relu fused into the fp32 -> fp16x2 conversion
            o.x = pack_half2_relu(f[0], f[1]); o.y = pack_half2_relu(f[2], f[3]);
            o.z = pack_half2_relu(f[4], f[5]); o.w = pack_half2_relu(f[6], f[7]);
            *reinterpret_cast<uint4*>(tile + swz(t, 4 * q + h)) = o;
        }
    }
}

template <bool LIDAR>
__global__ void __launch_bounds__(kCThreads, 1)
k_composite_tc(const __grid_constant__ nvsf_field_config_t cfg, const unsigned char* __restrict__ wimg,
               const __half* __restrict__ mlp, const float* __restrict__ rays_d,
               const float* __restrict__ nears, const float* __restrict__ fars,
               const float* __restrict__ noise, const float* __restrict__ sigma,
               const __half* __restrict__ geo, uint32_t N, uint32_t S, float bg_color,
               float* __restrict__ depth_out, float* __restrict__ image_out, float* __restrict__ ws_out,
               float* __restrict__ weights_out, float* __restrict__ z_out, float* __restrict__ rgbs_out) {
    constexpr int NETS = LIDAR ? 2 : 1;
    constexpr int NDIR = LIDAR ? 72 : 16;
    constexpr int NCH = LIDAR ? 2 : 3;
    constexpr uint32_t kCols = NETS * kHidden;             // TMEM columns of one warpgroup
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* sm = smem_raw + (base - raw);
    const uint32_t tid = threadIdx.x, wg = tid >> 7, t = tid & 127u, lane = tid & 31u, wq = (tid >> 5) & 3u;
    constexpr uint32_t kOffScr = kCOffTiles + kCWG * NETS * kCTile;
    constexpr uint32_t kOffBarC = kOffScr + kCWG * kCScratchFloats * 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBarC + 16 * kCWG);
    float* scr = reinterpret_cast<float*>(sm + kOffScr) + wg * kCScratchFloats;
    float* enc_s = scr;            // [72]
    float* u_s = scr + 72;         // [NETS * 64]  (16-byte aligned: 72 * 4 = 288)
    float* ptot = scr + 200;       // [4]
    float* red = scr + 208;        // [4][8]
    const __half* W1d = reinterpret_cast<const __half*>(sm + kCOffW1d);

    for (uint32_t i = tid; i < kHImgBytes / 16; i += kCThreads)
        reinterpret_cast<uint4*>(sm)[i] = __ldg(reinterpret_cast<const uint4*>(wimg) + i);
    for (int net = 0; net < NETS; ++net)
        for (uint32_t i = tid; i < (uint32_t)kHidden * kHeadDirMax / 8; i += kCThreads)
            reinterpret_cast<uint4*>(sm + kCOffW1d)[net * (kHidden * kHeadDirMax / 8) + i] =
                __ldg(reinterpret_cast<const uint4*>(mlp + kHeadBase + net * kHeadHalves + kHeadW1d) + i);
    if (tid < (uint32_t)(2 * kCWG)) mbar_init(base + kOffBarC + 8 * tid, 1);
    if (tid < 32) {
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(
                         smem_u32(tmem_slot)),
                     "r"((uint32_t)(kCWG * kCols))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tcol = tmem + wg * kCols;
    const uint32_t tlane = tcol + ((wq * 32u) << 16);
    const uint32_t tiles = base + kCOffTiles + wg * NETS * kCTile;
    unsigned char* tileg = sm + kCOffTiles + wg * NETS * kCTile;
    const uint32_t bar = base + kOffBarC + 16 * wg;   // one mbarrier per net
    constexpr uint32_t kIdesc2 = umma_idesc(kRows, kHidden), kIdesc3 = umma_idesc(kRows, 16);
    const float kexp = cfg.active_sensor ? 2.0f : 1.0f;
    uint32_t phase = 0;

    for (uint32_t r = blockIdx.x * kCWG + wg; r < N; r += gridDim.x * kCWG) {
        const float near = __ldg(nears + r), far = __ldg(fars + r);
        const float dx = __ldg(rays_d + (size_t)r * 3), dy = __ldg(rays_d + (size_t)r * 3 + 1),
                    dz = __ldg(rays_d + (size_t)r * 3 + 2);
        // first tile's rows
        float sg = 0.f;
        uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0;
        if (t < S) {
            const size_t g = (size_t)r * S + t;
            sg = __ldg(sigma + g);
            a0 = __ldg(reinterpret_cast<const uint4*>(geo + g * kGeo));
            a1 = __ldg(reinterpret_cast<const uint4*>(geo + g * kGeo) + 1);
        }
        wg_barrier(wg);  // the previous ray's readers of enc / u / red are done
        if (LIDAR) {
            if (t < (uint32_t)NDIR) {  // tcnn Frequency, 12 octaves: sin(2^k pi x + (j&1) pi/2), x = (d+1)/2
                const int dim = t / 24, oct = (t >> 1) % 12;
                const float v = ((dim == 0 ? dx : (dim == 1 ? dy : dz)) + 1.0f) * 0.5f;
                enc_s[t] = sinpif(scalbnf(v, oct) + 0.5f * (float)(t & 1));
            }
        } else if (t < 16) {
            enc_s[t] = sh4_term((int)t, dx, dy, dz);
        }
        wg_barrier(wg);
        if (t < (uint32_t)(NETS * kHidden)) {  // u[net][n] = sum_j W1[n][dir j] * enc[j]
            const __half* wrow = W1d + (size_t)t * kHeadDirMax;
            float acc = 0.f;
            for (int j = 0; j < NDIR; j += 2) {
                const float2 w = __half22float2(*reinterpret_cast<const __half2*>(wrow + j));
                acc = fmaf(w.x, enc_s[j], acc);
                acc = fmaf(w.y, enc_s[j + 1], acc);
            }
            u_s[t] = acc;
        }
        float carry = 1.0f, ws = 0.f, dep = 0.f, img[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) img[c] = 0.f;

        for (uint32_t c0 = 0; c0 < S; c0 += kRows) {
            const uint32_t i = c0 + t;
            const bool in = i < S;
            const size_t g = (size_t)r * S + (in ? i : S - 1);
            const float z = uniform_z2(near, far, in ? i : S - 1, S, noise, g);
            float delta;
            if (i + 1 < S) delta = uniform_z2(near, far, i + 1, S, noise, g + 1) - z;
            else delta = (far - near) / (float)S;  // renderer_dynamic.py:160,182
            const float alpha = in ? 1.0f - expf(((-kexp * delta) * cfg.density_scale) * sg) : 0.f;
            const float v = (1.0f - alpha) + 1e-15f;
            float incl = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float o = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= (uint32_t)d) incl *= o;
            }
            float excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = 1.0f;
            if (lane == 31) ptot[wq] = incl;
            wg_barrier(wg);
            const float p0 = ptot[0], p1 = ptot[1], p2 = ptot[2], p3 = ptot[3];
            const float pre = wq == 0 ? 1.0f : (wq == 1 ? p0 : (wq == 2 ? p0 * p1 : (p0 * p1) * p2));
            const float T = (carry * pre) * excl;
            carry *= ((p0 * p1) * p2) * p3;
            const float w = in ? alpha * T : 0.f;
            ws += w;
            dep = fmaf(w, z, dep);
            if (weights_out && in) { weights_out[g] = w; z_out[g] = z; }
            const bool m = w > 1e-4f;  // renderer_dynamic.py:202
            // geo rows of this tile -> operand tile (it aliases the LAST net's hidden tile, see the
            // hazards below); then the next tile's rows start travelling
            a0.x = (a0.x & 0xffff0000u) | kOneH;  // col 0: sigma logit -> the constant-1 padding input (weight = pad-column sum)
            *reinterpret_cast<uint4*>(tileg + (NETS - 1) * kCTile + swz(t, 0)) = a0;
            *reinterpret_cast<uint4*>(tileg + (NETS - 1) * kCTile + swz(t, 1)) = a1;
            {
                const uint32_t in2 = c0 + kRows + t;
                sg = 0.f; a0 = make_uint4(0, 0, 0, 0); a1 = a0;
                if (in2 < S) {
                    const size_t g2 = (size_t)r * S + in2;
                    sg = __ldg(sigma + g2);
                    a0 = __ldg(reinterpret_cast<const uint4*>(geo + g2 * kGeo));
                    a1 = __ldg(reinterpret_cast<const uint4*>(geo + g2 * kGeo) + 1);
                }
            }
            fence_async_smem();
            tc_fence_before();
            // one barrier: the tile rows are complete, every thread has read ptot, and the OR of the mask
            if (!wg_any(wg, m)) {
                if (rgbs_out && in) *reinterpret_cast<float4*>(rgbs_out + g * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                continue;
            }
            // The two LiDAR nets are independent chains with their own mbarrier: while one net's MMA
            // batch is in flight the warpgroup runs the other net's epilogue.  Hazards: H[0] is
            // written while MMA1(net 1) may still read the geo tile -> the geo tile lives in H[1];
            // H[1] is written after bar 1, whose commit follows both layer-1 MMAs.
            if (t == 0) {
                tc_fence_after();
#pragma unroll
                for (uint32_t net = 0; net < (uint32_t)NETS; ++net) {
                    umma_f16(tcol + net * kHidden, umma_desc(tiles + (NETS - 1) * kCTile),
                             umma_desc(base + kHOffW1 + net * (kHidden * 128)), kIdesc2, 0u);
                    umma_commit(bar + 8 * net);
                }
            }
            // H1 = relu(D1 + u) -> D2 = H1 W2^T
#pragma unroll
            for (uint32_t net = 0; net < (uint32_t)NETS; ++net) {
                mbar_wait(bar + 8 * net, phase);
                tc_fence_after();
                hidden_to_tile<true>(tlane + net * kHidden, u_s + net * kHidden, tileg + net * kCTile, t);
                fence_async_smem();
                tc_fence_before();
                wg_barrier(wg);
                if (t == 0) {
                    tc_fence_after();
#pragma unroll
                    for (uint32_t k = 0; k < 4; ++k)
                        umma_f16(tcol + net * kHidden, umma_desc(tiles + net * kCTile + k * 32),
                                 umma_desc(base + kHOffW2 + net * (kHidden * 128) + k * 32), kIdesc2, k);
                    umma_commit(bar + 8 * net);
                }
            }
            phase ^= 1u;
            // H2 = relu(D2) -> D3 = H2 W3^T (16 columns at the start of the net's column block)
#pragma unroll
            for (uint32_t net = 0; net < (uint32_t)NETS; ++net) {
                mbar_wait(bar + 8 * net, phase);
                tc_fence_after();
                hidden_to_tile<false>(tlane + net * kHidden, nullptr, tileg + net * kCTile, t);
                fence_async_smem();
                tc_fence_before();
                wg_barrier(wg);
                if (t == 0) {
                    tc_fence_after();
#pragma unroll
                    for (uint32_t k = 0; k < 4; ++k)
                        umma_f16(tcol + net * kHidden, umma_desc(tiles + net * kCTile + k * 32),
                                 umma_desc(base + kHOffW3 + net * (16 * 128) + k * 32), kIdesc3, k);
                    umma_commit(bar + 8 * net);
                }
            }
            phase ^= 1u;
#pragma unroll
            for (uint32_t net = 0; net < (uint32_t)NETS; ++net) mbar_wait(bar + 8 * net, phase);
            phase ^= 1u;
            tc_fence_after();
            // colours of this thread's sample
            const float wm = m ? w : 0.f;
            float4 col = make_float4(0.f, 0.f, 0.f, 0.f);
            {
                uint32_t o[16];
                tmem_ld16(tlane, o);
                tmem_ld_wait();
                if (LIDAR) {
                    // h = [raydrop, intensity] (network_dynamic.py:317): net 0 = intensity -> channel 1
                    uint32_t o2[16];
                    tmem_ld16(tlane + kHidden, o2);
                    tmem_ld_wait();
                    const float s_int = sigmoidf_(__uint_as_float(o[0])), s_drop = sigmoidf_(__uint_as_float(o2[0]));
                    img[1] += wm * s_int;
                    img[0] += wm * s_drop;
                    if (m) col = make_float4(s_drop, s_int, 0.f, 0.f);
                } else {
                    const float s0 = sigmoidf_(__uint_as_float(o[0])), s1 = sigmoidf_(__uint_as_float(o[1])),
                                s2 = sigmoidf_(__uint_as_float(o[2]));
                    img[0] += wm * s0; img[1] += wm * s1; img[2] += wm * s2;
                    if (m) col = make_float4(s0, s1, s2, 0.f);
                }
            }
            if (rgbs_out && in) *reinterpret_cast<float4*>(rgbs_out + g * 4) = col;
            tc_fence_before();
        }
        // ---- reduce over the warpgroup and write the ray ----
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            ws += __shfl_xor_sync(0xffffffffu, ws, d);
            dep += __shfl_xor_sync(0xffffffffu, dep, d);
#pragma unroll
            for (int c = 0; c < NCH; ++c) img[c] += __shfl_xor_sync(0xffffffffu, img[c], d);
        }
        if (lane == 0) {
            red[wq * 8 + 0] = ws; red[wq * 8 + 1] = dep;
#pragma unroll
            for (int c = 0; c < NCH; ++c) red[wq * 8 + 2 + c] = img[c];
        }
        wg_barrier(wg);
        if (t == 0) {
            const float wsum = ((red[0] + red[8]) + red[16]) + red[24];
            ws_out[r] = wsum;
            depth_out[r] = ((red[1] + red[9]) + red[17]) + red[25];
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                const float v = ((red[2 + c] + red[10 + c]) + red[18 + c]) + red[26 + c];
                image_out[(size_t)r * NCH + c] = LIDAR ? v : v + (1.0f - wsum) * bg_color;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (tid < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem),
                     "r"((uint32_t)(kCWG * kCols))
                     : "memory");
}

// ---- eight warpgroups per CTA, nets one after the other (option heads_tc = 2) --------------------------
// k_composite_tc keeps four tile contexts per SM (TMEM: 4 x 128 columns, 512 threads x 123 registers) and
// ncu shows 49 % of its issue slots empty: 27 % of the warp samples spin on the MMA mbarriers, 17 % wait at
// warpgroup barriers — the serial issue -> commit -> epilogue chain of a tile is exposed.  This form trades the
// overlap of the two LiDAR nets inside a warpgroup for twice the warpgroups: a warpgroup owns 64 TMEM columns and
// ONE operand tile and runs net 0 then net 1 of a tile through them (the geo rows stay in registers and are
// written into the tile again for net 1), so eight independent chains per SM come from 32 warps instead of 16.
// The per-ray direction term u[net][n] = W1[n][dir] . enc(d) enters layer 1 through the tensor core as well: the geo
// operand's column 0 is the constant 1 (tcnn's input padding), so D1 = geo W1g^T + geo U^T with U[n][0] = u[n] and
// zeros elsewhere adds u to every row of the tile.  U is a per-warpgroup [64][16] fp16 image in the un-swizzled
// K-major core-matrix layout (8 rows x 16 B contiguous; row groups SBO = 256 B apart, the two K chunks LBO = 128 B
// apart): 2 KB per net, 64 halves rewritten per ray.  The layer-1 epilogue loses its 64 FADD + 16 LDS per thread.
constexpr uint32_t kCUImg = 2048;
__device__ __forceinline__ uint64_t umma_desc_k_noswz(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(lbo >> 4) << 16;
    d |= (uint64_t)(sbo >> 4) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
// 4 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&v)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
                 : "r"(taddr)
                 : "memory");
}

template <int W>
constexpr size_t composite_tc8_smem() {
    return kCOffTiles + (size_t)W * kCTile + W * kCScratchFloats * 4 + (size_t)W * 2 * kCUImg + 8 * W + 16 + 1024;
}

// H row `t` = fp16(relu(D[:, 0..63] (+ u))) in 16-column steps (64-register budget)
template <bool ADD_U>
__device__ __forceinline__ void hidden_to_tile16(uint32_t taddr, const float* __restrict__ u,
                                                 unsigned char* tile, uint32_t t) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint32_t v[16];
        tmem_ld16(taddr + q * 16, v);
        tmem_ld_wait();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[8 * h + i]);
            if (ADD_U) {
                const float4 ua = *reinterpret_cast<const float4*>(u + q * 16 + 8 * h);
                const float4 ub = *reinterpret_cast<const float4*>(u + q * 16 + 8 * h + 4);
                f[0] += ua.x; f[1] += ua.y; f[2] += ua.z; f[3] += ua.w;
                f[4] += ub.x; f[5] += ub.y; f[6] += ub.z; f[7] += ub.w;
            }
            uint4 o;
            o.x = pack_half2_relu(f[0], f[1]); o.y = pack_half2_relu(f[2], f[3]);
            o.z = pack_half2_relu(f[4], f[5]); o.w = pack_half2_relu(f[6], f[7]);
            *reinterpret_cast<uint4*>(tile + swz(t, 2 * q + h)) = o;
        }
    }
}

template <bool LIDAR, int W>
__global__ void __launch_bounds__(W * kRows, 1)
k_composite_tc8(const __grid_constant__ nvsf_field_config_t cfg, const unsigned char* __restrict__ wimg,
                const __half* __restrict__ mlp, const float* __restrict__ rays_d,
                const float* __restrict__ nears, const float* __restrict__ fars,
                const float* __restrict__ noise, const float* __restrict__ sigma,
                const __half* __restrict__ geo, uint32_t N, uint32_t S, float bg_color,
                float* __restrict__ depth_out, float* __restrict__ image_out, float* __restrict__ ws_out,
                float* __restrict__ weights_out, float* __restrict__ z_out, float* __restrict__ rgbs_out) {
    constexpr int NETS = LIDAR ? 2 : 1;
    constexpr int NDIR = LIDAR ? 72 : 16;
    constexpr int NCH = LIDAR ? 2 : 3;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* sm = smem_raw + (base - raw);
    const uint32_t tid = threadIdx.x, wg = tid >> 7, t = tid & 127u, lane = tid & 31u, wq = (tid >> 5) & 3u;
    constexpr uint32_t kOffScr = kCOffTiles + W * kCTile;
    constexpr uint32_t kOffU = kOffScr + W * kCScratchFloats * 4;           // [W][2] U images
    constexpr uint32_t kOffBarC = kOffU + W * 2 * kCUImg;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBarC + 8 * W);
    float* scr = reinterpret_cast<float*>(sm + kOffScr) + wg * kCScratchFloats;
    float* enc_s = scr;            // [72]
    float* ptot = scr + 200;       // [4]
    float* red = scr + 208;        // [4][8]
    const __half* W1d = reinterpret_cast<const __half*>(sm + kCOffW1d);

    for (uint32_t i = tid; i < kHImgBytes / 16; i += (uint32_t)(W * kRows))
        reinterpret_cast<uint4*>(sm)[i] = __ldg(reinterpret_cast<const uint4*>(wimg) + i);
    for (int net = 0; net < NETS; ++net)
        for (uint32_t i = tid; i < (uint32_t)kHidden * kHeadDirMax / 8; i += (uint32_t)(W * kRows))
            reinterpret_cast<uint4*>(sm + kCOffW1d)[net * (kHidden * kHeadDirMax / 8) + i] =
                __ldg(reinterpret_cast<const uint4*>(mlp + kHeadBase + net * kHeadHalves + kHeadW1d) + i);
    for (uint32_t i = tid; i < (uint32_t)(W * 2 * kCUImg / 16); i += (uint32_t)(W * kRows))
        reinterpret_cast<uint4*>(sm + kOffU)[i] = make_uint4(0, 0, 0, 0);
    if (tid < (uint32_t)W) mbar_init(base + kOffBarC + 8 * tid, 1);
    if (tid < 32) {
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(
                         smem_u32(tmem_slot)),
                     "r"((uint32_t)512)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tcol = tmem + wg * kHidden;
    const uint32_t tlane = tcol + ((wq * 32u) << 16);
    const uint32_t tile_a = base + kCOffTiles + wg * kCTile;
    unsigned char* tileg = sm + kCOffTiles + wg * kCTile;
    const uint32_t bar = base + kOffBarC + 8 * wg;
    constexpr uint32_t kIdesc2 = umma_idesc(kRows, kHidden), kIdesc3 = umma_idesc(kRows, 16);
    const float kexp = cfg.active_sensor ? 2.0f : 1.0f;
    uint32_t phase = 0;

    for (uint32_t r = blockIdx.x * W + wg; r < N; r += gridDim.x * W) {
        const float near = __ldg(nears + r), far = __ldg(fars + r);
        float sg = 0.f;
        uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0;
        if (t < S) {
            const size_t g = (size_t)r * S + t;
            sg = __ldg(sigma + g);
            a0 = __ldg(reinterpret_cast<const uint4*>(geo + g * kGeo));
            a1 = __ldg(reinterpret_cast<const uint4*>(geo + g * kGeo) + 1);
        }
        wg_barrier(wg);  // the previous ray's readers of enc / u / red are done
        {
            const float dx = __ldg(rays_d + (size_t)r * 3), dy = __ldg(rays_d + (size_t)r * 3 + 1),
                        dz = __ldg(rays_d + (size_t)r * 3 + 2);
            if (LIDAR) {
                if (t < (uint32_t)NDIR) {  // tcnn Frequency, 12 octaves: sin(2^k pi x + (j&1) pi/2), x = (d+1)/2
                    const int dim = t / 24, oct = (t >> 1) % 12;
                    const float v = ((dim == 0 ? dx : (dim == 1 ? dy : dz)) + 1.0f) * 0.5f;
                    enc_s[t] = sinpif(scalbnf(v, oct) + 0.5f * (float)(t & 1));
                }
            } else if (t < 16) {
                enc_s[t] = sh4_term((int)t, dx, dy, dz);
            }
        }
        wg_barrier(wg);
        if (t < (uint32_t)(NETS * kHidden)) {  // u[net][n] = sum_j W1[n][dir j] * enc[j]
            const __half* wrow = W1d + (size_t)t * kHeadDirMax;
            float acc = 0.f;
            for (int j = 0; j < NDIR; j += 2) {
                const float2 w = __half22float2(*reinterpret_cast<const __half2*>(wrow + j));
                acc = fmaf(w.x, enc_s[j], acc);
                acc = fmaf(w.y, enc_s[j + 1], acc);
            }
            // U[net][n][0] = u: row n = (group n / 8, row n % 8) of the core-matrix layout
            const uint32_t net = t >> 6, n = t & 63u;
            *reinterpret_cast<__half*>(sm + kOffU + (wg * 2 + net) * kCUImg + (n >> 3) * 256 + (n & 7u) * 16) =
                __float2half_rn(acc);
        }
        float carry = 1.0f, ws = 0.f, dep = 0.f, img[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) img[c] = 0.f;

        for (uint32_t c0 = 0; c0 < S; c0 += kRows) {
            const uint32_t i = c0 + t;
            const bool in = i < S;
            const size_t g = (size_t)r * S + (in ? i : S - 1);
            const float z = uniform_z2(near, far, in ? i : S - 1, S, noise, g);
            float delta;
            if (i + 1 < S) delta = uniform_z2(near, far, i + 1, S, noise, g + 1) - z;
            else delta = (far - near) / (float)S;  // renderer_dynamic.py:160,182
            const float alpha = in ? 1.0f - expf(((-kexp * delta) * cfg.density_scale) * sg) : 0.f;
            const float v = (1.0f - alpha) + 1e-15f;
            float incl = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float o = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= (uint32_t)d) incl *= o;
            }
            float excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = 1.0f;
            if (lane == 31) ptot[wq] = incl;
            wg_barrier(wg);
            const float p0 = ptot[0], p1 = ptot[1], p2 = ptot[2], p3 = ptot[3];
            const float pre = wq == 0 ? 1.0f : (wq == 1 ? p0 : (wq == 2 ? p0 * p1 : (p0 * p1) * p2));
            const float T = (carry * pre) * excl;
            carry *= ((p0 * p1) * p2) * p3;
            const float w = in ? alpha * T : 0.f;
            ws += w;
            dep = fmaf(w, z, dep);
            if (weights_out && in) { weights_out[g] = w; z_out[g] = z; }
            const bool m = w > 1e-4f;  // renderer_dynamic.py:202
            a0.x = (a0.x & 0xffff0000u) | kOneH;  // col 0: sigma logit -> the constant-1 padding input
            // one barrier: every thread has read ptot, and the OR of the mask
            const bool any = wg_any(wg, m);
            float4 col = make_float4(0.f, 0.f, 0.f, 0.f);
            if (any) {
                const float wm = m ? w : 0.f;
#pragma unroll
                for (uint32_t net = 0; net < (uint32_t)NETS; ++net) {
                    // geo rows -> chunks 0, 1 of the tile (for net 1 again: H2 of net 0 has overwritten them; the
                    // layer-3 MMA that read H2 has committed, see the wait below)
                    *reinterpret_cast<uint4*>(tileg + swz(t, 0)) = a0;
                    *reinterpret_cast<uint4*>(tileg + swz(t, 1)) = a1;
                    fence_async_smem();
                    tc_fence_before();
                    wg_barrier(wg);
                    if (t == 0) {
                        tc_fence_after();
                        umma_f16(tcol, umma_desc(tile_a), umma_desc(base + kHOffW1 + net * (kHidden * 128)), kIdesc2, 0u);
                        umma_f16(tcol, umma_desc(tile_a),
                                 umma_desc_k_noswz(base + kOffU + (wg * 2 + net) * kCUImg, 128u, 256u), kIdesc2, 1u);
                        umma_commit(bar);
                    }
                    if (net == (uint32_t)NETS - 1) {   // the next tile's rows start travelling
                        const uint32_t in2 = c0 + kRows + t;
                        sg = 0.f; a0 = make_uint4(0, 0, 0, 0); a1 = a0;
                        if (in2 < S) {
                            const size_t g2 = (size_t)r * S + in2;
                            sg = __ldg(sigma + g2);
                            a0 = __ldg(reinterpret_cast<const uint4*>(geo + g2 * kGeo));
                            a1 = __ldg(reinterpret_cast<const uint4*>(geo + g2 * kGeo) + 1);
                        }
                    }
                    // H1 = relu(D1 + u) -> D2 = H1 W2^T
                    mbar_wait(bar, phase); phase ^= 1u;
                    tc_fence_after();
                    hidden_to_tile16<false>(tlane, nullptr, tileg, t);
                    fence_async_smem();
                    tc_fence_before();
                    wg_barrier(wg);
                    if (t == 0) {
                        tc_fence_after();
#pragma unroll
                        for (uint32_t k = 0; k < 4; ++k)
                            umma_f16(tcol, umma_desc(tile_a + k * 32),
                                     umma_desc(base + kHOffW2 + net * (kHidden * 128) + k * 32), kIdesc2, k);
                        umma_commit(bar);
                    }
                    // H2 = relu(D2) -> D3 = H2 W3^T (16 columns)
                    mbar_wait(bar, phase); phase ^= 1u;
                    tc_fence_after();
                    hidden_to_tile16<false>(tlane, nullptr, tileg, t);
                    fence_async_smem();
                    tc_fence_before();
                    wg_barrier(wg);
                    if (t == 0) {
                        tc_fence_after();
#pragma unroll
                        for (uint32_t k = 0; k < 4; ++k)
                            umma_f16(tcol, umma_desc(tile_a + k * 32),
                                     umma_desc(base + kHOffW3 + net * (16 * 128) + k * 32), kIdesc3, k);
                        umma_commit(bar);
                    }
                    mbar_wait(bar, phase); phase ^= 1u;
                    tc_fence_after();
                    uint32_t o[4];
                    tmem_ld4(tlane, o);
                    tmem_ld_wait();
                    tc_fence_before();
                    if (LIDAR) {
                        // h = [raydrop, intensity] (network_dynamic.py:317): net 0 = intensity -> channel 1
                        const float sv = sigmoidf_(__uint_as_float(o[0]));
                        if (net == 0) { img[1] += wm * sv; if (m) col.y = sv; }
                        else { img[0] += wm * sv; if (m) col.x = sv; }
                    } else {
                        const float s0 = sigmoidf_(__uint_as_float(o[0])), s1 = sigmoidf_(__uint_as_float(o[1])),
                                    s2 = sigmoidf_(__uint_as_float(o[2]));
                        img[0] += wm * s0; img[1] += wm * s1; img[2] += wm * s2;
                        if (m) col = make_float4(s0, s1, s2, 0.f);
                    }
                }
            } else {
                const uint32_t in2 = c0 + kRows + t;
                sg = 0.f; a0 = make_uint4(0, 0, 0, 0); a1 = a0;
                if (in2 < S) {
                    const size_t g2 = (size_t)r * S + in2;
                    sg = __ldg(sigma + g2);
                    a0 = __ldg(reinterpret_cast<const uint4*>(geo + g2 * kGeo));
                    a1 = __ldg(reinterpret_cast<const uint4*>(geo + g2 * kGeo) + 1);
                }
            }
            if (rgbs_out && in) *reinterpret_cast<float4*>(rgbs_out + g * 4) = col;
        }
        // ---- reduce over the warpgroup and write the ray ----
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            ws += __shfl_xor_sync(0xffffffffu, ws, d);
            dep += __shfl_xor_sync(0xffffffffu, dep, d);
#pragma unroll
            for (int c = 0; c < NCH; ++c) img[c] += __shfl_xor_sync(0xffffffffu, img[c], d);
        }
        if (lane == 0) {
            red[wq * 8 + 0] = ws; red[wq * 8 + 1] = dep;
#pragma unroll
            for (int c = 0; c < NCH; ++c) red[wq * 8 + 2 + c] = img[c];
        }
        wg_barrier(wg);
        if (t == 0) {
            const float wsum = ((red[0] + red[8]) + red[16]) + red[24];
            ws_out[r] = wsum;
            depth_out[r] = ((red[1] + red[9]) + red[17]) + red[25];
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                const float v = ((red[2 + c] + red[10 + c]) + red[18 + c]) + red[26 + c];
                image_out[(size_t)r * NCH + c] = LIDAR ? v : v + (1.0f - wsum) * bg_color;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (tid < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem),
                     "r"((uint32_t)512)
                     : "memory");
}

// ---- hidden activations as the A operand FROM TENSOR MEMORY (option heads_tc = 6) ----------------------
// ncu on k_composite_tc8 (profiles/r02_composite_tc8_ncu.txt): l1tex 67 %, tensor pipe 25 %, and neither twice the
// warpgroups, nor 40 % fewer epilogue instructions, nor half the TMEM reads moved its 2.65 ms: what a tile costs is
// shared-memory bandwidth — 16 KB of fp16 activations written per layer (STS) and the MMA reading its A operand
// back (M128 x K16 = 4 KB of A per 32-cycle N = 64 instruction: 192 B/clk asked of a 128 B/clk pipe), about
// 172 KB per 128-sample LiDAR tile.  Here the activations never touch shared memory: a thread reads its
// accumulator row (TMEM lane = sample), applies relu, packs to fp16 and stores it back into TMEM IN PLACE
// (tcgen05.st; packed column j = elements 2j, 2j+1, which the thread has already consumed), and the next layer's
// tcgen05.mma takes A from tensor memory (the .ts form: [d_tmem], [a_tmem], b_desc).  Shared memory keeps only
// the weights (B operands), a 4 KB un-swizzled geo tile and the 2 KB direction image per net: 52 KB per tile.
// TMEM per warpgroup, 96 columns:  D1 [0,64) -> H1 packed in place [0,32) -> D2 [32,96) -> H2 packed in place
// [32,64) -> D3 [0,16).  Five warpgroups (480 columns, 640 threads x 96 registers), nets one after the other.
constexpr int kTsWG = 5;
constexpr uint32_t kTsCols = 96;
constexpr uint32_t kTsGeoTile = 4096;   // [128 rows][16 halves], un-swizzled K-major core matrices
constexpr size_t composite_ts_smem() {
    return kCOffTiles + (size_t)kTsWG * (kTsGeoTile + 2 * kCUImg + kCScratchFloats * 4) + 8 * kTsWG + 16 + 1024;
}
template <bool LIDAR>
__global__ void __launch_bounds__(kTsWG * kRows, 1)
k_composite_ts(const __grid_constant__ nvsf_field_config_t cfg, const unsigned char* __restrict__ wimg,
               const __half* __restrict__ mlp, const float* __restrict__ rays_d,
               const float* __restrict__ nears, const float* __restrict__ fars,
               const float* __restrict__ noise, const float* __restrict__ sigma,
               const __half* __restrict__ geo, uint32_t N, uint32_t S, float bg_color,
               float* __restrict__ depth_out, float* __restrict__ image_out, float* __restrict__ ws_out,
               float* __restrict__ weights_out, float* __restrict__ z_out, float* __restrict__ rgbs_out) {
    constexpr int NETS = LIDAR ? 2 : 1;
    constexpr int NDIR = LIDAR ? 72 : 16;
    constexpr int NCH = LIDAR ? 2 : 3;
    constexpr int W = kTsWG;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* sm = smem_raw + (base - raw);
    const uint32_t tid = threadIdx.x, wg = tid >> 7, t = tid & 127u, lane = tid & 31u, wq = (tid >> 5) & 3u;
    constexpr uint32_t kOffGeo = kCOffTiles;                                  // [W] geo tiles
    constexpr uint32_t kOffU = kOffGeo + W * kTsGeoTile;                      // [W][2] U images
    constexpr uint32_t kOffScr = kOffU + W * 2 * kCUImg;
    constexpr uint32_t kOffBarC = kOffScr + W * kCScratchFloats * 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBarC + 8 * W);
    float* scr = reinterpret_cast<float*>(sm + kOffScr) + wg * kCScratchFloats;
    float* enc_s = scr;            // [72]
    float* ptot = scr + 200;       // [4]
    float* red = scr + 208;        // [4][8]
    const __half* W1d = reinterpret_cast<const __half*>(sm + kCOffW1d);

    for (uint32_t i = tid; i < kHImgBytes / 16; i += (uint32_t)(W * kRows))
        reinterpret_cast<uint4*>(sm)[i] = __ldg(reinterpret_cast<const uint4*>(wimg) + i);
    for (int net = 0; net < NETS; ++net)
        for (uint32_t i = tid; i < (uint32_t)kHidden * kHeadDirMax / 8; i += (uint32_t)(W * kRows))
            reinterpret_cast<uint4*>(sm + kCOffW1d)[net * (kHidden * kHeadDirMax / 8) + i] =
                __ldg(reinterpret_cast<const uint4*>(mlp + kHeadBase + net * kHeadHalves + kHeadW1d) + i);
    for (uint32_t i = tid; i < (uint32_t)(W * 2 * kCUImg / 16); i += (uint32_t)(W * kRows))
        reinterpret_cast<uint4*>(sm + kOffU)[i] = make_uint4(0, 0, 0, 0);
    if (tid < (uint32_t)W) mbar_init(base + kOffBarC + 8 * tid, 1);
    if (tid < 32) {
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(
                         smem_u32(tmem_slot)),
                     "r"((uint32_t)512)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tcol = tmem + wg * kTsCols;
    const uint32_t tlane = tcol + ((wq * 32u) << 16);
    const uint32_t geo_a = base + kOffGeo + wg * kTsGeoTile;
    unsigned char* geo_p = sm + kOffGeo + wg * kTsGeoTile + (t >> 3) * 256 + (t & 7u) * 16;  // K chunk 0 of row t
    const uint32_t bar = base + kOffBarC + 8 * wg;
    constexpr uint32_t kIdesc2 = umma_idesc(kRows, kHidden), kIdesc3 = umma_idesc(kRows, 16);
    const float kexp = cfg.active_sensor ? 2.0f : 1.0f;
    uint32_t phase = 0;

    // rows of the tile after the current one: the same ray's next 128 samples, or — on a ray's last tile — the first
    // tile of this warpgroup's NEXT ray (ncu had 12 % of the samples on the first use of a ray's freshly issued loads)
    float sg = 0.f;
    uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0;
    {
        const uint32_t r0 = blockIdx.x * W + wg;
        if (r0 < N && t < S) {
            const size_t g = (size_t)r0 * S + t;
            sg = __ldg(sigma + g);
            a0 = __ldg(reinterpret_cast<const uint4*>(geo + g * kGeo));
            a1 = __ldg(reinterpret_cast<const uint4*>(geo + g * kGeo) + 1);
        }
    }
    for (uint32_t r = blockIdx.x * W + wg; r < N; r += gridDim.x * W) {
        const float near = __ldg(nears + r), far = __ldg(fars + r);
        wg_barrier(wg);  // the previous ray's readers of enc / red are done
        {
            const float dx = __ldg(rays_d + (size_t)r * 3), dy = __ldg(rays_d + (size_t)r * 3 + 1),
                        dz = __ldg(rays_d + (size_t)r * 3 + 2);
            if (LIDAR) {
                if (t < (uint32_t)NDIR) {  // tcnn Frequency, 12 octaves: sin(2^k pi x + (j&1) pi/2), x = (d+1)/2
                    const int dim = t / 24, oct = (t >> 1) % 12;
                    const float v = ((dim == 0 ? dx : (dim == 1 ? dy : dz)) + 1.0f) * 0.5f;
                    enc_s[t] = sinpif(scalbnf(v, oct) + 0.5f * (float)(t & 1));
                }
            } else if (t < 16) {
                enc_s[t] = sh4_term((int)t, dx, dy, dz);
            }
        }
        wg_barrier(wg);
        if (t < (uint32_t)(NETS * kHidden)) {  // u[net][n] = sum_j W1[n][dir j] * enc[j] -> U[net][n][0]
            const __half* wrow = W1d + (size_t)t * kHeadDirMax;
            float acc = 0.f;
            for (int j = 0; j < NDIR; j += 2) {
                const float2 w = __half22float2(*reinterpret_cast<const __half2*>(wrow + j));
                acc = fmaf(w.x, enc_s[j], acc);
                acc = fmaf(w.y, enc_s[j + 1], acc);
            }
            const uint32_t net = t >> 6, n = t & 63u;
            *reinterpret_cast<__half*>(sm + kOffU + (wg * 2 + net) * kCUImg + (n >> 3) * 256 + (n & 7u) * 16) =
                __float2half_rn(acc);
        }
        float carry = 1.0f, ws = 0.f, dep = 0.f, img[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) img[c] = 0.f;

        for (uint32_t c0 = 0; c0 < S; c0 += kRows) {
            const uint32_t i = c0 + t;
            const bool in = i < S;
            const size_t g = (size_t)r * S + (in ? i : S - 1);
            const float z = uniform_z2(near, far, in ? i : S - 1, S, noise, g);
            float delta;
            if (i + 1 < S) delta = uniform_z2(near, far, i + 1, S, noise, g + 1) - z;
            else delta = (far - near) / (float)S;  // renderer_dynamic.py:160,182
            const float alpha = in ? 1.0f - expf(((-kexp * delta) * cfg.density_scale) * sg) : 0.f;
            const float v = (1.0f - alpha) + 1e-15f;
            float incl = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float o = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= (uint32_t)d) incl *= o;
            }
            float excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = 1.0f;
            if (lane == 31) ptot[wq] = incl;
            wg_barrier(wg);
            const float p0 = ptot[0], p1 = ptot[1], p2 = ptot[2], p3 = ptot[3];
            const float pre = wq == 0 ? 1.0f : (wq == 1 ? p0 : (wq == 2 ? p0 * p1 : (p0 * p1) * p2));
            const float T = (carry * pre) * excl;
            carry *= ((p0 * p1) * p2) * p3;
            const float w = in ? alpha * T : 0.f;
            ws += w;
            dep = fmaf(w, z, dep);
            if (weights_out && in) { weights_out[g] = w; z_out[g] = z; }
            const bool m = w > 1e-4f;  // renderer_dynamic.py:202
            a0.x = (a0.x & 0xffff0000u) | kOneH;  // col 0: sigma logit -> the constant-1 padding input
            // geo rows -> the un-swizzled A tile (read by the layer-1 MMA of both nets)
            *reinterpret_cast<uint4*>(geo_p) = a0;
            *reinterpret_cast<uint4*>(geo_p + 128) = a1;
            {   // the next tile's rows start travelling
                const bool same = c0 + kRows < S;
                const uint32_t rn = same ? r : r + gridDim.x * W;
                const uint32_t in2 = (same ? c0 + kRows : 0u) + t;
                sg = 0.f; a0 = make_uint4(0, 0, 0, 0); a1 = a0;
                if (rn < N && in2 < S) {
                    const size_t g2 = (size_t)rn * S + in2;
                    sg = __ldg(sigma + g2);
                    a0 = __ldg(reinterpret_cast<const uint4*>(geo + g2 * kGeo));
                    a1 = __ldg(reinterpret_cast<const uint4*>(geo + g2 * kGeo) + 1);
                }
            }
            fence_async_smem();
            tc_fence_before();
            // one barrier: the geo tile is complete, every thread has read ptot, and the OR of the mask
            float4 col = make_float4(0.f, 0.f, 0.f, 0.f);
            if (wg_any(wg, m)) {
                const float wm = m ? w : 0.f;
#pragma unroll
                for (uint32_t net = 0; net < (uint32_t)NETS; ++net) {
                    if (t == 0) {   // D1 [0,64) = geo W1g^T + geo U^T
                        tc_fence_after();
                        const uint64_t ga = umma_desc_k_noswz(geo_a, 128u, 256u);
                        umma_f16(tcol, ga, umma_desc(base + kHOffW1 + net * (kHidden * 128)), kIdesc2, 0u);
                        umma_f16(tcol, ga, umma_desc_k_noswz(base + kOffU + (wg * 2 + net) * kCUImg, 128u, 256u),
                                 kIdesc2, 1u);
                        umma_commit(bar);
                    }
                    mbar_wait(bar, phase); phase ^= 1u;
                    tc_fence_after();
                    hidden_to_tmem(tlane, tlane);                 // H1 packed in place [0,32)
                    tc_fence_before();
                    wg_barrier(wg);
                    if (t == 0) {   // D2 [32,96) = H1 W2^T, A from tensor memory (8 packed columns per K = 16)
                        tc_fence_after();
#pragma unroll
                        for (uint32_t k = 0; k < 4; ++k)
                            umma_f16_ts(tcol + 32, tcol + 8 * k,
                                        umma_desc(base + kHOffW2 + net * (kHidden * 128) + k * 32), kIdesc2, k);
                        umma_commit(bar);
                    }
                    mbar_wait(bar, phase); phase ^= 1u;
                    tc_fence_after();
                    hidden_to_tmem(tlane + 32, tlane + 32);       // H2 packed in place [32,64)
                    tc_fence_before();
                    wg_barrier(wg);
                    if (t == 0) {   // D3 [0,16) = H2 W3^T
                        tc_fence_after();
#pragma unroll
                        for (uint32_t k = 0; k < 4; ++k)
                            umma_f16_ts(tcol, tcol + 32 + 8 * k,
                                        umma_desc(base + kHOffW3 + net * (16 * 128) + k * 32), kIdesc3, k);
                        umma_commit(bar);
                    }
                    mbar_wait(bar, phase); phase ^= 1u;
                    tc_fence_after();
                    uint32_t o[4];
                    tmem_ld4(tlane, o);
                    tmem_ld_wait();
                    tc_fence_before();
                    if (LIDAR) {
                        // h = [raydrop, intensity] (network_dynamic.py:317): net 0 = intensity -> channel 1
                        const float sv = sigmoidf_(__uint_as_float(o[0]));
                        if (net == 0) { img[1] += wm * sv; if (m) col.y = sv; }
                        else { img[0] += wm * sv; if (m) col.x = sv; }
                        if (net == 0) wg_barrier(wg);   // every thread has read D3 before net 1's D1 overwrites it
                    } else {
                        const float s0 = sigmoidf_(__uint_as_float(o[0])), s1 = sigmoidf_(__uint_as_float(o[1])),
                                    s2 = sigmoidf_(__uint_as_float(o[2]));
                        img[0] += wm * s0; img[1] += wm * s1; img[2] += wm * s2;
                        if (m) col = make_float4(s0, s1, s2, 0.f);
                    }
                }
            }
            if (rgbs_out && in) *reinterpret_cast<float4*>(rgbs_out + g * 4) = col;
        }
        // ---- reduce over the warpgroup and write the ray ----
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            ws += __shfl_xor_sync(0xffffffffu, ws, d);
            dep += __shfl_xor_sync(0xffffffffu, dep, d);
#pragma unroll
            for (int c = 0; c < NCH; ++c) img[c] += __shfl_xor_sync(0xffffffffu, img[c], d);
        }
        if (lane == 0) {
            red[wq * 8 + 0] = ws; red[wq * 8 + 1] = dep;
#pragma unroll
            for (int c = 0; c < NCH; ++c) red[wq * 8 + 2 + c] = img[c];
        }
        wg_barrier(wg);
        if (t == 0) {
            const float wsum = ((red[0] + red[8]) + red[16]) + red[24];
            ws_out[r] = wsum;
            depth_out[r] = ((red[1] + red[9]) + red[17]) + red[25];
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                const float v = ((red[2 + c] + red[10 + c]) + red[18 + c]) + red[26 + c];
                image_out[(size_t)r * NCH + c] = LIDAR ? v : v + (1.0f - wsum) * bg_color;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (tid < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"((uint32_t)512)
                     : "memory");
}

int g_heads_tc = 6;  // nvsf_set_option("heads_tc", 0..6): head MLPs of the uniform renderer: 0 mma.sync; 1 tcgen05, four
                     // warpgroups with the two nets overlapped; 2..5 eight / six / five / seven warpgroups, nets in turn, direction
                     // term through a second layer-1 MMA; 6 (default) = 4 with the activations as the A operand from TMEM
bool g_tc_attr8 = false, g_tc_attr_ts = false;
bool g_tc_attr2 = false;

bool g_attr = false;
int ensure_attrs() {
    if (g_attr) return NVSF_OK;
    cudaError_t e = cudaFuncSetAttribute(k_render_composite<true>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)render_smem<true>());
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(k_render_composite<false>,
                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)render_smem<false>());
    if (e != cudaSuccess) return (int)e;
    g_attr = true;
    return NVSF_OK;
}

}  // namespace

extern "C" {

size_t nvsf_render_uniform_scratch_bytes(uint32_t N, uint32_t S) {
    const size_t n = (size_t)N * S;
    return ws_align(n * sizeof(float)) + ws_align(n * kGeo * sizeof(__half)) +
           nvsf_density_split_scratch_bytes(n);
}

/* phase 1: field evaluation of all N*S samples into scratch (sigma f32, geo f16[16]) */
int nvsf_render_uniform_density(const nvsf_field_config_t* cfg, const void* workspace,
                                const float* rays_o, const float* rays_d, const float* nears,
                                const float* fars, const float* noise, uint32_t N, uint32_t S,
                                void* scratch, size_t scratch_bytes, void* stream) {
    if (N == 0) return NVSF_OK;
    if (!field_cfg_ok(cfg) || !workspace || !rays_o || !rays_d || !nears || !fars || !scratch ||
        S == 0)
        return NVSF_E_INVALID;
    if (scratch_bytes < nvsf_render_uniform_scratch_bytes(N, S)) return NVSF_E_WORKSPACE;
    const size_t n = (size_t)N * S;
    float* sigma = reinterpret_cast<float*>(scratch);
    __half* geo = reinterpret_cast<__half*>(reinterpret_cast<unsigned char*>(scratch) +
                                            ws_align(n * sizeof(float)));
    void* split = reinterpret_cast<unsigned char*>(geo) + ws_align(n * kGeo * sizeof(__half));
    return nvsf_launch_density(cfg, workspace, nullptr, rays_o, rays_d, nears, fars, noise, S, n,
                               sigma, geo, nullptr, nullptr, split, (cudaStream_t)stream);
}

/* phase 2: compositing + colour heads from scratch */
int nvsf_render_uniform_composite(const nvsf_field_config_t* cfg, const void* workspace,
                                  uint32_t lidar, const float* rays_d, const float* nears,
                                  const float* fars, const float* noise, uint32_t N, uint32_t S,
                                  float bg_color, const void* scratch, size_t scratch_bytes,
                                  float* depth, float* image, float* weights_sum, float* weights,
                                  float* z_vals, void* stream) {
    return nvsf_render_composite_launch(cfg, workspace, lidar, rays_d, nears, fars, noise, N, S,
                                        bg_color, scratch, scratch_bytes, depth, image, weights_sum,
                                        weights, z_vals, nullptr, stream);
}

}  // extern "C"

int nvsf_render_composite_launch(const nvsf_field_config_t* cfg, const void* workspace,
                                 uint32_t lidar, const float* rays_d, const float* nears,
                                 const float* fars, const float* noise, uint32_t N, uint32_t S,
                                 float bg_color, const void* scratch, size_t scratch_bytes,
                                 float* depth, float* image, float* weights_sum, float* weights,
                                 float* z_vals, void* rgbs, void* stream) {
    if (N == 0) return NVSF_OK;
    if (!field_cfg_ok(cfg) || !workspace || !rays_d || !nears || !fars || !scratch || !depth ||
        !image || !weights_sum || S == 0)
        return NVSF_E_INVALID;
    if ((weights == nullptr) != (z_vals == nullptr)) return NVSF_E_INVALID;
    if (scratch_bytes < ws_align((size_t)N * S * sizeof(float)) + (size_t)N * S * kGeo * sizeof(__half))
        return NVSF_E_WORKSPACE;
    int st = ensure_attrs();
    if (st != NVSF_OK) return st;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)N * S;
    const float* sigma = reinterpret_cast<const float*>(scratch);
    const __half* geo = reinterpret_cast<const __half*>(
        reinterpret_cast<const unsigned char*>(scratch) + ws_align(n * sizeof(float)));
    const FieldPtrs P = nvsf_make_field_ptrs(cfg, workspace);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_heads_tc == 6) {   // hidden activations as the A operand from tensor memory
        if (!g_tc_attr_ts) {
            cudaError_t e = cudaFuncSetAttribute(k_composite_ts<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)composite_ts_smem());
            if (e != cudaSuccess) return (int)e;
            e = cudaFuncSetAttribute(k_composite_ts<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)composite_ts_smem());
            if (e != cudaSuccess) return (int)e;
            g_tc_attr_ts = true;
        }
        const unsigned char* wimg = reinterpret_cast<const unsigned char*>(P.heads_tc);
        const uint32_t grid = std::min<uint32_t>(nvsf_div_up(N, (uint32_t)kTsWG), (uint32_t)sms);
        if (lidar)
            k_composite_ts<true><<<grid, kTsWG * kRows, composite_ts_smem(), s>>>(
                *cfg, wimg, P.mlp, rays_d, nears, fars, noise, sigma, geo, N, S, bg_color, depth, image,
                weights_sum, weights, z_vals, reinterpret_cast<float*>(rgbs));
        else
            k_composite_ts<false><<<grid, kTsWG * kRows, composite_ts_smem(), s>>>(
                *cfg, wimg, P.mlp, rays_d, nears, fars, noise, sigma, geo, N, S, bg_color, depth, image,
                weights_sum, weights, z_vals, reinterpret_cast<float*>(rgbs));
        return nvsf_launch_status();
    }
    if (g_heads_tc >= 2 && g_heads_tc <= 5) {   // 2..5 -> 8, 6, 5, 7 warpgroups per CTA
        const int wsel = g_heads_tc - 2;
        const uint32_t W = wsel == 0 ? 8u : (wsel == 1 ? 6u : (wsel == 2 ? 5u : 7u));
        if (!g_tc_attr8) {
            cudaError_t e = cudaSuccess;
#define NVSF_ATTR_TC8(WW)                                                                                           \
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k_composite_tc8<true, WW>,                                  \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)composite_tc8_smem<WW>()); \
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k_composite_tc8<false, WW>,                                 \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)composite_tc8_smem<WW>());
            NVSF_ATTR_TC8(8) NVSF_ATTR_TC8(6) NVSF_ATTR_TC8(5) NVSF_ATTR_TC8(7)
#undef NVSF_ATTR_TC8
            if (e != cudaSuccess) return (int)e;
            g_tc_attr8 = true;
        }
        const unsigned char* wimg = reinterpret_cast<const unsigned char*>(P.heads_tc);
        const uint32_t grid = std::min<uint32_t>(nvsf_div_up(N, W), (uint32_t)sms);
#define NVSF_LAUNCH_TC8(LID, WW)                                                                              \
        k_composite_tc8<LID, WW><<<grid, WW * kRows, composite_tc8_smem<WW>(), s>>>(                              \
            *cfg, wimg, P.mlp, rays_d, nears, fars, noise, sigma, geo, N, S, bg_color, depth, image, weights_sum, \
            weights, z_vals, reinterpret_cast<float*>(rgbs))
#define NVSF_LAUNCH_TC8_W(LID)                                                           \
        switch (W) {                                                                     \
            case 8: NVSF_LAUNCH_TC8(LID, 8); break;                                      \
            case 7: NVSF_LAUNCH_TC8(LID, 7); break;                                      \
            case 6: NVSF_LAUNCH_TC8(LID, 6); break;                                      \
            default: NVSF_LAUNCH_TC8(LID, 5); break;                                     \
        }
        if (lidar) { NVSF_LAUNCH_TC8_W(true) } else { NVSF_LAUNCH_TC8_W(false) }
#undef NVSF_LAUNCH_TC8_W
#undef NVSF_LAUNCH_TC8
        return nvsf_launch_status();
    }
    if (g_heads_tc) {
        if (!g_tc_attr2) {
            cudaError_t e = cudaFuncSetAttribute(k_composite_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)composite_tc_smem<true>());
            if (e != cudaSuccess) return (int)e;
            e = cudaFuncSetAttribute(k_composite_tc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)composite_tc_smem<false>());
            if (e != cudaSuccess) return (int)e;
            g_tc_attr2 = true;
        }
        const uint32_t grid = std::min<uint32_t>(nvsf_div_up(N, (uint32_t)kCWG), (uint32_t)sms);
        const unsigned char* wimg = reinterpret_cast<const unsigned char*>(P.heads_tc);
        if (lidar)
            k_composite_tc<true><<<grid, kCThreads, composite_tc_smem<true>(), s>>>(
                *cfg, wimg, P.mlp, rays_d, nears, fars, noise, sigma, geo, N, S, bg_color, depth, image,
                weights_sum, weights, z_vals, reinterpret_cast<float*>(rgbs));
        else
            k_composite_tc<false><<<grid, kCThreads, composite_tc_smem<false>(), s>>>(
                *cfg, wimg, P.mlp, rays_d, nears, fars, noise, sigma, geo, N, S, bg_color, depth, image,
                weights_sum, weights, z_vals, reinterpret_cast<float*>(rgbs));
        return nvsf_launch_status();
    }
    const uint32_t blocks = std::min<uint32_t>(nvsf_div_up(N, (uint32_t)kRWarps), (uint32_t)sms * 4);
    if (lidar) {
        k_render_composite<true><<<blocks, kRWarps * 32, render_smem<true>(), s>>>(
            *cfg, P.mlp, rays_d, nears, fars, noise, sigma, geo, N, S, bg_color, depth, image,
            weights_sum, weights, z_vals, reinterpret_cast<float*>(rgbs));
    } else {
        k_render_composite<false><<<blocks, kRWarps * 32, render_smem<false>(), s>>>(
            *cfg, P.mlp, rays_d, nears, fars, noise, sigma, geo, N, S, bg_color, depth, image,
            weights_sum, weights, z_vals, reinterpret_cast<float*>(rgbs));
    }
    return nvsf_launch_status();
}

extern "C" {

int nvsf_render_uniform(const nvsf_field_config_t* cfg, const void* workspace, uint32_t lidar,
                        const float* rays_o, const float* rays_d, const float* nears,
                        const float* fars, const float* noise, uint32_t N, uint32_t S,
                        float bg_color, void* scratch, size_t scratch_bytes, float* depth,
                        float* image, float* weights_sum, float* weights, float* z_vals,
                        void* stream) {
    int st = nvsf_render_uniform_density(cfg, workspace, rays_o, rays_d, nears, fars, noise, N, S,
                                         scratch, scratch_bytes, stream);
    if (st != NVSF_OK) return st;
    return nvsf_render_uniform_composite(cfg, workspace, lidar, rays_d, nears, fars, noise, N, S,
                                         bg_color, scratch, scratch_bytes, depth, image,
                                         weights_sum, weights, z_vals, stream);
}

}  // extern "C"

void nvsf_pack_heads_tc(const __half* mlp, void* dst, int nets, cudaStream_t stream) {
    cudaMemsetAsync(dst, 0, kHImgBytes, stream);
    const int chunks = nets * (kHidden * 2 + kHidden * 8 + 8 * 8) + (nets == 1 ? kHidden * 4 : 0);
    k_pack_heads_tc<<<nvsf_div_up(chunks, 128), 128, 0, stream>>>(mlp, reinterpret_cast<unsigned char*>(dst), nets);
}

// ---- tuning options of the renderer (nvsf_train_set_option falls through to here) -----------------
int nvsf_render_set_option(const char* name, int value) {
    if (std::string(name) == "heads_tc") {
        if (value < 0 || value > 6) return NVSF_E_INVALID;
        g_heads_tc = value;
        return NVSF_OK;
    }
    return nvsf_chamfer_set_option(name, value);
}
int nvsf_heads_tc() { return g_heads_tc; }
int nvsf_render_get_option(const char* name) {
    if (std::string(name) == "heads_tc") return g_heads_tc;
    return nvsf_chamfer_get_option(name);
}
