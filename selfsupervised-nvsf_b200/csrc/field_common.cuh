// Shared definitions of the field kernels: packed-workspace layout, time tables, warp-level
// tensor-core helpers (mma.sync m16n8k16, fp16 in / fp32 accumulate) for the small MLPs.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

constexpr int kHidden = 64;       // n_neurons of every MLP (main_nvsf.py:53-59)
constexpr int kFeat = 128;        // sigma-net input: 120 features padded to 128 with ONES
// tcnn pads the input of a Network up to a multiple of 16 with the constant 1 (the torch binding's
// tcnn.Network wraps the MLP in an Identity encoding whose padded outputs are 1), so the weight columns
// behind the padding act as a learned first-layer bias.  sigma_net: columns 120..127 of the feature row
// are 1.  Head nets: the geo16 operand row (col 0 = sigma logit, never a head input) carries 1 in
// column 0 and the packed geo weight image carries the SUM of the padded columns there.
constexpr uint32_t kOnesH2 = 0x3C003C00u;  // (1.0h, 1.0h)
constexpr uint32_t kOneH = 0x3C00u;
constexpr int kGeo = 16;          // sigma-net output: logit + 15 geo features
constexpr int kHashF = 4;         // features per hash level == temporal basis functions
constexpr int kFlowF = 8;
constexpr int kPlaneF = 8;
constexpr int kHsLevels = 8, kHdLevels = 8, kFlLevels = 16, kPlScales = 4;
constexpr int kFlowIn = 32;       // flow MLP input = 16 levels x (8/4) features

// ---- per-call time tables (device), written by k_time_setup ---------------------------------
struct TimeInfo {
    float t[3];       // query times: t, (f+1)/F, (f-1)/F   (network_dynamic.py:244,260)
    int valid[3];     // [0]=1, [1]= f < F-1, [2]= f > 0      (network_dynamic.py:242,258)
    float lag[3][4];  // cubic Lagrange basis at t[q] on nodes {0,1/3,2/3,1} (hash_field.py:65-74)
    int k1[3], k2[3]; // time slices floor/ceil(t*(Tres-1))   (hash_field.py:79-81)
    float wk[3];      // idx - k1
    int y0[3], y1[3]; // time rows of the (.,t) planes (grid_sample align_corners, border)
    float wy[3];
};

// ---- packed workspace -------------------------------------------------------------------------
// All offsets in bytes, 256-byte aligned.
struct WsLayout {
    size_t time;      // TimeInfo
    size_t hs16;      // __half [hs_entries][4]                     static hash table in fp16
    size_t pls;       // float  per scale: [3 planes xy,xz,yz][R][R][8]   channel-last space planes
    size_t dyn;       // float  [3 queries][sum_p hd_entries[p]]    time-collapsed dynamic hash
    size_t flow;      // float2 [fl_entries]                        time-collapsed flow grid
    size_t pld;       // float  [3 queries] per scale: [3 planes xt,yt,zt][R][8]
    size_t mlp;       // __half smem images of the MLP weights
    size_t dyn16;     // __half [3 queries][sum_p hd_entries[p]]    fp16 mirror of dyn (shared-memory staging)
    size_t pls16;     // __half mirror of pls (same element offsets): one 16-byte texel
    size_t pld16;     // __half mirror of pld
    size_t flow16;    // __half2 [fl_entries]                       fp16 mirror of flow
    size_t heads_tc;  // head-MLP operand images for tcgen05.mma (render.cu k_composite_tc), 36 KB
    size_t mlp_tc;    // sigma-net and flow-MLP operand images for tcgen05.mma (sigma_tc.cu), 2 x 18 KB
    size_t total;
    size_t pls_scale[NVSF_MAX_PLANE_SCALES];  // float offsets inside pls
    size_t pld_scale[NVSF_MAX_PLANE_SCALES];  // float offsets inside one query of pld
    size_t pls_floats, pld_floats_per_q, dyn_per_q;
    size_t dyn_plane[3];                      // float offsets inside one query of dyn
};

// MLP weight images (in halves), padded row strides so ldmatrix rows hit distinct banks.
constexpr int kLdK32 = 40, kLdK64 = 72, kLdK128 = 136, kLdK16 = 24;
constexpr int kFlowW1 = 0;                                   // [64][40]
constexpr int kFlowW2 = kFlowW1 + kHidden * kLdK32;          // [64][72]
constexpr int kFlowW3 = kFlowW2 + kHidden * kLdK64;          // [8][72]   rows 6,7 zero
constexpr int kSigW1 = kFlowW3 + 8 * kLdK64;                 // [64][136]
constexpr int kSigW2 = kSigW1 + kHidden * kLdK128;           // [16][72]
constexpr int kDensityWHalves = kSigW2 + kGeo * kLdK64;      // end of the density-kernel image
// head nets (2 slots; camera uses slot 0 only): per slot
constexpr int kHeadDirMax = 72;                              // Frequency: 72, SH: 16
constexpr int kHeadW1d = 0;                                  // [64][72]  direction part of layer 1
constexpr int kHeadW1g = kHeadW1d + kHidden * kHeadDirMax;   // [64][24]  geo part (col 0 = sum of the padded input columns)
constexpr int kHeadW2 = kHeadW1g + kHidden * kLdK16;         // [64][72]
constexpr int kHeadW3 = kHeadW2 + kHidden * kLdK64;          // [8][72]
constexpr int kHeadHalves = kHeadW3 + 8 * kLdK64;
constexpr int kHeadBase = (kDensityWHalves + 7) / 8 * 8;
constexpr int kMlpHalves = kHeadBase + 2 * kHeadHalves;

static inline size_t ws_align(size_t x) { return (x + 255) & ~(size_t)255; }

static inline bool field_cfg_ok(const nvsf_field_config_t* c) {
    if (!c) return false;
    if (c->hs_levels != kHsLevels || c->hd_levels != kHdLevels || c->fl_levels != kFlLevels ||
        c->pl_scales != kPlScales)
        return false;
    if (c->time_resolution < 1 || c->num_frames < 1 || !(c->bound > 0.f)) return false;
    for (int s = 0; s < kPlScales; ++s)
        if (c->pl_res[s] < 2) return false;
    return true;
}

static inline WsLayout make_ws_layout(const nvsf_field_config_t* c) {
    WsLayout L;
    size_t off = 0;
    L.time = off; off = ws_align(off + sizeof(TimeInfo));
    L.hs16 = off; off = ws_align(off + (size_t)c->hs_entries * kHashF * sizeof(__half));
    size_t f = 0;
    for (int s = 0; s < kPlScales; ++s) {
        L.pls_scale[s] = f;
        f += (size_t)3 * c->pl_res[s] * c->pl_res[s] * kPlaneF;
    }
    L.pls_floats = f;
    L.pls = off; off = ws_align(off + f * sizeof(float));
    size_t d = 0;
    for (int p = 0; p < 3; ++p) { L.dyn_plane[p] = d; d += c->hd_entries[p]; }
    L.dyn_per_q = d;
    L.dyn = off; off = ws_align(off + 3 * d * sizeof(float));
    L.flow = off; off = ws_align(off + (size_t)c->fl_entries * sizeof(float2));
    size_t g = 0;
    for (int s = 0; s < kPlScales; ++s) {
        L.pld_scale[s] = g;
        g += (size_t)3 * c->pl_res[s] * kPlaneF;
    }
    L.pld_floats_per_q = g;
    L.pld = off; off = ws_align(off + 3 * g * sizeof(float));
    L.mlp = off; off = ws_align(off + (size_t)kMlpHalves * sizeof(__half));
    L.dyn16 = off; off = ws_align(off + 3 * d * sizeof(__half));
    L.pls16 = off; off = ws_align(off + f * sizeof(__half));
    L.pld16 = off; off = ws_align(off + 3 * g * sizeof(__half));
    L.flow16 = off; off = ws_align(off + (size_t)c->fl_entries * sizeof(__half2));
    L.mlp_tc = off; off = ws_align(off + 2 * (size_t)(kHidden * kFeat + kGeo * kHidden) * sizeof(__half));
    L.heads_tc = off; off = ws_align(off + (size_t)36864);  // render.cu kHImgBytes
    L.total = off;
    return L;
}

// ---- device pointers into the packed workspace (kernel argument) -------------------------------
struct FieldPtrs {
    const uint2* hs16;
    const float* pls;
    const float* dyn;
    const __half* dyn16;
    const __half* pls16;
    const __half* pld16;
    const __half2* flow16;
    const float2* flow;
    const float* pld;
    const __half* mlp;
    const void* mlp_tc;
    const void* heads_tc;
    const TimeInfo* ti;
    uint32_t pls_scale[kPlScales];
    uint32_t pld_scale[kPlScales];
    uint32_t pld_per_q, dyn_per_q;
    uint32_t dyn_plane[3];
};

FieldPtrs nvsf_make_field_ptrs(const nvsf_field_config_t* cfg, const void* workspace);
// Density launcher shared by field.cu (explicit points) and render.cu (points from rays).
// split_scratch != NULL and density mode 1 select the staged variant (field_split.cu).
int nvsf_launch_density(const nvsf_field_config_t* cfg, const void* workspace, const float* x,
                        const float* rays_o, const float* rays_d, const float* nears,
                        const float* fars, const float* noise, uint32_t S, size_t n, float* sigma,
                        void* geo, void* features, float* flow, void* split_scratch,
                        cudaStream_t stream);
constexpr size_t kSplitChunk = (size_t)64 << 20;  // largest samples-per-chunk option of the staged variant
constexpr size_t kFeatChunk = (size_t)4 << 20;    // chunk of the un-fused path (its [chunk,128] fp16 feature rows)
size_t nvsf_density_split_scratch_bytes(size_t n);
size_t nvsf_density_keep_scratch_bytes(size_t n);  // mode-2 intermediates of the training forward
// Intermediates of the staged evaluation that the training forward keeps for the backward pass.
struct DensityKeep {
    float* flow;        // [n,8]   flow MLP output (6 used)
    __half* feats;      // [n,128] sigma-net input
    __half* flowfeat;   // [n,32]  flow MLP input
};
int nvsf_launch_density_split(const nvsf_field_config_t* cfg, const void* workspace,
                              const float* x, const float* rays_o, const float* rays_d,
                              const float* nears, const float* fars, const float* noise,
                              uint32_t S, size_t n, float* sigma, void* geo, void* features,
                              float* flow, void* split_scratch, cudaStream_t stream,
                              const DensityKeep* keep = nullptr);
int nvsf_density_mode();
// tcgen05 sigma stage (sigma_tc.cu)
void nvsf_pack_sigma_tc(const __half* mlp, void* dst, cudaStream_t stream);
void nvsf_pack_heads_tc(const __half* mlp, void* dst, int nets, cudaStream_t stream);  // render.cu
int nvsf_launch_sigma_tc(const void* wimg, const __half* feat, size_t count, float* sigma,
                         __half* geo, int sms, cudaStream_t stream);
// flow stage on tcgen05 (mode 2): flow [n,8] + planar query positions qpos[9][stride]
int nvsf_launch_flow_tc(const nvsf_field_config_t* cfg, const FieldPtrs& P, const float* x,
                        const float* rays_o, const float* rays_d, const float* nears, const float* fars,
                        const float* noise, uint32_t S, size_t begin, size_t count, float* flow_out,
                        float* qpos, size_t stride, __half* flowfeat, int sms, cudaStream_t stream);
// gather stage fused with the sigma MLP (mode 2 intermediates: query positions + dyn rows)
int nvsf_launch_encode_sigma_tc(const nvsf_field_config_t* cfg, const FieldPtrs& P, const float* qpos,
                                const void* dyn_in, size_t stride, size_t count, float* sigma,
                                __half* geo, int sms, cudaStream_t stream, int half_math,
                                __half* feat_out /* [n,128] kept rows or NULL */);
void nvsf_stage_timing_enable(int on);
int nvsf_split_set_option(const char* name, int value);
int nvsf_split_get_option(const char* name);
int nvsf_train_set_option(const char* name, int value);  // train.cu
int nvsf_train_get_option(const char* name);
int nvsf_render_set_option(const char* name, int value);  // render.cu
int nvsf_render_get_option(const char* name);
int nvsf_chamfer_set_option(const char* name, int value);  // chamfer.cu
int nvsf_chamfer_get_option(const char* name);
int nvsf_heads_tc();                                    // render.cu: option "heads_tc"
// Compositing + heads launcher (render.cu); scratch = sigma f32 [N*S] then geo f16 [N*S,16];
// rgbs (f32 [N*S,4], may be NULL) receives the per-sample colours for the backward pass.
int nvsf_render_composite_launch(const nvsf_field_config_t* cfg, const void* workspace,
                                 uint32_t lidar, const float* rays_d, const float* nears,
                                 const float* fars, const float* noise, uint32_t N, uint32_t S,
                                 float bg_color, const void* scratch, size_t scratch_bytes,
                                 float* depth, float* image, float* weights_sum, float* weights,
                                 float* z_vals, void* rgbs, void* stream);

// ---- tensor-core helpers ------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x2(uint32_t (&r)[2], const void* p) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];\n"
                 : "=r"(r[0]), "=r"(r[1]) : "r"(a));
}
// D(16x8,f32) += A(16x16,f16,row) * B(16x8,f16,col)
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0,
                                         uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, "
        "{%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// The reference's MLP outputs are half-precision tensors (tcnn returns __half; the flow MLP runs under
// fp16 autocast, configs/kitti360_1908.txt:23 / trainer.py:1318): what leaves an MLP is rounded to fp16
// before anything else reads it (trunc_exp of the sigma logit, x + flow of the warped queries).
__device__ __forceinline__ float round_f16(float v) { return __half2float(__float2half_rn(v)); }

__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
    __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}
// fp16x2(relu(lo), relu(hi)) in ONE conversion (cvt.rn.relu.f16x2.f32): the hidden-layer epilogues of
// the tcgen05 kernels are fp32 accumulator -> relu -> fp16 operand tile
__device__ __forceinline__ uint32_t pack_half2_relu(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// One warp: acc[2 m-tiles][NT n-tiles] += A[32 x 16*KT] (registers) * W^T, W in smem [8*NT][ldw].
template <int KT, int NT>
__device__ __forceinline__ void warp_gemm_regA(const uint32_t (&a)[2][KT][4], const __half* W,
                                               int ldw, float (&acc)[2][NT][4], int lane) {
#pragma unroll
    for (int kk = 0; kk < KT; ++kk) {
#pragma unroll
        for (int j = 0; j < NT; j += 2) {
            if (j + 1 < NT) {
                uint32_t b[4];
                ldsm_x4(b, W + ((j + (lane >> 4)) * 8 + (lane & 7)) * ldw + kk * 16 +
                               ((lane >> 3) & 1) * 8);
                mma16816(acc[0][j], a[0][kk], b[0], b[1]);
                mma16816(acc[1][j], a[1][kk], b[0], b[1]);
                mma16816(acc[0][j + 1], a[0][kk], b[2], b[3]);
                mma16816(acc[1][j + 1], a[1][kk], b[2], b[3]);
            } else {
                uint32_t b[2];
                ldsm_x2(b, W + (j * 8 + (lane & 7)) * ldw + kk * 16 + ((lane >> 3) & 1) * 8);
                mma16816(acc[0][j], a[0][kk], b[0], b[1]);
                mma16816(acc[1][j], a[1][kk], b[0], b[1]);
            }
        }
    }
}

// Load the A fragments of a [32 x 16*KT] fp16 tile in shared memory (row stride lda halves).
template <int KT>
__device__ __forceinline__ void load_a_frags(const __half* A, int lda, uint32_t (&a)[2][KT][4],
                                             int lane) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int kk = 0; kk < KT; ++kk)
            ldsm_x4(a[mt][kk], A + (mt * 16 + (lane & 15)) * lda + kk * 16 + (lane >> 4) * 8);
}

// ReLU + fp16 pack: accumulators of a layer with 8*NT outputs -> A fragments of the next layer.
template <int NT>
__device__ __forceinline__ void relu_to_a(const float (&acc)[2][NT][4],
                                          uint32_t (&a)[2][NT / 2][4]) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int kk = 0; kk < NT / 2; ++kk) {
            const float(&c0)[4] = acc[mt][2 * kk];
            const float(&c1)[4] = acc[mt][2 * kk + 1];
            a[mt][kk][0] = pack_half2(fmaxf(c0[0], 0.f), fmaxf(c0[1], 0.f));
            a[mt][kk][1] = pack_half2(fmaxf(c0[2], 0.f), fmaxf(c0[3], 0.f));
            a[mt][kk][2] = pack_half2(fmaxf(c1[0], 0.f), fmaxf(c1[1], 0.f));
            a[mt][kk][3] = pack_half2(fmaxf(c1[2], 0.f), fmaxf(c1[3], 0.f));
        }
}

template <int NT>
__device__ __forceinline__ void zero_acc(float (&acc)[2][NT][4]) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[mt][j][i] = 0.f;
}

// Block-wide copy of 16-byte units global -> shared.
__device__ __forceinline__ void block_copy16(void* dst, const void* src, int n16, int tid,
                                             int nthreads) {
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    for (int i = tid; i < n16; i += nthreads) d[i] = __ldg(s + i);
}

// ---- encoders -----------------------------------------------------------------------------------
struct LevelArgs {
    float scale;
    uint32_t res, size, offset, hashed;
};
__device__ __forceinline__ LevelArgs lv(const nvsf_grid_level_t& g) {
    LevelArgs a;
    a.scale = g.scale; a.res = g.res; a.size = g.size; a.offset = g.offset; a.hashed = g.hashed;
    return a;
}

// floor(p) for |p| < 2^22 without the quarter-rate F2I / FRND conversions: adding 1.5 * 2^23 with
// round-toward-minus-infinity lands in the binade [2^23, 2^24) whose ulp is 1, so the sum IS
// floor(p) + bias, its bit pattern minus the bias pattern is the (signed) integer, and subtracting
// the bias back is exact.  Bit-identical to floorf() + (int) cast on that range.
__device__ __forceinline__ float floor_int(float p, int& i) {
    const float t = __fadd_rd(p, 12582912.0f);
    i = __float_as_int(t) - 0x4B400000;
    return t - 12582912.0f;
}

// tcnn grid position: pos = scale*x + 0.5, cell = floor(pos), w = pos - cell
__device__ __forceinline__ void grid_pos(float scale, float x, uint32_t& cell, float& w) {
    const float p = fmaf(scale, x, 0.5f);
    int c;   // |p| < 2^22 for x in [0,1] (+ flow) and scale <= 32768; any other p still yields an
    const float f = floor_int(p, c);  // in-range table index below (hash mask / wrap_dense)
    cell = (uint32_t)c;
    w = p - f;
}

// Hashed levels always have a power-of-two size (2^log2_hashmap_size).  Dense ones wrap with
// tcnn's `% size`; there the linear index is below res^D + res^(D-1) + .. <= 2 * size for
// coordinates in [0, res] (x in [0,1]), so one conditional subtraction is the same modulo — and
// keeps a 20-instruction integer division out of every unrolled corner (instruction cache).
__device__ __forceinline__ uint32_t wrap_dense(uint32_t lin, uint32_t size) {
    return lin >= size ? (lin - size < size ? lin - size : lin % size) : lin;
}
__device__ __forceinline__ uint32_t idx2(const LevelArgs& L, uint32_t cx, uint32_t cy) {
    if (L.hashed) return (cx ^ (cy * 2654435761u)) & (L.size - 1);
    return wrap_dense(cx + cy * L.res, L.size);
}
__device__ __forceinline__ uint32_t idx3(const LevelArgs& L, uint32_t cx, uint32_t cy,
                                         uint32_t cz) {
    if (L.hashed) return (cx ^ (cy * 2654435761u) ^ (cz * 805459861u)) & (L.size - 1);
    return wrap_dense(cx + cy * L.res + cz * L.res * L.res, L.size);
}

// ---- per-sample encoder primitives ----------------------------------------------------------
__device__ __forceinline__ void st8(__half* row, int col, const float (&v)[8]) {
    uint4 o;
    o.x = pack_half2(v[0], v[1]); o.y = pack_half2(v[2], v[3]);
    o.z = pack_half2(v[4], v[5]); o.w = pack_half2(v[6], v[7]);
    *reinterpret_cast<uint4*>(row + col) = o;
}

// grid_sample unnormalise (align_corners=True) + border clamp
__device__ __forceinline__ void plane_coord(float p, uint32_t R, uint32_t& i0, uint32_t& i1,
                                            float& w) {
    float f = ((p * 2.0f - 1.0f) + 1.0f) * 0.5f * (float)(R - 1);
    f = fminf(fmaxf(f, 0.f), (float)(R - 1));
    int fi;
    const float fl = floor_int(f, fi);   // 0 <= f <= R-1 < 2^22
    i0 = (uint32_t)fi;
    i1 = min(i0 + 1, R - 1);
    w = f - fl;
}

__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// bilinear sample of a channel-last [R][R][8] plane at (pa -> column, pb -> row); out *= sample
__device__ __forceinline__ void plane2d_mul(const float* __restrict__ base, uint32_t R, float pa,
                                            float pb, float (&out)[8], bool first) {
    uint32_t x0, x1, y0, y1;
    float wx, wy;
    plane_coord(pa, R, x0, x1, wx);
    plane_coord(pb, R, y0, y1, wy);
    float a[8], b[8], c[8], d[8];
    ld8(base + ((size_t)y0 * R + x0) * 8, a);
    ld8(base + ((size_t)y0 * R + x1) * 8, b);
    ld8(base + ((size_t)y1 * R + x0) * 8, c);
    ld8(base + ((size_t)y1 * R + x1) * 8, d);
    const float w00 = (1.f - wx) * (1.f - wy), w01 = wx * (1.f - wy), w10 = (1.f - wx) * wy,
                w11 = wx * wy;
#pragma unroll
    for (int f = 0; f < 8; ++f) {
        const float s = w00 * a[f] + w01 * b[f] + w10 * c[f] + w11 * d[f];
        out[f] = first ? s : out[f] * s;
    }
}

// linear sample of a time-collapsed [R][8] row table
__device__ __forceinline__ void plane1d_mul(const float* __restrict__ base, uint32_t R, float pa,
                                            float (&out)[8], bool first) {
    uint32_t x0, x1;
    float wx;
    plane_coord(pa, R, x0, x1, wx);
    float a[8], b[8];
    ld8(base + (size_t)x0 * 8, a);
    ld8(base + (size_t)x1 * 8, b);
#pragma unroll
    for (int f = 0; f < 8; ++f) {
        const float s = (1.f - wx) * a[f] + wx * b[f];
        out[f] = first ? s : out[f] * s;
    }
}

// fp16 mirrors of the plane tables: one texel = 8 halves = one 16-byte load (half the register
// write-back bytes of the fp32 texel, which is what bounds the gather stage: ncu
// l1tex__data_pipe_lsu_wavefronts 89 %, profiles/r01_dyn_encode_ncu.txt).  Interpolation in fp32.
__device__ __forceinline__ void ld8h(const __half* p, float (&v)[8]) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
    const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&a.x));
    const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&a.y));
    const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&a.z));
    const float2 f3 = __half22float2(*reinterpret_cast<const __half2*>(&a.w));
    v[0] = f0.x; v[1] = f0.y; v[2] = f1.x; v[3] = f1.y;
    v[4] = f2.x; v[5] = f2.y; v[6] = f3.x; v[7] = f3.y;
}
__device__ __forceinline__ void plane2d_mul_h(const __half* __restrict__ base, uint32_t R, float pa,
                                              float pb, float (&out)[8], bool first) {
    uint32_t x0, x1, y0, y1;
    float wx, wy;
    plane_coord(pa, R, x0, x1, wx);
    plane_coord(pb, R, y0, y1, wy);
    float a[8], b[8], c[8], d[8];
    ld8h(base + ((size_t)y0 * R + x0) * 8, a);
    ld8h(base + ((size_t)y0 * R + x1) * 8, b);
    ld8h(base + ((size_t)y1 * R + x0) * 8, c);
    ld8h(base + ((size_t)y1 * R + x1) * 8, d);
    const float w00 = (1.f - wx) * (1.f - wy), w01 = wx * (1.f - wy), w10 = (1.f - wx) * wy,
                w11 = wx * wy;
#pragma unroll
    for (int f = 0; f < 8; ++f) {
        const float s = w00 * a[f] + w01 * b[f] + w10 * c[f] + w11 * d[f];
        out[f] = first ? s : out[f] * s;
    }
}
__device__ __forceinline__ void plane1d_mul_h(const __half* __restrict__ base, uint32_t R, float pa,
                                              float (&out)[8], bool first) {
    uint32_t x0, x1;
    float wx;
    plane_coord(pa, R, x0, x1, wx);
    float a[8], b[8];
    ld8h(base + (size_t)x0 * 8, a);
    ld8h(base + (size_t)x1 * 8, b);
#pragma unroll
    for (int f = 0; f < 8; ++f) {
        const float s = (1.f - wx) * a[f] + wx * b[f];
        out[f] = first ? s : out[f] * s;
    }
}

// Packed-half arithmetic for the fused gather + sigma stage (k_encode_sigma_tc<true>): the feature row
// is stored as fp16 in the UMMA operand tile anyway and tcnn itself interpolates its grids in half
// precision (`fma((T)weight, val, result)` with T = __half), so the interpolation runs on HFMA2 —
// one instruction per two channels and no fp16 -> fp32 conversions (22 % of the fp32 kernel's
// instructions).  Weights are formed in fp32 and rounded once.
__device__ __forceinline__ void ld8h2(const __half* p, __half2 (&v)[4]) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
    v[0] = *reinterpret_cast<const __half2*>(&a.x); v[1] = *reinterpret_cast<const __half2*>(&a.y);
    v[2] = *reinterpret_cast<const __half2*>(&a.z); v[3] = *reinterpret_cast<const __half2*>(&a.w);
}
__device__ __forceinline__ void plane2d_mul_h2(const __half* __restrict__ base, uint32_t R, float pa,
                                               float pb, __half2 (&out)[4], bool first) {
    uint32_t x0, x1, y0, y1;
    float wx, wy;
    plane_coord(pa, R, x0, x1, wx);
    plane_coord(pb, R, y0, y1, wy);
    __half2 a[4], b[4], c[4], d[4];
    ld8h2(base + ((size_t)y0 * R + x0) * 8, a);
    ld8h2(base + ((size_t)y0 * R + x1) * 8, b);
    ld8h2(base + ((size_t)y1 * R + x0) * 8, c);
    ld8h2(base + ((size_t)y1 * R + x1) * 8, d);
    const __half2 w00 = __float2half2_rn((1.f - wx) * (1.f - wy)), w01 = __float2half2_rn(wx * (1.f - wy)),
                  w10 = __float2half2_rn((1.f - wx) * wy), w11 = __float2half2_rn(wx * wy);
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        const __half2 s = __hfma2(w11, d[f], __hfma2(w10, c[f], __hfma2(w01, b[f], __hmul2(w00, a[f]))));
        out[f] = first ? s : __hmul2(out[f], s);
    }
}
__device__ __forceinline__ void plane1d_mul_h2(const __half* __restrict__ base, uint32_t R, float pa,
                                               __half2 (&out)[4], bool first) {
    uint32_t x0, x1;
    float wx;
    plane_coord(pa, R, x0, x1, wx);
    __half2 a[4], b[4];
    ld8h2(base + (size_t)x0 * 8, a);
    ld8h2(base + (size_t)x1 * 8, b);
    const __half2 w0 = __float2half2_rn(1.f - wx), w1 = __float2half2_rn(wx);
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        const __half2 s = __hfma2(w1, b[f], __hmul2(w0, a[f]));
        out[f] = first ? s : __hmul2(out[f], s);
    }
}

// Paired variant of hash3_f4 for hashed levels: the hash multiplies x by 1, so for even cx the two
// x-corners of a cell edge are the entries i0 and i0 ^ 1 — one aligned 16-byte load fetches both;
// odd cx needs a second, predicated 8-byte load (half of the lanes on a fine level).  Per edge the
// L1 sees ~1.5 divergent requests instead of 2.  (First measured when the gather stage was
// instruction bound — 18 % slower; it is L1-data-pipe bound since the fp16 texel mirrors.)
__device__ __forceinline__ void hash3_f4_pair(const uint2* __restrict__ tab, const LevelArgs& L,
                                              float x, float y, float z, float* out) {
    uint32_t cx, cy, cz;
    float wx, wy, wz;
    grid_pos(L.scale, x, cx, wx);
    grid_pos(L.scale, y, cy, wy);
    grid_pos(L.scale, z, cz, wz);
    const uint32_t m = L.size - 1;
    const bool odd = cx & 1u;
    const uint2* base = tab + L.offset;
    uint2 v[8];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const uint32_t h = ((cy + (e & 1)) * 2654435761u) ^ ((cz + (e >> 1)) * 805459861u);
        const uint32_t i0 = (cx ^ h) & m;
        const uint4 q = __ldg(reinterpret_cast<const uint4*>(base + (i0 & ~1u)));
        const bool hi = i0 & 1u;
        v[2 * e] = hi ? make_uint2(q.z, q.w) : make_uint2(q.x, q.y);
        uint2 nb = hi ? make_uint2(q.x, q.y) : make_uint2(q.z, q.w);
        if (odd) nb = __ldg(base + (((cx + 1) ^ h) & m));
        v[2 * e + 1] = nb;
    }
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float w = ((c & 1) ? wx : 1.f - wx) * ((c & 2) ? wy : 1.f - wy) *
                        ((c & 4) ? wz : 1.f - wz);
        const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&v[c].x));
        const float2 hi2 = __half22float2(*reinterpret_cast<const __half2*>(&v[c].y));
        a0 = fmaf(w, lo.x, a0); a1 = fmaf(w, lo.y, a1);
        a2 = fmaf(w, hi2.x, a2); a3 = fmaf(w, hi2.y, a3);
    }
    out[0] = a0; out[1] = a1; out[2] = a2; out[3] = a3;
}

// (Measured and rejected on B200: ld.global.nc.L1::no_allocate for the fine hashed levels — the
// gather stage went from 13.1 to 17.7 ms per frame; the x-neighbour of a corner sits in the same
// 32-byte sector three times out of four and is an L1 hit only if the first load allocated.)
// one level of the 3-D fp16 static hash grid (4 features)
__device__ __forceinline__ void hash3_f4(const uint2* __restrict__ tab, const LevelArgs& L,
                                         float x, float y, float z, float* out) {
    uint32_t cx, cy, cz;
    float wx, wy, wz;
    grid_pos(L.scale, x, cx, wx);
    grid_pos(L.scale, y, cy, wy);
    grid_pos(L.scale, z, cz, wz);
    uint2 v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c)
        v[c] = __ldg(tab + L.offset + idx3(L, cx + (c & 1), cy + ((c >> 1) & 1), cz + (c >> 2)));
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float w = ((c & 1) ? wx : 1.f - wx) * ((c & 2) ? wy : 1.f - wy) *
                        ((c & 4) ? wz : 1.f - wz);
        const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&v[c].x));
        const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&v[c].y));
        a0 = fmaf(w, lo.x, a0); a1 = fmaf(w, lo.y, a1);
        a2 = fmaf(w, hi.x, a2); a3 = fmaf(w, hi.y, a3);
    }
    out[0] = a0; out[1] = a1; out[2] = a2; out[3] = a3;
}

// same level in packed-half arithmetic (see plane2d_mul_h2): out = 2 x half2
__device__ __forceinline__ void hash3_f4_h2(const uint2* __restrict__ tab, const LevelArgs& L,
                                            float x, float y, float z, __half2* out) {
    uint32_t cx, cy, cz;
    float wx, wy, wz;
    grid_pos(L.scale, x, cx, wx);
    grid_pos(L.scale, y, cy, wy);
    grid_pos(L.scale, z, cz, wz);
    uint2 v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c)
        v[c] = __ldg(tab + L.offset + idx3(L, cx + (c & 1), cy + ((c >> 1) & 1), cz + (c >> 2)));
    __half2 a0 = __float2half2_rn(0.f), a1 = a0;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const __half2 w = __float2half2_rn(((c & 1) ? wx : 1.f - wx) * ((c & 2) ? wy : 1.f - wy) *
                                           ((c & 4) ? wz : 1.f - wz));
        a0 = __hfma2(w, *reinterpret_cast<const __half2*>(&v[c].x), a0);
        a1 = __hfma2(w, *reinterpret_cast<const __half2*>(&v[c].y), a1);
    }
    out[0] = a0; out[1] = a1;
}

// one level of a time-collapsed 2-D dynamic hash grid (1 value)
__device__ __forceinline__ float hash2_f1(const float* __restrict__ tab, const LevelArgs& L,
                                          float u, float v) {
    uint32_t cu, cv;
    float wu, wv;
    grid_pos(L.scale, u, cu, wu);
    grid_pos(L.scale, v, cv, wv);
    const float t00 = __ldg(tab + L.offset + idx2(L, cu, cv));
    const float t10 = __ldg(tab + L.offset + idx2(L, cu + 1, cv));
    const float t01 = __ldg(tab + L.offset + idx2(L, cu, cv + 1));
    const float t11 = __ldg(tab + L.offset + idx2(L, cu + 1, cv + 1));
    return (1.f - wu) * (1.f - wv) * t00 + wu * (1.f - wv) * t10 + (1.f - wu) * wv * t01 +
           wu * wv * t11;
}

// one level of the time-collapsed 3-D flow grid (2 values)
__device__ __forceinline__ float2 hash3_f2(const float2* __restrict__ tab, const LevelArgs& L,
                                           float x, float y, float z) {
    uint32_t cx, cy, cz;
    float wx, wy, wz;
    grid_pos(L.scale, x, cx, wx);
    grid_pos(L.scale, y, cy, wy);
    grid_pos(L.scale, z, cz, wz);
    float2 v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c)
        v[c] = __ldg(tab + L.offset + idx3(L, cx + (c & 1), cy + ((c >> 1) & 1), cz + (c >> 2)));
    float a0 = 0.f, a1 = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float w = ((c & 1) ? wx : 1.f - wx) * ((c & 2) ? wy : 1.f - wy) *
                        ((c & 4) ? wz : 1.f - wz);
        a0 = fmaf(w, v[c].x, a0);
        a1 = fmaf(w, v[c].y, a1);
    }
    return make_float2(a0, a1);
}

// same from the fp16 mirror (4-byte entries: half the L2 footprint and register write-back)
__device__ __forceinline__ float2 hash3_h2(const __half2* __restrict__ tab, const LevelArgs& L,
                                           float x, float y, float z) {
    uint32_t cx, cy, cz;
    float wx, wy, wz;
    grid_pos(L.scale, x, cx, wx);
    grid_pos(L.scale, y, cy, wy);
    grid_pos(L.scale, z, cz, wz);
    __half2 v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c)
        v[c] = __ldg(tab + L.offset + idx3(L, cx + (c & 1), cy + ((c >> 1) & 1), cz + (c >> 2)));
    float a0 = 0.f, a1 = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float w = ((c & 1) ? wx : 1.f - wx) * ((c & 2) ? wy : 1.f - wy) *
                        ((c & 4) ? wz : 1.f - wz);
        const float2 f = __half22float2(v[c]);
        a0 = fmaf(w, f.x, a0);
        a1 = fmaf(w, f.y, a1);
    }
    return make_float2(a0, a1);
}

// z value of uniform sample k of S in [near, far]  (torch.linspace(0,1,S), renderer_dynamic.py:155-164)
__device__ __forceinline__ float uniform_z(float near, float far, uint32_t k, uint32_t S,
                                           const float* __restrict__ noise, size_t g) {
    const float step = 1.0f / (float)(S > 1 ? S - 1 : 1);
    const float lin = (k < S / 2) ? step * (float)k : 1.0f - step * (float)(S - 1 - k);
    float z = near + (far - near) * lin;
    if (noise) z = z + (__ldg(noise + g) - 0.5f) * ((far - near) / (float)S);
    return z;
}

// normalised position in [0,1]^3 of sample g: explicit point xin[g], or uniform sample g % S of ray
// g / S (renderer_dynamic.py:155-169: linspace z, optional jitter, clip to the box)
template <bool FROM_RAYS>
__device__ __forceinline__ void sample_position(const nvsf_field_config_t& cfg, size_t g,
                                                const float* __restrict__ xin,
                                                const float* __restrict__ rays_o,
                                                const float* __restrict__ rays_d,
                                                const float* __restrict__ nears,
                                                const float* __restrict__ fars,
                                                const float* __restrict__ noise, uint32_t S,
                                                float& x, float& y, float& z) {
    float px, py, pz;
    if (FROM_RAYS) {
        size_t r;
        uint32_t k;
        if ((g >> 32) == 0) {  // 32-bit division: the 64-bit one costs ~100 instructions per call
            const uint32_t g32 = (uint32_t)g, r32 = g32 / S;
            r = r32;
            k = g32 - r32 * S;
        } else {
            r = g / S;
            k = (uint32_t)(g - r * S);
        }
        const float zz = uniform_z(__ldg(nears + r), __ldg(fars + r), k, S, noise, g);
        px = __ldg(rays_o + r * 3 + 0) + __ldg(rays_d + r * 3 + 0) * zz;
        py = __ldg(rays_o + r * 3 + 1) + __ldg(rays_d + r * 3 + 1) * zz;
        pz = __ldg(rays_o + r * 3 + 2) + __ldg(rays_d + r * 3 + 2) * zz;
        px = fminf(fmaxf(px, -cfg.bound), cfg.bound);
        py = fminf(fmaxf(py, -cfg.bound), cfg.bound);
        pz = fminf(fmaxf(pz, -cfg.bound), cfg.bound);
    } else {
        px = __ldg(xin + g * 3 + 0); py = __ldg(xin + g * 3 + 1); pz = __ldg(xin + g * 3 + 2);
    }
    const float inv2b = 1.0f / (2.0f * cfg.bound);
    x = (px + cfg.bound) * inv2b; y = (py + cfg.bound) * inv2b; z = (pz + cfg.bound) * inv2b;
}
