// Shared helpers for the nvsf_b200 CUDA sources (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/nvsf_b200.h"

#define NVSF_WARP 32

static inline int nvsf_launch_status() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? NVSF_OK : (int)e;
}

template <typename T>
static inline T nvsf_div_up(T a, T b) {
    return (a + b - 1) / b;
}

// ---- warp primitives -------------------------------------------------------

__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += o;
    }
    return v;
}

__device__ __forceinline__ uint64_t warp_inclusive_scan(uint64_t v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint64_t o = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += o;
    }
    return v;
}

__device__ __forceinline__ uint32_t warp_reduce_sum(uint32_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}

// Coalesced, vectorised copy of `nfloats` contiguous floats from global to
// shared memory by the whole block (float4 when the source is 16-byte aligned).
template <int BLOCK>
__device__ __forceinline__ void block_load_floats(const float* __restrict__ src, float* dst,
                                                  uint32_t nfloats) {
    const uint32_t tid = threadIdx.x;
    if ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
        const uint32_t nv = nfloats >> 2;
        const float4* s4 = reinterpret_cast<const float4*>(src);
        float4* d4 = reinterpret_cast<float4*>(dst);
        for (uint32_t i = tid; i < nv; i += BLOCK) d4[i] = __ldg(s4 + i);
        for (uint32_t i = (nv << 2) + tid; i < nfloats; i += BLOCK) dst[i] = __ldg(src + i);
    } else {
        for (uint32_t i = tid; i < nfloats; i += BLOCK) dst[i] = __ldg(src + i);
    }
}
