// Exact order statistic of n unsigned 32-bit keys by one CTA: a 4-pass, 8-bit radix select (shared by the
// metric medians of eval.cu and the error-map sampler of scene.cu).
#pragma once
#include "common.cuh"

// The k-th smallest (0-based) of key(0..n-1); every thread of the CTA calls it and gets the same result.
// *ties = how many keys equal to the result rank before it (k minus the number of smaller keys), so the
// k + 1 smallest keys are all keys below the result plus the first *ties + 1 keys equal to it.
// `hist` holds 256 counters in shared memory; `key` must be valid on every thread for every i < n.
template <int BLOCK, typename Key>
__device__ __forceinline__ uint32_t radix_select(Key key, uint32_t n, uint32_t k, uint32_t* hist,
                                                 uint32_t& ties) {
    __shared__ uint32_t digit_s, rank_s;
    uint32_t prefix = 0, mask = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (uint32_t i = threadIdx.x; i < 256; i += BLOCK) hist[i] = 0;
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n; i += BLOCK) {
            const uint32_t u = key(i);
            if ((u & mask) == prefix) atomicAdd(&hist[(u >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t below = 0, d = 0;
            for (; d < 255; ++d) {
                if (below + hist[d] > k) break;
                below += hist[d];
            }
            digit_s = d;
            rank_s = k - below;
        }
        __syncthreads();
        prefix |= digit_s << shift;
        mask |= 0xffu << shift;
        k = rank_s;
        __syncthreads();
    }
    ties = k;
    return prefix;
}
