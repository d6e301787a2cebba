// nvsf_b200 — Adam step over a flat fp32 parameter segment (sm_100a).
//
// Replaces torch.optim.Adam as the reference configures it (reference nvsf/scripts/main_nvsf.py:350-352:
// betas (0.9, 0.99), eps 1e-15, no weight decay, no amsgrad) for the parameters of the field, which
// live in ONE flat buffer per model replica (dist.py GradSync / optim.py): one streaming pass,
// 16 B read (p, g, m, v) + 12 B written (p, m, v) per parameter, 128-bit accesses, grid-stride
// over a multiple of the SM count.  `grad_scale` folds the 1/world_size of the gradient average
// and the inverse loss scale of a GradScaler into the same pass.
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace {

__global__ void __launch_bounds__(256)
k_adam(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
       float4* __restrict__ v, size_t n4, float step_size, float beta1, float beta2, float eps,
       float inv_sqrt_bc2, float grad_scale) {
    const float ob1 = 1.0f - beta1, ob2 = 1.0f - beta2;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
         i += (size_t)gridDim.x * blockDim.x) {
        float4 pi = p[i], mi = m[i], vi = v[i];
        float4 gi = __ldcs(g + i);
        gi.x *= grad_scale; gi.y *= grad_scale; gi.z *= grad_scale; gi.w *= grad_scale;
#define NVSF_ADAM1(c)                                                        \
        mi.c = beta1 * mi.c + ob1 * gi.c;                                    \
        vi.c = beta2 * vi.c + ob2 * gi.c * gi.c;                             \
        pi.c -= step_size * (mi.c / (sqrtf(vi.c) * inv_sqrt_bc2 + eps));
        NVSF_ADAM1(x) NVSF_ADAM1(y) NVSF_ADAM1(z) NVSF_ADAM1(w)
#undef NVSF_ADAM1
        p[i] = pi; m[i] = mi; v[i] = vi;
    }
}

// ---- guarded form (AMP semantics of trainer.py:1332-1334 without a host sync) ---------------------------
// torch's GradScaler.step() reads found_inf back to the host and skips optimizer.step() when a gradient
// is non-finite.  Here the decision stays on the device: `state` = {applied steps t, 1/(1-beta1^t),
// 1/sqrt(1-beta2^t), skip}.  k_adam_begin (one thread) advances t and the bias corrections unless
// *found_inf != 0; the guarded Adam pass returns at once when skip is set, so a skipped step costs two
// tiny launches and the moments / step count are untouched, exactly like a skipped optimizer.step().
__global__ void k_adam_begin(float* __restrict__ state, const float* __restrict__ found_inf, float beta1,
                             float beta2) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const bool skip = found_inf != nullptr && !(*found_inf == 0.0f);
    state[3] = skip ? 1.0f : 0.0f;
    if (skip) return;
    const double t = (double)state[0] + 1.0;
    state[0] = (float)t;
    state[1] = (float)(1.0 / (1.0 - pow((double)beta1, t)));
    state[2] = (float)(1.0 / sqrt(1.0 - pow((double)beta2, t)));
}

__global__ void __launch_bounds__(256)
k_adam_guarded(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
               float4* __restrict__ v, size_t n4, float lr, float beta1, float beta2, float eps,
               const float* __restrict__ state, float grad_scale) {
    if (__ldg(state + 3) != 0.0f) return;
    const float step_size = lr * __ldg(state + 1), inv_sqrt_bc2 = __ldg(state + 2);
    const float ob1 = 1.0f - beta1, ob2 = 1.0f - beta2;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
         i += (size_t)gridDim.x * blockDim.x) {
        float4 pi = p[i], mi = m[i], vi = v[i];
        float4 gi = __ldcs(g + i);
        gi.x *= grad_scale; gi.y *= grad_scale; gi.z *= grad_scale; gi.w *= grad_scale;
#define NVSF_ADAM1(c)                                                        \
        mi.c = beta1 * mi.c + ob1 * gi.c;                                    \
        vi.c = beta2 * vi.c + ob2 * gi.c * gi.c;                             \
        pi.c -= step_size * (mi.c / (sqrtf(vi.c) * inv_sqrt_bc2 + eps));
        NVSF_ADAM1(x) NVSF_ADAM1(y) NVSF_ADAM1(z) NVSF_ADAM1(w)
#undef NVSF_ADAM1
        p[i] = pi; m[i] = mi; v[i] = vi;
    }
}

// found = 1 if any of g[0..n) is inf / nan (x - x != 0 exactly for those); the flag only ever rises, so
// several launches (one per gradient segment) accumulate into the same word without atomics.
__global__ void __launch_bounds__(256)
k_nonfinite(const float4* __restrict__ g, size_t n4, float* __restrict__ found) {
    bool bad = false;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
         i += (size_t)gridDim.x * blockDim.x) {
        const float4 x = __ldg(g + i);
        const float s = (x.x - x.x) + (x.y - x.y) + (x.z - x.z) + (x.w - x.w);
        bad |= !(s == 0.0f);
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) *found = 1.0f;
}

// EMA of the parameters (torch_ema.ExponentialMovingAverage.update, reference trainer.py:112-114):
// s -= (s - p) * omd, rounded after every operation like torch_ema's three tensor ops
// (tmp = s - p; tmp.mul_(omd); s.sub_(tmp)); the _rn intrinsics keep the compiler from contracting
// the product and the subtraction into an FMA, so the shadow stays bit-identical to torch_ema's.
__global__ void __launch_bounds__(256)
k_ema(float4* __restrict__ s, const float4* __restrict__ p, size_t n4, float omd) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
         i += (size_t)gridDim.x * blockDim.x) {
        float4 si = s[i];
        const float4 pi = __ldg(p + i);
#define NVSF_EMA1(c) si.c = __fsub_rn(si.c, __fmul_rn(__fsub_rn(si.c, pi.c), omd));
        NVSF_EMA1(x) NVSF_EMA1(y) NVSF_EMA1(z) NVSF_EMA1(w)
#undef NVSF_EMA1
        s[i] = si;
    }
}

__global__ void k_adam_tail(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, size_t begin, size_t n, float step_size, float beta1,
                            float beta2, float eps, float inv_sqrt_bc2, float grad_scale) {
    const size_t i = begin + threadIdx.x;
    if (i >= n) return;
    const float gi = g[i] * grad_scale;
    const float mi = beta1 * m[i] + (1.0f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;
    p[i] -= step_size * (mi / (sqrtf(vi) * inv_sqrt_bc2 + eps));
    m[i] = mi; v[i] = vi;
}

}  // namespace

static unsigned adam_blocks(size_t n4) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (unsigned)std::min<size_t>(nvsf_div_up(n4, (size_t)256), (size_t)sms * 8);
}

extern "C" int nvsf_grad_found_inf(const float* grads, size_t n, float* found_inf, void* stream) {
    if (n == 0) return NVSF_OK;
    if (!grads || !found_inf || (n & 3) != 0 || ((uintptr_t)grads & 15) != 0) return NVSF_E_INVALID;
    k_nonfinite<<<adam_blocks(n / 4), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(grads), n / 4, found_inf);
    return nvsf_launch_status();
}

extern "C" int nvsf_adam_begin(float* state, const float* found_inf, float beta1, float beta2, void* stream) {
    if (!state) return NVSF_E_INVALID;
    k_adam_begin<<<1, 32, 0, (cudaStream_t)stream>>>(state, found_inf, beta1, beta2);
    return nvsf_launch_status();
}

extern "C" int nvsf_adam_step_guarded(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                                      size_t n, float lr, float beta1, float beta2, float eps,
                                      const float* state, float grad_scale, void* stream) {
    if (n == 0) return NVSF_OK;
    if (!params || !grads || !exp_avg || !exp_avg_sq || !state || (n & 3) != 0) return NVSF_E_INVALID;
    if ((((uintptr_t)params | (uintptr_t)grads | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) != 0)
        return NVSF_E_INVALID;
    k_adam_guarded<<<adam_blocks(n / 4), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<float4*>(params), reinterpret_cast<const float4*>(grads),
        reinterpret_cast<float4*>(exp_avg), reinterpret_cast<float4*>(exp_avg_sq), n / 4, lr, beta1, beta2,
        eps, state, grad_scale);
    return nvsf_launch_status();
}

extern "C" int nvsf_ema_update(float* shadow, const float* params, size_t n, float one_minus_decay, void* stream) {
    if (n == 0) return NVSF_OK;
    if (!shadow || !params || (n & 3) != 0) return NVSF_E_INVALID;
    if ((((uintptr_t)shadow | (uintptr_t)params) & 15) != 0) return NVSF_E_INVALID;
    k_ema<<<adam_blocks(n / 4), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<float4*>(shadow), reinterpret_cast<const float4*>(params), n / 4, one_minus_decay);
    return nvsf_launch_status();
}

extern "C" int nvsf_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                              size_t n, float lr, float beta1, float beta2, float eps, uint32_t step,
                              float grad_scale, void* stream) {
    if (n == 0) return NVSF_OK;
    if (!params || !grads || !exp_avg || !exp_avg_sq || step == 0) return NVSF_E_INVALID;
    if ((((uintptr_t)params | (uintptr_t)grads | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) != 0)
        return NVSF_E_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    // torch.optim.Adam: step_size = lr / (1 - beta1^t), denom = sqrt(v) / sqrt(1 - beta2^t) + eps
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    const float step_size = (float)((double)lr / bc1), inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    const size_t n4 = n / 4;
    if (n4) {
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const unsigned blocks = (unsigned)std::min<size_t>(nvsf_div_up(n4, (size_t)256), (size_t)sms * 8);
        k_adam<<<blocks, 256, 0, s>>>(reinterpret_cast<float4*>(params), reinterpret_cast<const float4*>(grads),
                                      reinterpret_cast<float4*>(exp_avg), reinterpret_cast<float4*>(exp_avg_sq),
                                      n4, step_size, beta1, beta2, eps, inv_sqrt_bc2, grad_scale);
    }
    if (n4 * 4 < n)
        k_adam_tail<<<1, 4, 0, s>>>(params, grads, exp_avg, exp_avg_sq, n4 * 4, n, step_size, beta1, beta2,
                                    eps, inv_sqrt_bc2, grad_scale);
    return nvsf_launch_status();
}
