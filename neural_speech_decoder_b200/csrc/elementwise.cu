// Element-wise kernels of the path: inter-layer dropout (nn.GRU dropout=p, reference model.py:55).
#include <algorithm>

#include "common.cuh"

namespace nsd {

template <typename T>
__global__ void dropout_kernel(const T* __restrict__ x, T* __restrict__ out, size_t n, float p, float inv_keep, uint64_t seed) {
    pdl_enter();
    // one Philox call covers 4 consecutive elements; the mask depends only on (seed, element index)
    const size_t nq = (n + 3) / 4;
    const uint32_t thresh = dropout_threshold(p);
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (size_t)gridDim.x * blockDim.x) {
        const uint4 r = dropout_bits(q, seed);
        const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const size_t e = q * 4 + i;
            if (e < n) out[e] = from_f32<T>(rr[i] >= thresh ? to_f32<T>(x[e]) * inv_keep : 0.f);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Multi-tensor Adam (torch.optim.Adam semantics: g += wd*p; m,v EMA; bias correction; p -= lr/bc1 * m / (sqrt(v)/sqrt(bc2) + eps)).
// Replaces the foreach Adam step of the reference trainer (neural_decoder_trainer.py:163-169, 259).
// HBM-bound: 16 B read + 12 B written per element; every thread moves float4s.
constexpr int ADAM_MAX_TENSORS = 48;
constexpr int ADAM_CHUNK = 16384;       // elements per CTA

struct AdamTable {
    float* p[ADAM_MAX_TENSORS]; const float* g[ADAM_MAX_TENSORS]; float* m[ADAM_MAX_TENSORS]; float* v[ADAM_MAX_TENSORS];
    long long n[ADAM_MAX_TENSORS];
    __nv_bfloat16* s[ADAM_MAX_TENSORS];     // optional bf16 shadow of the updated parameter (tensor-core operand copy) or null
    int chunk_start[ADAM_MAX_TENSORS + 1];   // first CTA of each tensor
    int count;
};

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float b1, float b2, float wd,
                                         float gs, float step_size, float inv_sqrt_bc2, float eps, float decay_mul) {
    g = fmaf(wd, p, g * gs);                 // Adam: L2 term in the gradient (wd = 0 for AdamW)
    p *= decay_mul;                          // AdamW: decoupled decay p *= 1 - lr*wd (1 for Adam)
    m = fmaf(b1, m, (1.0f - b1) * g);
    v = fmaf(b2, v, (1.0f - b2) * g * g);
    const float denom = sqrtf(v) * inv_sqrt_bc2 + eps;
    p -= step_size * (m / denom);
}

// late_wait (the optimizer under the recurrence): the launch sits behind a K3 kernel whose OUTPUT it does not need -- its gradients were
// final before that kernel started -- so it must not wait for it: the CTAs start as soon as every K3 CTA is resident (they get the SMs
// the recurrence leaves free) and stream their update under it.  The grid must still not COMPLETE before K3 has, because the next kernel
// in the stream orders itself after THIS grid only: the last CTA to finish its work (device counter) executes griddepcontrol.wait.
__device__ unsigned int g_adam_done = 0;
__global__ void __launch_bounds__(256) adam_kernel(const __grid_constant__ AdamTable tab, float b1, float b2, float wd, float gs,
                                                   float step_size, float inv_sqrt_bc2, float eps, float decay_mul,
                                                   const float* __restrict__ grad_sqnorm, float max_norm, const float* __restrict__ hyper, int late_wait) {
    if (!late_wait) { pdl_launch_dependents(); pdl_wait(); }   // late_wait: the next kernel's CTAs must not crowd the few SMs this launch runs on
    if (hyper != nullptr) { step_size = hyper[0]; inv_sqrt_bc2 = hyper[1]; decay_mul = hyper[2]; }   // device-resident schedule (graph replay)
    if (grad_sqnorm != nullptr) {            // clip_grad_norm_(max_norm): coefficient from the device-resident squared norm, no host sync
        const float norm = sqrtf(*grad_sqnorm) * gs;
        gs *= fminf(1.0f, max_norm / (norm + 1e-6f));
    }
    // locate this CTA's tensor (count <= 48: linear scan by one thread is cheap, but all threads can do it)
    int ti = 0;
    while (ti + 1 < tab.count && (int)blockIdx.x >= tab.chunk_start[ti + 1]) ++ti;
    const long long n = tab.n[ti];
    const long long base = (long long)(blockIdx.x - tab.chunk_start[ti]) * ADAM_CHUNK;
    const long long end = min(n, base + ADAM_CHUNK);
    float* __restrict__ P = tab.p[ti]; const float* __restrict__ G = tab.g[ti];
    float* __restrict__ M = tab.m[ti]; float* __restrict__ V = tab.v[ti];
    __nv_bfloat16* __restrict__ S = tab.s[ti];
    const bool vec = ((((uintptr_t)P | (uintptr_t)G | (uintptr_t)M | (uintptr_t)V) & 15) | ((uintptr_t)S & 7)) == 0;
    if (vec) {
        const long long e4 = base + ((end - base) & ~3LL);
        for (long long i = base + 4LL * threadIdx.x; i < e4; i += 4LL * blockDim.x) {
            float4 p = *reinterpret_cast<float4*>(P + i), m = *reinterpret_cast<float4*>(M + i), v = *reinterpret_cast<float4*>(V + i);
            const float4 g = __ldcs(reinterpret_cast<const float4*>(G + i));
            adam_one(p.x, g.x, m.x, v.x, b1, b2, wd, gs, step_size, inv_sqrt_bc2, eps, decay_mul);
            adam_one(p.y, g.y, m.y, v.y, b1, b2, wd, gs, step_size, inv_sqrt_bc2, eps, decay_mul);
            adam_one(p.z, g.z, m.z, v.z, b1, b2, wd, gs, step_size, inv_sqrt_bc2, eps, decay_mul);
            adam_one(p.w, g.w, m.w, v.w, b1, b2, wd, gs, step_size, inv_sqrt_bc2, eps, decay_mul);
            *reinterpret_cast<float4*>(P + i) = p; *reinterpret_cast<float4*>(M + i) = m; *reinterpret_cast<float4*>(V + i) = v;
            if (S) {
                const __nv_bfloat162 lo = __floats2bfloat162_rn(p.x, p.y), hi = __floats2bfloat162_rn(p.z, p.w);
                *reinterpret_cast<uint2*>(S + i) = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
            }
        }
        for (long long i = e4 + threadIdx.x; i < end; i += blockDim.x) {
            adam_one(P[i], G[i], M[i], V[i], b1, b2, wd, gs, step_size, inv_sqrt_bc2, eps, decay_mul);
            if (S) S[i] = __float2bfloat16_rn(P[i]);
        }
    } else {
        for (long long i = base + threadIdx.x; i < end; i += blockDim.x) {
            adam_one(P[i], G[i], M[i], V[i], b1, b2, wd, gs, step_size, inv_sqrt_bc2, eps, decay_mul);
            if (S) S[i] = __float2bfloat16_rn(P[i]);
        }
    }
    if (late_wait) {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            if (atomicAdd(&g_adam_done, 1u) == gridDim.x - 1) {
                g_adam_done = 0;
                pdl_wait();
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------
// Multi-tensor gather: up to 64 small f32 vectors copied to their destinations in ONE launch (the per-direction GRU
// biases packed side by side, so that one GEMM epilogue / one recurrence launch serves both directions).
constexpr int COPY_MAX_TENSORS = 64;
struct CopyTable {
    const float* src[COPY_MAX_TENSORS]; float* dst[COPY_MAX_TENSORS]; long long n[COPY_MAX_TENSORS];
    int count;
};
__global__ void __launch_bounds__(256) multi_copy_kernel(const __grid_constant__ CopyTable tab) {
    pdl_enter();
    const int ti = blockIdx.y;
    const float* __restrict__ S = tab.src[ti];
    float* __restrict__ D = tab.dst[ti];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tab.n[ti]; i += (long long)gridDim.x * blockDim.x) D[i] = S[i];
}

}  // namespace nsd

extern "C" {

int nsd_multi_copy_f32(int n_tensors, const void* const* src, void* const* dst, const int64_t* numel, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(n_tensors >= 0, "multi_copy: bad n_tensors=%d", n_tensors);
    for (int t0 = 0; t0 < n_tensors; t0 += COPY_MAX_TENSORS) {
        CopyTable tab;
        tab.count = std::min(COPY_MAX_TENSORS, n_tensors - t0);
        long long nmax = 0;
        for (int i = 0; i < tab.count; ++i) {
            NSD_CHECK_ARG(numel[t0 + i] >= 0 && (numel[t0 + i] == 0 || (src[t0 + i] && dst[t0 + i])), "multi_copy: null tensor %d", t0 + i);
            tab.src[i] = (const float*)src[t0 + i]; tab.dst[i] = (float*)dst[t0 + i]; tab.n[i] = numel[t0 + i];
            nmax = std::max<long long>(nmax, numel[t0 + i]);
        }
        if (nmax == 0) continue;
        const dim3 grid((unsigned)std::min<long long>((nmax + 255) / 256, 64), (unsigned)tab.count);
        nsd::launch_k(multi_copy_kernel, grid, 256, 0, (cudaStream_t)stream, tab);
        NSD_LAUNCH_CHECK();
    }
    return NSD_OK;
}


static int g_adam_late_wait = 0;
static int adam_impl(int n_tensors, void* const* params, const void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
                     const int64_t* numel, void* const* shadow_bf16, float lr, float beta1, float beta2, float eps, float wd_l2, float decay_mul,
                     int step, float grad_scale, const float* grad_sqnorm, float max_norm, const float* hyper, void* stream, const char* who) {
    using namespace nsd;
    NSD_CHECK_ARG(n_tensors >= 0 && step >= 1, "%s: bad n_tensors=%d step=%d", who, n_tensors, step);
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    const float step_size = (float)((double)lr / bc1), inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    for (int t0 = 0; t0 < n_tensors; t0 += ADAM_MAX_TENSORS) {
        AdamTable tab;
        tab.count = std::min(ADAM_MAX_TENSORS, n_tensors - t0);
        int chunks = 0;
        for (int i = 0; i < tab.count; ++i) {
            NSD_CHECK_ARG(params[t0 + i] && grads[t0 + i] && exp_avg[t0 + i] && exp_avg_sq[t0 + i] && numel[t0 + i] >= 0, "%s: null tensor %d", who, t0 + i);
            tab.p[i] = (float*)params[t0 + i]; tab.g[i] = (const float*)grads[t0 + i];
            tab.m[i] = (float*)exp_avg[t0 + i]; tab.v[i] = (float*)exp_avg_sq[t0 + i];
            tab.n[i] = numel[t0 + i];
            tab.s[i] = shadow_bf16 ? (__nv_bfloat16*)shadow_bf16[t0 + i] : nullptr;
            tab.chunk_start[i] = chunks;
            chunks += (int)cdivz((size_t)numel[t0 + i], ADAM_CHUNK);
        }
        tab.chunk_start[tab.count] = chunks;
        if (chunks == 0) continue;
        nsd::launch_k(adam_kernel, chunks, 256, 0, (cudaStream_t)stream, tab, beta1, beta2, wd_l2, grad_scale, step_size, inv_sqrt_bc2, eps, decay_mul, grad_sqnorm,
                                                               max_norm, hyper, (g_adam_late_wait && n_tensors <= ADAM_MAX_TENSORS) ? 1 : 0);
        NSD_LAUNCH_CHECK();
    }
    return NSD_OK;
}

int nsd_set_adam_late_wait(int on) { g_adam_late_wait = on ? 1 : 0; return NSD_OK; }

int nsd_adam_step(int n_tensors, void* const* params, const void* const* grads, void* const* exp_avg,
                  void* const* exp_avg_sq, const int64_t* numel, void* const* shadow_bf16, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int step, float grad_scale, void* stream) {
    return adam_impl(n_tensors, params, grads, exp_avg, exp_avg_sq, numel, shadow_bf16, lr, beta1, beta2, eps, weight_decay, 1.0f, step, grad_scale,
                     nullptr, 0.f, nullptr, stream, "adam_step");
}

int nsd_adamw_step(int n_tensors, void* const* params, const void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
                   const int64_t* numel, void* const* shadow_bf16, float lr, float beta1, float beta2, float eps, float weight_decay, int step,
                   float grad_scale, const float* grad_sqnorm, float max_norm, const float* hyper_dev, void* stream) {
    return adam_impl(n_tensors, params, grads, exp_avg, exp_avg_sq, numel, shadow_bf16, lr, beta1, beta2, eps, 0.f, 1.0f - lr * weight_decay, step,
                     grad_scale, grad_sqnorm, max_norm, hyper_dev, stream, "adamw_step");
}

int nsd_dropout(const void* x, void* out, int dtype, size_t n, float p, uint64_t seed, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(p >= 0.f && p < 1.f, "dropout: p=%f not in [0,1)", (double)p);
    if (n == 0) return NSD_OK;
    const int blocks = (int)std::min<size_t>(cdivz(cdivz(n, 4), 256), (size_t)sm_count() * 16);
    const float inv_keep = 1.0f / (1.0f - p);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NSD_F32) nsd::launch_k(dropout_kernel<float>, blocks, 256, 0, s, (const float*)x, (float*)out, n, p, inv_keep, seed);
    else if (dtype == NSD_BF16) nsd::launch_k(dropout_kernel<__nv_bfloat16>, blocks, 256, 0, s, (const __nv_bfloat16*)x, (__nv_bfloat16*)out, n, p, inv_keep, seed);
    else { set_error("dropout: bad dtype"); return NSD_ERR_INVALID; }
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

}  // extern "C"
