// Shared helpers for the nsd_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/nsd_b200.h"

namespace nsd {

void set_error(const char* fmt, ...);

#define NSD_CHECK_ARG(cond, ...)            \
    do {                                    \
        if (!(cond)) {                      \
            nsd::set_error(__VA_ARGS__);    \
            return NSD_ERR_INVALID;         \
        }                                   \
    } while (0)

#define NSD_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            nsd::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return NSD_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

void count_launch(int n);   // kernels enqueued by this library (nsd_launch_count)

#define NSD_LAUNCH_CHECK()              \
    do {                                \
        nsd::count_launch(1);           \
        NSD_CUDA(cudaGetLastError());   \
    } while (0)

// Programmatic dependent launch.  Every kernel launched through launch_k() carries the programmatic-stream-serialization attribute: it
// may be scheduled while its predecessor in the stream is still running, and MUST execute pdl_enter() (or pdl_wait()) before it touches
// global memory -- griddepcontrol.wait returns once every prerequisite grid has completed and its writes are visible.
// pdl_launch_dependents() at the top of a kernel lets the next launch's CTAs take SM resources as they free up and run their prologue
// (barrier init, TMEM allocation, descriptor prefetch) under this kernel's tail: it removes the few microseconds of launch latency and
// ramp between the ~100 (GRU step) / ~750 (Conformer step) short kernels of a training step.  Both instructions are no-ops in a kernel
// launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() { pdl_launch_dependents(); pdl_wait(); }
template <typename... KArgs, typename... Args>
static inline void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    (void)cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);      // errors surface through cudaGetLastError (NSD_LAUNCH_CHECK)
}

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline size_t cdivz(size_t a, size_t b) { return (a + b - 1) / b; }

int sm_count();   // cached multiProcessorCount of the current device

// Device-resident offset added to every Philox seed of the Conformer kernels and nsd_input_noise (nsd_set_seed_offset_ptr): lets a
// captured CUDA graph draw fresh masks on every replay.  nullptr = none.
const unsigned long long* seed_offset_ptr();

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }
// tanh via exp, accurate to ~1e-7 relative for the fp32 parity path
__device__ __forceinline__ float tanhf_(float x) { return tanhf(x); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Philox4x32-10 counter-based generator: 4 uniform 32-bit words per (key, counter).
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0; key.y += W1;
    }
    return ctr;
}

// Inter-layer dropout (reference model.py:55): the keep/drop decision of element e of a contiguous tensor depends only on
// (seed, e): one Philox call yields the bits for elements 4q .. 4q+3; element i is KEPT iff word i >= dropout_threshold(p).
__device__ __forceinline__ uint4 dropout_bits(size_t q, uint64_t seed) {
    return philox4x32_10(make_uint4((uint32_t)q, (uint32_t)(q >> 32), 0u, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}
__host__ __device__ __forceinline__ uint32_t dropout_threshold(float p) { return (uint32_t)fminf(4294967295.0f, p * 4294967296.0f); }

// In-loop training augmentation of the reference (neural_decoder_trainer.py:194-201): X += N(0,1)*whiteNoiseSD (per element)
// and X += N(0,1)*constantOffsetSD (per utterance and channel, constant over time).  Counter-based: the four standard
// normals of elements 4q .. 4q+3 of a stream depend only on (seed, stream, q) -- Philox bits through Box-Muller -- so the
// fused form inside K1 and the stand-alone kernel produce identical values wherever and however often an element is read.
__device__ __forceinline__ float4 normal4(size_t q, uint64_t seed, uint32_t stream) {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)q, (uint32_t)(q >> 32), stream, 0x6e6f6973u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float u0 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f), u1 = ((float)(r.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(r.z >> 8) + 0.5f) * (1.0f / 16777216.0f), u3 = ((float)(r.w >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float m0 = sqrtf(-2.0f * __logf(u0)), m1 = sqrtf(-2.0f * __logf(u2));
    float s0, c0, s1, c1;
    __sincosf(6.2831853071795865f * u1, &s0, &c0);
    __sincosf(6.2831853071795865f * u3, &s1, &c1);
    return make_float4(m0 * c0, m0 * s0, m1 * c1, m1 * s1);
}
__device__ __forceinline__ float normal1(size_t e, uint64_t seed, uint32_t stream) {
    const float4 v = normal4(e >> 2, seed, stream);
    const int i = (int)(e & 3);
    return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w));
}
// x[b,t,c] + white_sd * n0[(b*T+t)*N+c] + offset_sd * n1[b*N+c]   (N % 4 == 0 variant for four consecutive channels)
__device__ __forceinline__ float4 add_input_noise4(float4 v, size_t e, size_t eo, float white_sd, float offset_sd, uint64_t seed) {
    if (white_sd != 0.f) { const float4 n = normal4(e >> 2, seed, 0u); v.x = fmaf(white_sd, n.x, v.x); v.y = fmaf(white_sd, n.y, v.y); v.z = fmaf(white_sd, n.z, v.z); v.w = fmaf(white_sd, n.w, v.w); }
    if (offset_sd != 0.f) { const float4 n = normal4(eo >> 2, seed, 1u); v.x = fmaf(offset_sd, n.x, v.x); v.y = fmaf(offset_sd, n.y, v.y); v.z = fmaf(offset_sd, n.z, v.z); v.w = fmaf(offset_sd, n.w, v.w); }
    return v;
}
__device__ __forceinline__ float add_input_noise1(float v, size_t e, size_t eo, float white_sd, float offset_sd, uint64_t seed) {
    if (white_sd != 0.f) v = fmaf(white_sd, normal1(e, seed, 0u), v);
    if (offset_sd != 0.f) v = fmaf(offset_sd, normal1(eo, seed, 1u), v);
    return v;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

}  // namespace nsd
