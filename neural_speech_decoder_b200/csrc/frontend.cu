// K1: fused Gaussian smoothing + per-day affine + softsign + unfold, and its backward.
//
// Replaces F.conv1d(groups=N, padding="same") + index_select + einsum + Softsign + nn.Unfold
// (reference augmentations.py:91, model.py:84-101).  One pass over X: a CTA owns one utterance
// and a contiguous range of output frames, walks along time in blocks of TT rows, keeps the
// last K+TT rows of z in a shared-memory ring and emits every frame whose window is complete.
// X is read once (plus a (ntaps-1)-row halo per block), ys/z are written once for the backward,
// patches are written once with 16-byte stores in time-major row order (m = j*B + b).
#include <algorithm>

#include "common.cuh"

namespace nsd {

constexpr int FE_TT = 32;       // z rows computed per block
constexpr int FE_NTAPS = 20;    // the reference's smoothing kernel size (augmentations.py / model.py:84): unrolled fast path
constexpr int FE_TTP = 36;      // padded row length of the transposed ys tile (float4-aligned, conflict-free)

struct FrontendFwdParams {
    const float* x; const int64_t* day_idx; const float* day_w; const float* day_b; const float* taps;
    float* ys; float* z; void* patches; int* err_flag;
    int ntaps, B, T, N, n_days, K, S, Tp, frames_per_seg, ring;
    float white_sd, offset_sd; unsigned long long noise_seed;   // fused training augmentation (trainer:194-201); 0 = off
};

// ---- warp-level tensor-core pieces of the bf16 front end (the 256x256 day affine is a tiny GEMM fused between HBM-bound
// stages: mma.sync m16n8k16 on register-resident weight fragments, not a tcgen05 pipeline)
__device__ __forceinline__ uint32_t pack2_bf16(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(smem_row);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* smem_row) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(smem_row);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}

// NTW = 0: fp32 FFMA day affine (the fp32 parity path, any N).  NTW > 0: bf16 tensor-core day affine, N = 8*NTW*NWARPS:
// warp w owns output channels [8*NTW*w, 8*NTW*(w+1)) and keeps its slice of dayWeights[day] as mma B fragments in
// registers for the whole CTA; the smoothed block is the A operand (bf16, shared memory), fp32 accumulate.  The
// competition shape (N = 256) runs 16 warps with NTW = 2: 64 weight registers per thread instead of 128, twice the warps
// to hide the shared-memory and HBM latency of the four phases of a block.
template <typename OutT, int NTW, int NWARPS>
__global__ void __launch_bounds__(32 * NWARPS, 1) frontend_fwd_kernel(FrontendFwdParams p) {
    pdl_enter();
    constexpr int FE_THREADS = 32 * NWARPS;
    extern __shared__ __align__(16) float smem[];
    const int N = p.N, K = p.K, S = p.S, T = p.T, ntaps = p.ntaps;
    const int left = (ntaps - 1) / 2;
    const int xrows = FE_TT + ntaps - 1;
    const int NP = N + 1;
    constexpr int KS = NTW * NWARPS / 2;                    // k-steps of 16 input channels (N / 16)
    constexpr int NA = NTW * NWARPS * 8 + 8;                // padded row length (bf16) of the A tile: conflict-free ldmatrix
    float* taps_s = smem;                                   // [64]
    float* xs = smem + 64;                                  // [xrows][N]
    float* ysT = xs + (((size_t)xrows * N + 3) & ~(size_t)3);   // 16-byte aligned (float4 / ldmatrix reads) for any N.
                                                            // SIMT: [N][FE_TTP] f32;  TC: [FE_TT][NA] bf16
    float* zring = ysT + (NTW > 0 ? (size_t)FE_TT * NA / 2 : (size_t)N * FE_TTP);   // [ring][N+1]
    __nv_bfloat16* ysA = reinterpret_cast<__nv_bfloat16*>(ysT);

    const int b = blockIdx.x;
    const int j0 = blockIdx.y * p.frames_per_seg;
    const int j1 = min(p.Tp, j0 + p.frames_per_seg);
    if (j0 >= j1) return;
    const int tid = threadIdx.x;
    const bool noisy = (p.white_sd != 0.f) || (p.offset_sd != 0.f);

    long long day = p.day_idx[b];
    if (day < 0 || day >= p.n_days) {          // reference: index_select raises IndexError (model.py:89)
        if (tid == 0 && p.err_flag) *p.err_flag = 1;
        day = 0;
    }
    const float* W = p.day_w + (size_t)day * N * N;
    const float* bias = p.day_b + (size_t)day * N;
    if (tid < ntaps) taps_s[tid] = p.taps[tid];

    const int warp = tid >> 5, lane = tid & 31, fg = lane >> 2, fc = lane & 3;     // mma fragment coordinates
    uint32_t wfrag[NTW > 0 ? NTW : 1][NTW > 0 ? KS : 1][2];
    float bfrag[NTW > 0 ? NTW : 1][2];
    if constexpr (NTW > 0) {
#pragma unroll
        for (int j = 0; j < NTW; ++j) {
            const int n = (warp * NTW + j) * 8 + fg;                               // B[k = d][n]: this lane's output channel
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                const float* w0 = W + (size_t)(16 * ks + 2 * fc) * N + n;
                wfrag[j][ks][0] = pack2_bf16(__ldg(w0), __ldg(w0 + N));
                wfrag[j][ks][1] = pack2_bf16(__ldg(w0 + 8 * (size_t)N), __ldg(w0 + 9 * (size_t)N));
            }
            bfrag[j][0] = __ldg(bias + (warp * NTW + j) * 8 + 2 * fc);
            bfrag[j][1] = __ldg(bias + (warp * NTW + j) * 8 + 2 * fc + 1);
        }
    }

    // constant-offset noise of this thread's channel quad (valid when the staging loop's stride keeps the quad fixed)
    const bool off_fixed = ((N & 3) == 0) && (FE_THREADS % (N >> 2)) == 0;
    float4 off4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (noisy && off_fixed && p.offset_sd != 0.f) off4 = normal4(((size_t)b * N + 4 * (tid % (N >> 2))) >> 2, p.noise_seed, 1u);

    // z rows this CTA writes: its frames' windows and, when the stride is longer than the window, the rows up to the next
    // segment's first frame -- no frame reads them, but the backward walks every row of [0, (Tp-1)*S+K) (ys^T dpre)
    const int R0 = j0 * S, R1 = max((j1 - 1) * S + K, j1 < p.Tp ? j1 * S : 0);
    const float* xb = p.x + (size_t)b * T * N;
    float* ysb = p.ys + (size_t)b * T * N;
    float* zb = p.z + (size_t)b * T * N;
    int jnext = j0;

    for (int rb = R0; rb < R1; rb += FE_TT) {
        const int rows = min(FE_TT, R1 - rb);
        // 1. stage x rows [rb-left, rb-left+xrows) (zero outside [0,T))
        if ((N & 3) == 0) {
            const int n4 = N >> 2;
            for (int i = tid; i < xrows * n4; i += FE_THREADS) {
                int rr = i / n4, c4 = i - rr * n4;
                int t = rb - left + rr;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (t >= 0 && t < T && rr < rows + ntaps - 1) {
                    v = __ldg(reinterpret_cast<const float4*>(xb + (size_t)t * N) + c4);
                    if (noisy) {
                        // same operations, in the same order, as add_input_noise4 (the stand-alone kernel); the per-utterance
                        // offset does not depend on t: when the thread's channel quad is loop-invariant it is generated once
                        if (p.white_sd != 0.f) v = add_input_noise4(v, ((size_t)b * T + t) * N + 4 * c4, 0, p.white_sd, 0.f, p.noise_seed);
                        if (p.offset_sd != 0.f) {
                            const float4 o = off_fixed ? off4 : normal4(((size_t)b * N + 4 * c4) >> 2, p.noise_seed, 1u);
                            v.x = fmaf(p.offset_sd, o.x, v.x); v.y = fmaf(p.offset_sd, o.y, v.y);
                            v.z = fmaf(p.offset_sd, o.z, v.z); v.w = fmaf(p.offset_sd, o.w, v.w);
                        }
                    }
                }
                reinterpret_cast<float4*>(xs + (size_t)rr * N)[c4] = v;
            }
        } else {
            for (int i = tid; i < xrows * N; i += FE_THREADS) {
                int rr = i / N, c = i - rr * N;
                int t = rb - left + rr;
                float v = 0.f;
                if (t >= 0 && t < T) {
                    v = __ldg(xb + (size_t)t * N + c);
                    if (noisy) v = add_input_noise1(v, ((size_t)b * T + t) * N + c, (size_t)b * N + c, p.white_sd, p.offset_sd, p.noise_seed);
                }
                xs[i] = v;
            }
        }
        __syncthreads();
        // 2. depthwise FIR: ys[t][c] = sum_k taps[k] * x[t-left+k][c]
        if (ntaps == FE_NTAPS && (FE_THREADS % N) == 0 && (FE_TT % (FE_THREADS / N)) == 0) {
            // fast path: a thread owns one channel and FE_TT / (FE_THREADS / N) consecutive rows; the rows' input window is
            // read once into registers (RPT + 19 shared-memory loads instead of 2 * 20 * RPT) and the taps stay in registers
            constexpr int RPT_MAX = FE_TT;
            const int parts = FE_THREADS / N, rpt = FE_TT / parts;
            const int c = tid % N, r0 = (tid / N) * rpt;
            float tp[FE_NTAPS];
#pragma unroll
            for (int k = 0; k < FE_NTAPS; ++k) tp[k] = taps_s[k];
            if (rpt == 16) {
                float w[16 + FE_NTAPS - 1];
#pragma unroll
                for (int i = 0; i < 16 + FE_NTAPS - 1; ++i) w[i] = xs[(size_t)(r0 + i) * N + c];
#pragma unroll
                for (int tt = 0; tt < 16; ++tt) {
                    float acc = 0.f;
#pragma unroll
                    for (int k = 0; k < FE_NTAPS; ++k) acc = fmaf(tp[k], w[tt + k], acc);
                    if (r0 + tt < rows) ysb[(size_t)(rb + r0 + tt) * N + c] = acc; else acc = 0.f;
                    if constexpr (NTW > 0) ysA[(size_t)(r0 + tt) * NA + c] = __float2bfloat16_rn(acc);
                    else ysT[(size_t)c * FE_TTP + r0 + tt] = acc;
                }
            } else {
                (void)RPT_MAX;
                for (int tt = r0; tt < r0 + rpt; ++tt) {
                    float acc = 0.f;
                    if (tt < rows) {
#pragma unroll
                        for (int k = 0; k < FE_NTAPS; ++k) acc = fmaf(tp[k], xs[(size_t)(tt + k) * N + c], acc);
                        ysb[(size_t)(rb + tt) * N + c] = acc;
                    }
                    if constexpr (NTW > 0) ysA[(size_t)tt * NA + c] = __float2bfloat16_rn(acc);
                    else ysT[(size_t)c * FE_TTP + tt] = acc;
                }
            }
        } else
        for (int c = tid; c < N; c += FE_THREADS) {
            for (int tt = 0; tt < FE_TT; ++tt) {
                float acc = 0.f;
                if (tt < rows) {
                    for (int k = 0; k < ntaps; ++k) acc = fmaf(taps_s[k], xs[(size_t)(tt + k) * N + c], acc);
                    ysb[(size_t)(rb + tt) * N + c] = acc;
                }
                if constexpr (NTW > 0) ysA[(size_t)tt * NA + c] = __float2bfloat16_rn(acc);
                else ysT[(size_t)c * FE_TTP + tt] = acc;
            }
        }
        __syncthreads();
        // 3. day affine + softsign: pre[t][k] = sum_d ys[t][d] W[d][k] + bias[k]
        if constexpr (NTW > 0) {
            float acc[2][NTW][4];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int j = 0; j < NTW; ++j) { acc[mt][j][0] = acc[mt][j][2] = bfrag[j][0]; acc[mt][j][1] = acc[mt][j][3] = bfrag[j][1]; }
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    uint32_t a[4];
                    ldmatrix_x4(a, ysA + (size_t)(16 * mt + (lane & 7) + 8 * ((lane >> 3) & 1)) * NA + 16 * ks + 8 * (lane >> 4));
#pragma unroll
                    for (int j = 0; j < NTW; ++j) mma_bf16_16816(acc[mt][j], a, wfrag[j][ks][0], wfrag[j][ks][1]);
                }
            }
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int j = 0; j < NTW; ++j)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int i = 16 * mt + fg + 8 * h, col = (warp * NTW + j) * 8 + 2 * fc;
                        if (i < rows) {
                            const float a0 = acc[mt][j][2 * h], a1 = acc[mt][j][2 * h + 1];
                            const float v0 = a0 / (1.0f + fabsf(a0)), v1 = a1 / (1.0f + fabsf(a1));
                            float* zr = zring + (size_t)((rb + i) & (p.ring - 1)) * NP + col;
                            zr[0] = v0; zr[1] = v1;
                            *reinterpret_cast<float2*>(zb + (size_t)(rb + i) * N + col) = make_float2(v0, v1);
                        }
                    }
        } else
        for (int kc = tid; kc < N; kc += FE_THREADS) {
            float acc[FE_TT];
            const float bv = __ldg(bias + kc);
#pragma unroll
            for (int i = 0; i < FE_TT; ++i) acc[i] = bv;
            for (int d = 0; d < N; ++d) {
                const float w = __ldg(W + (size_t)d * N + kc);
                const float4* yr = reinterpret_cast<const float4*>(ysT + (size_t)d * FE_TTP);
#pragma unroll
                for (int q = 0; q < FE_TT / 4; ++q) {
                    float4 y = yr[q];
                    acc[4 * q + 0] = fmaf(y.x, w, acc[4 * q + 0]);
                    acc[4 * q + 1] = fmaf(y.y, w, acc[4 * q + 1]);
                    acc[4 * q + 2] = fmaf(y.z, w, acc[4 * q + 2]);
                    acc[4 * q + 3] = fmaf(y.w, w, acc[4 * q + 3]);
                }
            }
#pragma unroll
            for (int i = 0; i < FE_TT; ++i) {
                if (i < rows) {
                    float v = acc[i] / (1.0f + fabsf(acc[i]));
                    zring[(size_t)((rb + i) & (p.ring - 1)) * NP + kc] = v;
                    zb[(size_t)(rb + i) * N + kc] = v;
                }
            }
        }
        __syncthreads();
        // 4. emit every frame whose window [j*S, j*S+K) is now complete
        const int rend = rb + rows;
        int jend = jnext;
        while (jend < j1 && jend * S + K <= rend) ++jend;
        const int F = N * K;
        if ((K & 3) == 0) {
            const int f4n = F >> 2;
            // thread-invariant patch coordinates when the thread stride (4 * FE_THREADS features) is a multiple of K
            const bool fixed_kk = ((4 * FE_THREADS) % K) == 0;
            const int c_first = (4 * tid) / K, kk_first = (4 * tid) - c_first * K, c_step = (4 * FE_THREADS) / K;
            const int rmask = p.ring - 1;
            for (int j = jnext; j < jend; ++j) {
                OutT* orow = reinterpret_cast<OutT*>(p.patches) + ((size_t)j * p.B + b) * F;
                int c = c_first;
                for (int q = tid; q < f4n; q += FE_THREADS, c += c_step) {
                    int kk = kk_first;
                    if (!fixed_kk) { const int f = q << 2; c = f / K; kk = f - c * K; }
                    const int r = j * S + kk;
                    const float* zc = zring + c;
                    float v0 = zc[(size_t)((r + 0) & rmask) * NP];
                    float v1 = zc[(size_t)((r + 1) & rmask) * NP];
                    float v2 = zc[(size_t)((r + 2) & rmask) * NP];
                    float v3 = zc[(size_t)((r + 3) & rmask) * NP];
                    if constexpr (sizeof(OutT) == 4) {
                        reinterpret_cast<float4*>(orow)[q] = make_float4(v0, v1, v2, v3);
                    } else {
                        __nv_bfloat162 lo = __floats2bfloat162_rn(v0, v1), hi = __floats2bfloat162_rn(v2, v3);
                        uint2 u;
                        u.x = *reinterpret_cast<uint32_t*>(&lo);
                        u.y = *reinterpret_cast<uint32_t*>(&hi);
                        reinterpret_cast<uint2*>(orow)[q] = u;
                    }
                }
            }
        } else {
            for (int j = jnext; j < jend; ++j) {
                OutT* orow = reinterpret_cast<OutT*>(p.patches) + ((size_t)j * p.B + b) * F;
                for (int f = tid; f < F; f += FE_THREADS) {
                    int c = f / K, kk = f - c * K;
                    orow[f] = from_f32<OutT>(zring[(size_t)((j * S + kk) & (p.ring - 1)) * NP + c]);
                }
            }
        }
        jnext = jend;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// The benchmark shape's forward (N = 256 channels, 20 taps, bf16 patches, kernelLen in {8,16,32,64}, strideLen % 4 == 0): same four
// stages and the same arithmetic as frontend_fwd_kernel<bf16, 2, 16> (bit-identical outputs), re-cut to need a third of its instructions:
//   * the 19-row FIR halo of a block is moved inside shared memory instead of being re-read from HBM and re-noised (Philox + Box-Muller
//     ran on 51 rows per 32 produced), and the next block's 32 new rows are prefetched into registers under the day-affine MMAs;
//   * z lives in the ring as bf16 -- the rounding the patches get anyway -- TRANSPOSED (channel-major, time inner), so a 16-byte patch
//     store reads two 8-byte shared-memory words instead of eight strided fp32 cells + four converts; three CTA barriers per block, not four.
constexpr int FF_THREADS = 512, FF_N = 256, FF_NTW = 2, FF_KS = 16, FF_NA = FF_N + 8, FF_XROWS = FE_TT + FE_NTAPS - 1, FF_LEFT = (FE_NTAPS - 1) / 2;
constexpr int FF_HALO = FE_NTAPS - 1;                       // rows kept from one block to the next
constexpr int FF_NPRE = FE_TT * (FF_N / 4) / FF_THREADS;    // float4 prefetch registers per thread (4)

__device__ __forceinline__ float4 ff_noise(float4 v, const FrontendFwdParams& p, int b, int t, int c4, const float4& off4) {
    // same operations, in the same order, as add_input_noise4 (the stand-alone kernel)
    if (p.white_sd != 0.f) v = add_input_noise4(v, ((size_t)b * p.T + t) * FF_N + 4 * c4, 0, p.white_sd, 0.f, p.noise_seed);
    if (p.offset_sd != 0.f) {
        v.x = fmaf(p.offset_sd, off4.x, v.x); v.y = fmaf(p.offset_sd, off4.y, v.y);
        v.z = fmaf(p.offset_sd, off4.z, v.z); v.w = fmaf(p.offset_sd, off4.w, v.w);
    }
    return v;
}

template <int K8N>      // 16-byte chunks per channel of a patch row = kernelLen / 8
__global__ void __launch_bounds__(FF_THREADS, 1) frontend_fwd_fast_kernel(FrontendFwdParams p) {
    pdl_enter();
    extern __shared__ __align__(16) float smem[];
    constexpr int N = FF_N, K = 8 * K8N;
    const int S = p.S, T = p.T;
    const int pitch = p.ring + 4, rmask = p.ring - 1;                      // bf16 elements per channel row of the ring (pitch/2 = 2 mod 4 words)
    float* xs = smem;                                                      // [FF_XROWS][N] f32
    __nv_bfloat16* ysA = reinterpret_cast<__nv_bfloat16*>(xs + (size_t)FF_XROWS * N);      // [FE_TT][FF_NA] bf16
    __nv_bfloat16* zT = ysA + (size_t)FE_TT * FF_NA;                       // [N][pitch] bf16
    float* taps_s = reinterpret_cast<float*>(zT + (size_t)N * pitch);      // [FE_NTAPS]

    const int b = blockIdx.x;
    const int j0 = blockIdx.y * p.frames_per_seg;
    const int j1 = min(p.Tp, j0 + p.frames_per_seg);
    if (j0 >= j1) return;
    const int tid = threadIdx.x;
    const bool noisy = (p.white_sd != 0.f) || (p.offset_sd != 0.f);

    long long day = p.day_idx[b];
    if (day < 0 || day >= p.n_days) {          // reference: index_select raises IndexError (model.py:89)
        if (tid == 0 && p.err_flag) *p.err_flag = 1;
        day = 0;
    }
    const float* W = p.day_w + (size_t)day * N * N;
    const float* bias = p.day_b + (size_t)day * N;

    if (tid < FE_NTAPS) taps_s[tid] = p.taps[tid];
    const int warp = tid >> 5, lane = tid & 31, fg = lane >> 2, fc = lane & 3;     // mma fragment coordinates
    uint32_t wfrag[FF_NTW][FF_KS][2];
    float bfrag[FF_NTW][2];
#pragma unroll
    for (int j = 0; j < FF_NTW; ++j) {
        const int n = (warp * FF_NTW + j) * 8 + fg;                                // B[k = d][n]: this lane's output channel
#pragma unroll
        for (int ks = 0; ks < FF_KS; ++ks) {
            const float* w0 = W + (size_t)(16 * ks + 2 * fc) * N + n;
            wfrag[j][ks][0] = pack2_bf16(__ldg(w0), __ldg(w0 + N));
            wfrag[j][ks][1] = pack2_bf16(__ldg(w0 + 8 * (size_t)N), __ldg(w0 + 9 * (size_t)N));
        }
        bfrag[j][0] = __ldg(bias + (warp * FF_NTW + j) * 8 + 2 * fc);
        bfrag[j][1] = __ldg(bias + (warp * FF_NTW + j) * 8 + 2 * fc + 1);
    }

    const int c4 = tid & (N / 4 - 1), rq = tid >> 6;                               // staging: this thread's channel quad and first row
    float4 off4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (noisy && p.offset_sd != 0.f) off4 = normal4(((size_t)b * N + 4 * c4) >> 2, p.noise_seed, 1u);

    // z rows this CTA writes: its frames' windows and, when the stride is longer than the window, the rows up to the next
    // segment's first frame -- no frame reads them, but the backward walks every row of [0, (Tp-1)*S+K) (ys^T dpre)
    const int R0 = j0 * S, R1 = max((j1 - 1) * S + K, j1 < p.Tp ? j1 * S : 0);
    const float* xb = p.x + (size_t)b * T * N;
    float* ysb = p.ys + (size_t)b * T * N;
    float* zb = p.z + (size_t)b * T * N;
    int jnext = j0;

    // emission coordinates: a thread's 16-byte chunks all sit at the same offset inside the K-long window of a channel
    constexpr int E_CSTEP = FF_THREADS / K8N, E_NC = (N + E_CSTEP - 1) / E_CSTEP, F = N * K;        // channels a thread steps by; chunks per thread and frame
    const int e_k8 = tid & (K8N - 1), e_c0 = tid / K8N;
    const __nv_bfloat16* e_z = zT + (size_t)e_c0 * pitch;
    const size_t frame_stride = (size_t)p.B * F;

    // prologue: all FF_XROWS rows of the first block
    for (int rr = rq; rr < FF_XROWS; rr += FF_THREADS / (N / 4)) {
        const int t = R0 - FF_LEFT + rr;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t >= 0 && t < T) {
            v = __ldg(reinterpret_cast<const float4*>(xb + (size_t)t * N) + c4);
            if (noisy) v = ff_noise(v, p, b, t, c4, off4);
        }
        reinterpret_cast<float4*>(xs + (size_t)rr * N)[c4] = v;
    }
    __syncthreads();

    for (int rb = R0; rb < R1; rb += FE_TT) {
        const int rows = min(FE_TT, R1 - rb);
        const bool has_next = rb + FE_TT < R1;
        // 2. depthwise FIR: a thread owns one channel and 16 consecutive rows; window and taps in registers
        {
            const int c = tid & (N - 1), r0 = (tid >> 8) * 16;
            float tp[FE_NTAPS];
#pragma unroll
            for (int k = 0; k < FE_NTAPS; ++k) tp[k] = taps_s[k];
            float w[16 + FE_NTAPS - 1];
#pragma unroll
            for (int i = 0; i < 16 + FE_NTAPS - 1; ++i) w[i] = xs[(size_t)(r0 + i) * N + c];
            float* yo = ysb + (size_t)(rb + r0) * N + c;
            __nv_bfloat16* ya = ysA + (size_t)r0 * FF_NA + c;
            if (rows == FE_TT) {                            // every block but the last of a segment: no per-row predicates
#pragma unroll
                for (int tt = 0; tt < 16; ++tt) {
                    float acc = 0.f;
#pragma unroll
                    for (int k = 0; k < FE_NTAPS; ++k) acc = fmaf(tp[k], w[tt + k], acc);
                    yo[(size_t)tt * N] = acc;
                    ya[(size_t)tt * FF_NA] = __float2bfloat16_rn(acc);
                }
            } else {
#pragma unroll
                for (int tt = 0; tt < 16; ++tt) {
                    float acc = 0.f;
#pragma unroll
                    for (int k = 0; k < FE_NTAPS; ++k) acc = fmaf(tp[k], w[tt + k], acc);
                    if (r0 + tt < rows) yo[(size_t)tt * N] = acc; else acc = 0.f;
                    ya[(size_t)tt * FF_NA] = __float2bfloat16_rn(acc);
                }
            }
        }
        __syncthreads();
        // 3. halo rows move to the front of xs; the next block's new rows start their trip from HBM; day affine + softsign
        float4 pre[FF_NPRE];
        if (has_next) {
            for (int i = tid; i < FF_HALO * (N / 4); i += FF_THREADS)
                reinterpret_cast<float4*>(xs)[i] = reinterpret_cast<const float4*>(xs)[i + FE_TT * (N / 4)];
#pragma unroll
            for (int k = 0; k < FF_NPRE; ++k) {
                const int t = rb + FE_TT - FF_LEFT + FF_HALO + rq + 8 * k;
                pre[k] = (t >= 0 && t < T) ? __ldg(reinterpret_cast<const float4*>(xb + (size_t)t * N) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        {
            float acc[2][FF_NTW][4];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int j = 0; j < FF_NTW; ++j) { acc[mt][j][0] = acc[mt][j][2] = bfrag[j][0]; acc[mt][j][1] = acc[mt][j][3] = bfrag[j][1]; }
#pragma unroll
            for (int ks = 0; ks < FF_KS; ++ks) {
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    uint32_t a[4];
                    ldmatrix_x4(a, ysA + (size_t)(16 * mt + (lane & 7) + 8 * ((lane >> 3) & 1)) * FF_NA + 16 * ks + 8 * (lane >> 4));
#pragma unroll
                    for (int j = 0; j < FF_NTW; ++j) mma_bf16_16816(acc[mt][j], a, wfrag[j][ks][0], wfrag[j][ks][1]);
                }
            }
            const int col0 = warp * FF_NTW * 8 + 2 * fc;
            float* zo = zb + (size_t)(rb + fg) * N + col0;
            __nv_bfloat16* zr0 = zT + (size_t)col0 * pitch;
            const bool full = rows == FE_TT;
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int i = 16 * mt + fg + 8 * h;
                    if (full || i < rows) {
                        const int pos = (rb + i) & rmask;
#pragma unroll
                        for (int j = 0; j < FF_NTW; ++j) {
                            const float a0 = acc[mt][j][2 * h], a1 = acc[mt][j][2 * h + 1];
                            const float v0 = a0 / (1.0f + fabsf(a0)), v1 = a1 / (1.0f + fabsf(a1));
                            __nv_bfloat16* zr = zr0 + (size_t)(8 * j) * pitch + pos;
                            zr[0] = __float2bfloat16_rn(v0); zr[pitch] = __float2bfloat16_rn(v1);
                            *reinterpret_cast<float2*>(zo + (size_t)(16 * mt + 8 * h) * N + 8 * j) = make_float2(v0, v1);
                        }
                    }
                }
        }
        __syncthreads();
        // 4. the prefetched rows (+ noise) land behind the halo; emit every frame whose window [j*S, j*S+K) is now complete
        if (has_next) {
#pragma unroll
            for (int k = 0; k < FF_NPRE; ++k) {
                const int rr = FF_HALO + rq + 8 * k, t = rb + FE_TT - FF_LEFT + rr;
                float4 v = pre[k];
                if (noisy && t >= 0 && t < T) v = ff_noise(v, p, b, t, c4, off4);
                reinterpret_cast<float4*>(xs + (size_t)rr * N)[c4] = v;
            }
        }
        const int rend = rb + rows;
        int jend = jnext;
        while (jend < j1 && jend * S + K <= rend) ++jend;
        if (jnext < jend) {
            __nv_bfloat16* orow = reinterpret_cast<__nv_bfloat16*>(p.patches) + ((size_t)jnext * p.B + b) * F + (size_t)e_c0 * K + 8 * e_k8;
            int pos = jnext * S + 8 * e_k8;
            for (int j = jnext; j < jend; ++j, orow += frame_stride, pos += S) {
                const int pos0 = pos & rmask, pos1 = (pos + 4) & rmask;
#pragma unroll
                for (int i = 0; i < E_NC; ++i) {
                    if (E_CSTEP > N && e_c0 >= N) break;                    // kernelLen 8: fewer chunks per frame than threads
                    const __nv_bfloat16* zc = e_z + (size_t)(i * E_CSTEP) * pitch;
                    const uint2 lo = *reinterpret_cast<const uint2*>(zc + pos0), hi = *reinterpret_cast<const uint2*>(zc + pos1);
                    *reinterpret_cast<uint4*>(orow + (size_t)(i * E_CSTEP) * K) = make_uint4(lo.x, lo.y, hi.x, hi.y);
                }
            }
        }
        jnext = jend;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// backward: col2im (deterministic, thread-owned ring cells) -> softsign' -> ys^T dpre per utterance
// ---------------------------------------------------------------------------------------------
constexpr int FB_THREADS = 256;
constexpr int FB_CN = 128;     // channels (columns of dW) per CTA
constexpr int FB_G = 4;        // frames staged per group
constexpr int FB_RCH = 16;     // rows finalised per chunk

struct FrontendBwdParams {
    const void* dp; const float* ys; const float* z; float* partial_w; float* partial_b;
    int B, T, N, K, S, Tp, KP, ring;
};

template <typename InT>
__global__ void __launch_bounds__(FB_THREADS, 1) frontend_bwd_kernel(FrontendBwdParams p) {
    pdl_enter();
    extern __shared__ __align__(16) float smem[];
    const int N = p.N, K = p.K, S = p.S, T = p.T, KP = p.KP, B = p.B;
    const int b = blockIdx.x;
    const int c0 = blockIdx.y * FB_CN;
    const int cn = min(FB_CN, N - c0);
    const int tid = threadIdx.x;
    const int kl = tid & (FB_CN - 1);   // column within the chunk
    const int dh = tid >> 7;            // which 128-row half of d this thread accumulates
    const int RP = FB_CN + 1;
    float* ring = smem;                                     // [ring][FB_CN+1]
    float* ys_s = ring + (size_t)p.ring * RP;               // [FB_RCH][N]
    float* stage = ys_s + (size_t)FB_RCH * N;               // [FB_G][FB_CN][KP]

    for (int i = tid; i < p.ring * RP; i += FB_THREADS) ring[i] = 0.f;

    const int nd_chunks = (N + 255) / 256;                  // d handled in chunks of 256 (2 halves x 128)
    const float* ysb = p.ys + (size_t)b * T * N;
    const float* zb = p.z + (size_t)b * T * N;
    const InT* dp = reinterpret_cast<const InT*>(p.dp);
    const int F = N * K;

    for (int dc = 0; dc < nd_chunks; ++dc) {
        const int d0 = dc * 256 + dh * 128;
        float acc[128];
#pragma unroll
        for (int i = 0; i < 128; ++i) acc[i] = 0.f;
        float bacc = 0.f;
        __syncthreads();

        auto finalize = [&](int r_begin, int r_end) {
            for (int rc = r_begin; rc < r_end; rc += FB_RCH) {
                const int nr = min(FB_RCH, r_end - rc);
                for (int i = tid; i < nr * N; i += FB_THREADS) ys_s[i] = __ldg(ysb + (size_t)rc * N + i);
                __syncthreads();
                if (kl < cn) {
                    for (int rr = 0; rr < nr; ++rr) {
                        const int t = rc + rr;
                        float dz = ring[(size_t)(t & (p.ring - 1)) * RP + kl];
                        float zz = __ldg(zb + (size_t)t * N + c0 + kl);
                        float s = 1.0f - fabsf(zz);
                        float dpre = dz * s * s;
                        if (dh == 0) bacc += dpre;
                        const float* yr = ys_s + (size_t)rr * N + d0;
                        if ((N & 3) == 0 && d0 + 128 <= N) {          // float4 rows: 16-byte aligned only when N % 4 == 0
#pragma unroll
                            for (int q = 0; q < 32; ++q) {
                                float4 y = reinterpret_cast<const float4*>(yr)[q];
                                acc[4 * q + 0] = fmaf(y.x, dpre, acc[4 * q + 0]);
                                acc[4 * q + 1] = fmaf(y.y, dpre, acc[4 * q + 1]);
                                acc[4 * q + 2] = fmaf(y.z, dpre, acc[4 * q + 2]);
                                acc[4 * q + 3] = fmaf(y.w, dpre, acc[4 * q + 3]);
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < 128; ++i)
                                if (d0 + i < N) acc[i] = fmaf(yr[i], dpre, acc[i]);
                        }
                    }
                }
                __syncthreads();
                // consumed rows go back to zero for their next use
                for (int i = tid; i < nr * FB_CN; i += FB_THREADS)
                    ring[(size_t)((rc + i / FB_CN) & (p.ring - 1)) * RP + (i % FB_CN)] = 0.f;
                __syncthreads();
            }
        };

        for (int jg = 0; jg < p.Tp; jg += FB_G) {
            const int ng = min(FB_G, p.Tp - jg);
            // a. stage this CTA's slice of ng gradient rows (coalesced)
            for (int g = 0; g < ng; ++g) {
                const InT* row = dp + ((size_t)(jg + g) * B + b) * F + (size_t)c0 * K;
                float* st = stage + (size_t)g * FB_CN * KP;
                for (int i = tid; i < cn * K; i += FB_THREADS) {
                    int cl = i / K, kk = i - cl * K;
                    st[cl * KP + kk] = to_f32<InT>(row[i]);
                }
            }
            __syncthreads();
            // b. scatter-add into the ring; a thread owns (cl, phase) so no two threads touch one cell
            for (int pi = tid; pi < cn * S; pi += FB_THREADS) {
                const int cl = pi / S, ph = pi - cl * S;
                for (int g = 0; g < ng; ++g) {
                    const float* st = stage + (size_t)g * FB_CN * KP + cl * KP;
                    const int rbase = (jg + g) * S;
                    for (int kk = ph; kk < K; kk += S) ring[(size_t)((rbase + kk) & (p.ring - 1)) * RP + cl] += st[kk];
                }
            }
            __syncthreads();
            // c. rows below the next group's first row are complete
            const bool last = (jg + ng >= p.Tp);
            finalize(jg * S, last ? (p.Tp - 1) * S + K : (jg + ng) * S);
        }
        // write this utterance's partial dW rows / db
        if (kl < cn) {
            float* pw = p.partial_w + (size_t)b * N * N;
#pragma unroll
            for (int i = 0; i < 128; ++i)
                if (d0 + i < N) pw[(size_t)(d0 + i) * N + c0 + kl] = acc[i];
            if (dh == 0 && dc == 0) p.partial_b[(size_t)b * N + c0 + kl] = bacc;
        }
    }
}

// Tensor-core form of the backward for the bf16 model path (dpatches bf16, N = 128 * MT): same col2im ring and softsign',
// but the per-utterance ys^T dpre (the 2*T*N*N FLOPs that made the FFMA kernel instruction-bound) runs on mma.sync m16n8k16
// with bf16 operands and fp32 accumulators held in registers for the whole utterance: warp w owns rows d in
// [16*MT*w, 16*MT*(w+1)) of dW, all FB_CN = 128 columns of the CTA's column block.
template <int MT>
__global__ void __launch_bounds__(FB_THREADS, 1) frontend_bwd_tc_kernel(FrontendBwdParams p) {
    pdl_enter();
    extern __shared__ __align__(16) float smem[];
    constexpr int N = 128 * MT, NYS = N + 8, NDP = FB_CN + 8;
    const int K = p.K, S = p.S, T = p.T, KP = p.KP, B = p.B;
    const int b = blockIdx.x;
    const int c0 = blockIdx.y * FB_CN;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int kl = tid & (FB_CN - 1);   // column within the chunk
    const int half = tid >> 7;          // which 8 of a chunk's 16 rows this thread turns into dpre
    const int RP = FB_CN + 1;
    float* ring = smem;                                                           // [ring][FB_CN+1]
    float* stage = ring + (((size_t)p.ring * RP + 3) & ~(size_t)3);               // [FB_G][FB_CN][KP], 16-byte aligned
    __nv_bfloat16* ys_s = reinterpret_cast<__nv_bfloat16*>(stage + (size_t)FB_G * FB_CN * KP);   // [16][N+8]
    __nv_bfloat16* dp_s = ys_s + 16 * NYS;                                        // [16][FB_CN+8]
    float* bsum = reinterpret_cast<float*>(dp_s + 16 * NDP);                      // [FB_CN]

    for (int i = tid; i < p.ring * RP; i += FB_THREADS) ring[i] = 0.f;
    const float* ysb = p.ys + (size_t)b * T * N;
    const float* zb = p.z + (size_t)b * T * N;
    const __nv_bfloat16* dp = reinterpret_cast<const __nv_bfloat16*>(p.dp);
    const int F = N * K;

    float acc[MT][FB_CN / 8][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int nt = 0; nt < FB_CN / 8; ++nt)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;
    float bacc = 0.f;
    __syncthreads();

    auto finalize = [&](int r_begin, int r_end) {
        for (int rc = r_begin; rc < r_end; rc += 16) {
            const int nr = min(16, r_end - rc);
            // A^T tile: 16 rows of ys as bf16 (zero rows past nr)
            for (int i = tid; i < 16 * (N / 4); i += FB_THREADS) {
                const int rr = i / (N / 4), c4 = i - rr * (N / 4);
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (rr < nr) v = __ldg(reinterpret_cast<const float4*>(ysb + (size_t)(rc + rr) * N) + c4);
                *reinterpret_cast<uint2*>(ys_s + (size_t)rr * NYS + 4 * c4) = make_uint2(pack2_bf16(v.x, v.y), pack2_bf16(v.z, v.w));
            }
            // B tile: dpre = col2im(dpatches) * softsign'(z), this thread's column, 8 of the 16 rows
            {
                float zz[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int rr = 8 * half + q;
                    zz[q] = (rr < nr) ? __ldg(zb + (size_t)(rc + rr) * N + c0 + kl) : 0.f;
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int rr = 8 * half + q;
                    float dpre = 0.f;
                    if (rr < nr) {
                        const float sg = 1.0f - fabsf(zz[q]);
                        dpre = ring[(size_t)((rc + rr) & (p.ring - 1)) * RP + kl] * sg * sg;
                    }
                    bacc += dpre;
                    dp_s[(size_t)rr * NDP + kl] = __float2bfloat16_rn(dpre);
                }
            }
            __syncthreads();
            {
                uint32_t a[MT][4];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
                    ldmatrix_x4_trans(a[mt], ys_s + (size_t)((lane & 7) + 8 * (lane >> 4)) * NYS + (warp * MT + mt) * 16 + 8 * ((lane >> 3) & 1));
#pragma unroll
                for (int np = 0; np < FB_CN / 16; ++np) {
                    uint32_t bq[4];
                    ldmatrix_x4_trans(bq, dp_s + (size_t)((lane & 7) + 8 * ((lane >> 3) & 1)) * NDP + 16 * np + 8 * (lane >> 4));
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        mma_bf16_16816(acc[mt][2 * np], a[mt], bq[0], bq[1]);
                        mma_bf16_16816(acc[mt][2 * np + 1], a[mt], bq[2], bq[3]);
                    }
                }
            }
            // consumed rows go back to zero for their next use
            for (int i = tid; i < nr * FB_CN; i += FB_THREADS)
                ring[(size_t)((rc + i / FB_CN) & (p.ring - 1)) * RP + (i % FB_CN)] = 0.f;
            __syncthreads();
        }
    };

    for (int jg = 0; jg < p.Tp; jg += FB_G) {
        const int ng = min(FB_G, p.Tp - jg);
        // a. stage this CTA's slice of ng gradient rows (coalesced 16-byte loads when K % 8 == 0)
        for (int g = 0; g < ng; ++g) {
            const __nv_bfloat16* row = dp + ((size_t)(jg + g) * B + b) * F + (size_t)c0 * K;
            float* st = stage + (size_t)g * FB_CN * KP;
            if ((K & 7) == 0) {
                for (int i = tid; i < FB_CN * K / 8; i += FB_THREADS) {
                    const int e = 8 * i, cl = e / K, kk = e - cl * K;
                    const uint4 u = __ldg(reinterpret_cast<const uint4*>(row) + i);
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
                    float* d = st + cl * KP + kk;
                    const float2 f0 = __bfloat1622float2(h[0]), f1 = __bfloat1622float2(h[1]), f2 = __bfloat1622float2(h[2]), f3 = __bfloat1622float2(h[3]);
                    *reinterpret_cast<float4*>(d) = make_float4(f0.x, f0.y, f1.x, f1.y);
                    *reinterpret_cast<float4*>(d + 4) = make_float4(f2.x, f2.y, f3.x, f3.y);
                }
            } else {
                for (int i = tid; i < FB_CN * K; i += FB_THREADS) {
                    const int cl = i / K, kk = i - cl * K;
                    st[cl * KP + kk] = __bfloat162float(row[i]);
                }
            }
        }
        __syncthreads();
        // b. scatter-add into the ring; a thread owns (cl, phase) so no two threads touch one cell
        for (int pi = tid; pi < FB_CN * S; pi += FB_THREADS) {
            const int cl = pi / S, ph = pi - cl * S;
            for (int g = 0; g < ng; ++g) {
                const float* st = stage + (size_t)g * FB_CN * KP + cl * KP;
                const int rbase = (jg + g) * S;
                for (int kk = ph; kk < K; kk += S) ring[(size_t)((rbase + kk) & (p.ring - 1)) * RP + cl] += st[kk];
            }
        }
        __syncthreads();
        // c. rows below the next group's first row are complete
        const bool last = (jg + ng >= p.Tp);
        finalize(jg * S, last ? (p.Tp - 1) * S + K : (jg + ng) * S);
    }
    // this utterance's partial dW block / db: C fragment (row = lane/4 (+8), cols 2*(lane%4), +1)
    float* pw = p.partial_w + (size_t)b * N * N;
    const int fg = lane >> 2, fc = lane & 3;
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int nt = 0; nt < FB_CN / 8; ++nt)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int d = (warp * MT + mt) * 16 + fg + 8 * h;
                *reinterpret_cast<float2*>(pw + (size_t)d * N + c0 + 8 * nt + 2 * fc) = make_float2(acc[mt][nt][2 * h], acc[mt][nt][2 * h + 1]);
            }
    if (half == 1) bsum[kl] = bacc;
    __syncthreads();
    if (half == 0) p.partial_b[(size_t)b * N + c0 + kl] = bacc + bsum[kl];
}

// Competition-shape form of the tensor-core backward (N = 256, kernelLen 32, stride 4, bf16 dpatches): 16 warps, and the
// col2im runs in REGISTERS.  Thread (cl, ph) owns channel cl of the CTA's 128-column block and the rows t = ph (mod 4): a
// row receives one tap from each of the K/S = 8 frames that cover it, so 8 rotating partial sums per thread are enough -- frame j
// adds its taps ph, ph+4, .., ph+28 to the 8 sums and completes row 4j+ph.  No shared-memory ring, no read-modify-write,
// two barriers per group of 4 frames (= one 16-row mma chunk): stage -> [col2im, softsign', bf16 tiles] -> mma, with the
// tile buffers double-buffered so the mma of one group runs under the staging of the next.
constexpr int FB2_THREADS = 512;
__global__ void __launch_bounds__(FB2_THREADS, 1) frontend_bwd_tc2_kernel(FrontendBwdParams p) {
    pdl_enter();
    extern __shared__ __align__(16) float smem[];
    constexpr int N = 256, K = 32, S = 4, NYS = N + 8, NDP = FB_CN + 8, KP = 36, G = 4;
    const int T = p.T, B = p.B, Tp = p.Tp;
    const int b = blockIdx.x;
    const int c0 = blockIdx.y * FB_CN;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int cl = tid >> 2, ph = tid & 3;
    float* stage = smem;                                                                   // [G][FB_CN][KP] f32
    __nv_bfloat16* ys_s = reinterpret_cast<__nv_bfloat16*>(stage + (size_t)G * FB_CN * KP);   // [2][16][N+8]
    __nv_bfloat16* dp_s = ys_s + 2 * 16 * NYS;                                             // [2][16][FB_CN+8]
    const float* ysb = p.ys + (size_t)b * T * N;
    const float* zb = p.z + (size_t)b * T * N;
    const __nv_bfloat16* dp = reinterpret_cast<const __nv_bfloat16*>(p.dp);
    constexpr int F = N * K;

    float acc[FB_CN / 8][4];                     // dW rows [16*warp, 16*warp+16) x the CTA's 128 columns (mma C fragments)
#pragma unroll
    for (int nt = 0; nt < FB_CN / 8; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[nt][i] = 0.f;
    float slot[8];                               // partial col2im sums of rows 4j+ph .. 4(j+7)+ph
#pragma unroll
    for (int i = 0; i < 8; ++i) slot[i] = 0.f;
    float bacc = 0.f;
    const int last_row = (Tp - 1) * S + K - 1;   // last z row any frame touches
    const int ngroups = (Tp + 7 + G - 1) / G;    // real frames + 7 virtual (empty) frames that flush the rotating sums
    int buf = 0;
    for (int grp = 0; grp < ngroups; grp += 2) {
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
            const int jg = (grp + hf) * G;
            if (jg >= ngroups * G) break;
            // a. stage this CTA's slice of up to 4 gradient rows (coalesced 16-byte loads), f32 in shared memory
            for (int i = tid; i < G * FB_CN * K / 8; i += FB2_THREADS) {
                const int g = i / (FB_CN * K / 8), r = i - g * (FB_CN * K / 8);
                const int e = 8 * r, c = e / K, kk = e - c * K;
                if (jg + g < Tp) {
                    const uint4 u = __ldg(reinterpret_cast<const uint4*>(dp + ((size_t)(jg + g) * B + b) * F + (size_t)c0 * K) + r);
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
                    float* d = stage + (size_t)g * FB_CN * KP + c * KP + kk;
                    const float2 f0 = __bfloat1622float2(h[0]), f1 = __bfloat1622float2(h[1]), f2 = __bfloat1622float2(h[2]), f3 = __bfloat1622float2(h[3]);
                    *reinterpret_cast<float4*>(d) = make_float4(f0.x, f0.y, f1.x, f1.y);
                    *reinterpret_cast<float4*>(d + 4) = make_float4(f2.x, f2.y, f3.x, f3.y);
                }
            }
            // A^T tile: the 16 rows of ys this group completes, as bf16 (zero rows past the end)
            __nv_bfloat16* ysw = ys_s + (size_t)buf * 16 * NYS;
            __nv_bfloat16* dpw = dp_s + (size_t)buf * 16 * NDP;
            for (int i = tid; i < 16 * (N / 4); i += FB2_THREADS) {
                const int rr = i / (N / 4), c4 = i - rr * (N / 4);
                const int t = jg * S + rr;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (t <= last_row) v = __ldg(reinterpret_cast<const float4*>(ysb + (size_t)t * N) + c4);
                *reinterpret_cast<uint2*>(ysw + (size_t)rr * NYS + 4 * c4) = make_uint2(pack2_bf16(v.x, v.y), pack2_bf16(v.z, v.w));
            }
            float zz[G];
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int t = (jg + g) * S + ph;
                zz[g] = (t <= last_row) ? __ldg(zb + (size_t)t * N + c0 + cl) : 0.f;
            }
            __syncthreads();
            // b. register col2im: frame jg+g adds tap ph+4i to the sum of row 4(jg+g+i)+ph, then row 4(jg+g)+ph is complete
#pragma unroll
            for (int g = 0; g < G; ++g) {
                constexpr int dummy = 0; (void)dummy;
                const int sl0 = (4 * hf + g) & 7;                    // static after unrolling: slot of the row this frame completes
                if (jg + g < Tp) {
                    const float* st = stage + (size_t)g * FB_CN * KP + cl * KP + ph;
#pragma unroll
                    for (int i = 0; i < 8; ++i) slot[(sl0 + i) & 7] += st[4 * i];
                }
                const int t = (jg + g) * S + ph;
                float dpre = 0.f;
                if (t <= last_row) {
                    const float sg = 1.0f - fabsf(zz[g]);
                    dpre = slot[sl0] * sg * sg;
                }
                slot[sl0] = 0.f;
                bacc += dpre;
                dpw[(size_t)(4 * g + ph) * NDP + cl] = __float2bfloat16_rn(dpre);
            }
            __syncthreads();
            // c. dW[d][c] += sum over the 16 rows of ys[row][d] * dpre[row][c] on mma.sync (bf16 operands, fp32 accumulate)
            {
                uint32_t a[4];
                ldmatrix_x4_trans(a, ysw + (size_t)((lane & 7) + 8 * (lane >> 4)) * NYS + warp * 16 + 8 * ((lane >> 3) & 1));
#pragma unroll
                for (int np = 0; np < FB_CN / 16; ++np) {
                    uint32_t bq[4];
                    ldmatrix_x4_trans(bq, dpw + (size_t)((lane & 7) + 8 * ((lane >> 3) & 1)) * NDP + 16 * np + 8 * (lane >> 4));
                    mma_bf16_16816(acc[2 * np], a, bq[0], bq[1]);
                    mma_bf16_16816(acc[2 * np + 1], a, bq[2], bq[3]);
                }
            }
            buf ^= 1;
        }
    }
    // this utterance's partial dW block / db: C fragment (row = lane/4 (+8), cols 2*(lane%4), +1)
    float* pw = p.partial_w + (size_t)b * N * N;
    const int fg = lane >> 2, fc = lane & 3;
#pragma unroll
    for (int nt = 0; nt < FB_CN / 8; ++nt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int d = warp * 16 + fg + 8 * h;
            *reinterpret_cast<float2*>(pw + (size_t)d * N + c0 + 8 * nt + 2 * fc) = make_float2(acc[nt][2 * h], acc[nt][2 * h + 1]);
        }
    bacc += __shfl_xor_sync(0xffffffffu, bacc, 1);          // the four phases of a channel sit in adjacent lanes
    bacc += __shfl_xor_sync(0xffffffffu, bacc, 2);
    if (ph == 0) p.partial_b[(size_t)b * N + c0 + cl] = bacc;
}

// ---------------------------------------------------------------------------------------------
// backward w.r.t. X: col2im -> softsign' -> dy = dpre W_day^T -> transposed smoothing FIR, in one launch.
// The smoother is "same"-padded, ys[t] = sum_k taps[k] x[t-L+k] (L = (ntaps-1)/2, x zero outside [0,T)), so
// dx[s] = sum_k taps[k] dy[s+L-k] over 0 <= s+L-k < T.  A CTA owns utterance b and the output rows [R0, R1); it walks dy
// rows [R0-(ntaps-1-L), R1+L) in tiles of FI_TR, keeps the last rows of dy in a shared-memory ring and writes every dx row
// whose window is complete.  Neighbouring segments recompute the ntaps-1 rows of dy they share.  dz of a row is gathered
// straight from the frames that cover it, frames in ascending order as in nsd_frontend_bwd; every sum is in a fixed order.
// NTW = 0: fp32 FFMA product (any N, either dpatches dtype).  NTW > 0: bf16 dpatches, N = 8*NTW*NWARPS, the product on
// mma.sync m16n8k16 with W_day as register-resident B fragments (B[k][n] = W[n][k]), fp32 accumulate.
// ---------------------------------------------------------------------------------------------
constexpr int FI_TR = 16;       // dy rows per tile (one mma M tile)

struct FrontendBwdInputParams {
    const void* dp; const float* z; const int64_t* day_idx; const float* day_w; const float* taps; float* dx;
    int ntaps, B, T, N, n_days, K, S, Tp, Tz, rows_per_seg, ring;
};

template <typename InT, int NTW, int NWARPS>
__global__ void __launch_bounds__(32 * NWARPS, 1) frontend_bwd_input_kernel(FrontendBwdInputParams p) {
    pdl_enter();
    constexpr int THREADS = 32 * NWARPS;
    constexpr int KS = NTW * NWARPS / 2;                    // k-steps of 16 channels (N / 16)
    constexpr int NA = NTW * NWARPS * 8 + 8;                // padded row length (bf16) of the dpre tile: conflict-free ldmatrix
    extern __shared__ __align__(16) float smem[];
    const int N = p.N, K = p.K, S = p.S, T = p.T, ntaps = p.ntaps;
    const int L = (ntaps - 1) / 2, A = ntaps - 1 - L;
    const int NP = (N + 3) & ~3, rmask = p.ring - 1;
    float* taps_s = smem;                                   // [64]
    float* ring = smem + 64;                                // [ring][NP] rows of dy
    float* tile = ring + (size_t)p.ring * NP;               // SIMT: [FI_TR][NP] f32;  TC: [FI_TR][NA] bf16
    __nv_bfloat16* tileA = reinterpret_cast<__nv_bfloat16*>(tile);

    const int b = blockIdx.x;
    const int R0 = blockIdx.y * p.rows_per_seg, R1 = min(T, R0 + p.rows_per_seg);
    if (R0 >= R1) return;
    const int tid = threadIdx.x;
    long long day = p.day_idx[b];
    if (day < 0 || day >= p.n_days) day = 0;                // the forward has flagged it
    const float* W = p.day_w + (size_t)day * N * N;
    if (tid < ntaps) taps_s[tid] = p.taps[tid];

    const int warp = tid >> 5, lane = tid & 31, fg = lane >> 2, fc = lane & 3;     // mma fragment coordinates
    uint32_t wfrag[NTW > 0 ? NTW : 1][NTW > 0 ? KS : 1][2];
    if constexpr (NTW > 0) {
#pragma unroll
        for (int j = 0; j < NTW; ++j) {
            const float* w0 = W + (size_t)((warp * NTW + j) * 8 + fg) * N + 2 * fc;  // B[k][n] = W[n][k]: this lane's output channel n
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                wfrag[j][ks][0] = pack2_bf16(__ldg(w0 + 16 * ks), __ldg(w0 + 16 * ks + 1));
                wfrag[j][ks][1] = pack2_bf16(__ldg(w0 + 16 * ks + 8), __ldg(w0 + 16 * ks + 9));
            }
        }
    }

    const InT* dpb = reinterpret_cast<const InT*>(p.dp) + (size_t)b * N * K;
    const size_t frame_stride = (size_t)p.B * N * K;
    const float* zb = p.z + (size_t)b * T * N;
    const int Y1 = R1 + L;
    int s_next = R0;
    for (int ty = R0 - A; s_next < R1; ty += FI_TR) {
        const int nr = min(FI_TR, Y1 - ty);
        // 1. dpre tile: rows fastest, so that a warp's lanes read consecutive taps of one frame row
        for (int i = tid; i < FI_TR * N; i += THREADS) {
            const int c = i / FI_TR, r = i - c * FI_TR, t = ty + r;
            float dpre = 0.f;
            if (r < nr && t >= 0 && t < p.Tz) {
                const int jlo = t < K ? 0 : (t - K + S) / S, jhi = min(p.Tp - 1, t / S);
                float dz = 0.f;
                for (int j = jlo; j <= jhi; ++j) dz += to_f32<InT>(dpb[(size_t)j * frame_stride + (size_t)c * K + (t - j * S)]);
                const float sg = 1.0f - fabsf(__ldg(zb + (size_t)t * N + c));
                dpre = dz * sg * sg;
            }
            if constexpr (NTW > 0) tileA[(size_t)r * NA + c] = __float2bfloat16_rn(dpre);
            else tile[(size_t)r * NP + c] = dpre;
        }
        __syncthreads();
        // 2. dy[t][n] = sum_k dpre[t][k] W[n][k] into the ring
        if constexpr (NTW > 0) {
            float acc[NTW][4];
#pragma unroll
            for (int j = 0; j < NTW; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                uint32_t a[4];
                ldmatrix_x4(a, tileA + (size_t)((lane & 7) + 8 * ((lane >> 3) & 1)) * NA + 16 * ks + 8 * (lane >> 4));
#pragma unroll
                for (int j = 0; j < NTW; ++j) mma_bf16_16816(acc[j], a, wfrag[j][ks][0], wfrag[j][ks][1]);
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int r = fg + 8 * h;
                if (r < nr) {
                    float* dr = ring + (size_t)((ty + r) & rmask) * NP;
#pragma unroll
                    for (int j = 0; j < NTW; ++j)
                        *reinterpret_cast<float2*>(dr + (warp * NTW + j) * 8 + 2 * fc) = make_float2(acc[j][2 * h], acc[j][2 * h + 1]);
                }
            }
        } else {
            for (int n = tid; n < N; n += THREADS) {
                float acc[FI_TR];
#pragma unroll
                for (int r = 0; r < FI_TR; ++r) acc[r] = 0.f;
                const float* wr = W + (size_t)n * N;
                if ((N & 3) == 0) {                           // 16-byte aligned W rows and tile rows
                    for (int k4 = 0; k4 < N / 4; ++k4) {
                        const float4 w = __ldg(reinterpret_cast<const float4*>(wr) + k4);
#pragma unroll
                        for (int r = 0; r < FI_TR; ++r) {
                            const float4 a = reinterpret_cast<const float4*>(tile + (size_t)r * NP)[k4];
                            acc[r] = fmaf(a.x, w.x, acc[r]); acc[r] = fmaf(a.y, w.y, acc[r]);
                            acc[r] = fmaf(a.z, w.z, acc[r]); acc[r] = fmaf(a.w, w.w, acc[r]);
                        }
                    }
                } else {
                    for (int k = 0; k < N; ++k) {
                        const float w = __ldg(wr + k);
#pragma unroll
                        for (int r = 0; r < FI_TR; ++r) acc[r] = fmaf(tile[(size_t)r * NP + k], w, acc[r]);
                    }
                }
#pragma unroll
                for (int r = 0; r < FI_TR; ++r)
                    if (r < nr) ring[(size_t)((ty + r) & rmask) * NP + n] = acc[r];
            }
        }
        __syncthreads();
        // 3. dx rows whose window [s+L-(ntaps-1), s+L] is in the ring: a thread owns one channel and 4 consecutive rows, reads the
        // ntaps+3 dy rows they share once, and sums each output over k in ascending order
        const int s_end = min(R1, ty + FI_TR - L);
        if (s_end > s_next) {
            const int ngrp = (s_end - s_next + 3) >> 2;
            for (int i = tid; i < ngrp * N; i += THREADS) {
                const int g = i / N, c = i - g * N, s0 = s_next + 4 * g;
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                for (int m = ntaps + 2; m >= 0; --m) {
                    const float v = ring[(size_t)((s0 + L - ntaps + 1 + m) & rmask) * NP + c];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int k = q + ntaps - 1 - m;
                        if (k >= 0 && k < ntaps) acc[q] = fmaf(taps_s[k], v, acc[q]);
                    }
                }
                float* out = p.dx + ((size_t)b * T + s0) * N + c;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (s0 + q < s_end) out[(size_t)q * N] = acc[q];
            }
            s_next = s_end;
        }
        __syncthreads();
    }
}

// out[d][e] = sum_{b : day[b]==d} partial[b][e], utterances visited in index order (deterministic).
__global__ void day_segment_reduce_kernel(const float* __restrict__ pw, const float* __restrict__ pb,
                                          const int64_t* __restrict__ day_idx, int B, int NN, int N, int n_days,
                                          float* __restrict__ dw, float* __restrict__ db) {
    pdl_enter();
    const int d = blockIdx.y;
    const int per = NN + N;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < per; e += gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int b = 0; b < B; ++b) {
            if (day_idx[b] == d) s += (e < NN) ? pw[(size_t)b * NN + e] : pb[(size_t)b * N + (e - NN)];
        }
        if (e < NN) dw[(size_t)d * NN + e] = s;
        else db[(size_t)d * N + (e - NN)] = s;
    }
}

// stand-alone form of the augmentation (same values as the fused path): out = x + white + offset
__global__ void input_noise_kernel(const float* __restrict__ x, float* __restrict__ out, int B, int T, int N, float white_sd, float offset_sd,
                                   unsigned long long seed, const unsigned long long* __restrict__ seed_off) {
    pdl_enter();
    if (seed_off) seed += *seed_off;
    const size_t total = (size_t)B * T * N;
    if ((N & 3) == 0) {
        for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total / 4; q += (size_t)gridDim.x * blockDim.x) {
            const size_t e = 4 * q, b = e / ((size_t)T * N), c = e % N;
            float4 v = reinterpret_cast<const float4*>(x)[q];
            reinterpret_cast<float4*>(out)[q] = add_input_noise4(v, e, b * N + c, white_sd, offset_sd, seed);
        }
    } else {
        for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
            const size_t b = e / ((size_t)T * N), c = e % N;
            out[e] = add_input_noise1(x[e], e, b * N + c, white_sd, offset_sd, seed);
        }
    }
}

static int pick_segments(int B, int Tp, int sms, int S, int K) {
    // minimise waves/segments: time ~ ceil(B*nseg/sms)/nseg, halo recompute grows with nseg
    int best = 1;
    double best_cost = 1e30;
    for (int n = 1; n <= 16 && n <= Tp; ++n) {
        int fps = (Tp + n - 1) / n;
        double waves = (double)((B * n + sms - 1) / sms);
        double cost = waves * (fps * S + K - S);
        if (cost < best_cost - 1e-9) { best_cost = cost; best = n; }
    }
    return best;
}

}  // namespace nsd

extern "C" {

int nsd_frontend_fwd(const float* x, const int64_t* day_idx, const float* day_w, const float* day_b,
                     const float* taps, int ntaps, int B, int T, int N, int n_days, int kernel_len,
                     int stride_len, float* ys, float* z, void* patches, int patches_dtype, int* err_flag,
                     float white_noise_sd, float constant_offset_sd, uint64_t noise_seed, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(B > 0 && T > 0 && N > 0 && n_days > 0, "frontend_fwd: bad sizes B=%d T=%d N=%d", B, T, N);
    NSD_CHECK_ARG(ntaps >= 1 && ntaps <= 64, "frontend_fwd: ntaps=%d not in [1,64]", ntaps);
    NSD_CHECK_ARG(kernel_len >= 1 && stride_len >= 1, "frontend_fwd: bad kernel/stride");
    NSD_CHECK_ARG(T >= kernel_len, "frontend_fwd: T=%d shorter than kernelLen=%d", T, kernel_len);
    NSD_CHECK_ARG(patches_dtype == NSD_F32 || patches_dtype == NSD_BF16, "frontend_fwd: bad dtype");
    FrontendFwdParams p;
    p.x = x; p.day_idx = day_idx; p.day_w = day_w; p.day_b = day_b; p.taps = taps;
    p.ys = ys; p.z = z; p.patches = patches; p.err_flag = err_flag;
    p.white_sd = white_noise_sd; p.offset_sd = constant_offset_sd; p.noise_seed = noise_seed;
    p.ntaps = ntaps; p.B = B; p.T = T; p.N = N; p.n_days = n_days; p.K = kernel_len; p.S = stride_len;
    p.Tp = (T - kernel_len) / stride_len + 1;
    const int nseg = pick_segments(B, p.Tp, sm_count(), stride_len, kernel_len);
    p.frames_per_seg = cdiv(p.Tp, nseg);
    p.ring = 1;
    while (p.ring < kernel_len + FE_TT) p.ring <<= 1;      // power of two: ring rows are addressed with a mask
    // bf16 patches (the tensor-core model path) with N in {64, 128, 256}: day affine on mma.sync; otherwise the exact fp32 FFMA form
    const bool tc = patches_dtype == NSD_BF16 && (N == 64 || N == 128 || N == 256);
    size_t smem = sizeof(float) * (64 + (((size_t)(FE_TT + ntaps - 1) * N + 3) & ~(size_t)3) + (size_t)p.ring * (N + 1) +
                                   (tc ? (size_t)FE_TT * (N + 8) / 2 : (size_t)N * FE_TTP));
    NSD_CHECK_ARG(smem <= 227 * 1024, "frontend_fwd: N=%d kernelLen=%d need %zu B shared memory", N, kernel_len, smem);
    dim3 grid(B, cdiv(p.Tp, p.frames_per_seg));
    cudaStream_t s = (cudaStream_t)stream;
    auto go = [&](auto kern, int threads) -> int {
        NSD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        nsd::launch_k(kern, grid, threads, smem, s, p);
        return NSD_OK;
    };
    int rc;
    const bool fast = tc && N == FF_N && ntaps == FE_NTAPS && (stride_len & 3) == 0 &&
                      (kernel_len == 8 || kernel_len == 16 || kernel_len == 32 || kernel_len == 64);
    if (fast) {
        smem = sizeof(float) * ((size_t)FF_XROWS * FF_N + 32) + 2 * ((size_t)FE_TT * FF_NA + (size_t)FF_N * (p.ring + 4));
        rc = kernel_len == 8 ? go(frontend_fwd_fast_kernel<1>, FF_THREADS) : kernel_len == 16 ? go(frontend_fwd_fast_kernel<2>, FF_THREADS)
           : kernel_len == 32 ? go(frontend_fwd_fast_kernel<4>, FF_THREADS) : go(frontend_fwd_fast_kernel<8>, FF_THREADS);
    } else if (patches_dtype == NSD_F32) rc = go(frontend_fwd_kernel<float, 0, 8>, 256);
    else if (tc && N == 256) rc = go(frontend_fwd_kernel<__nv_bfloat16, 2, 16>, 512);
    else if (tc && N == 128) rc = go(frontend_fwd_kernel<__nv_bfloat16, 1, 16>, 512);
    else if (tc && N == 64) rc = go(frontend_fwd_kernel<__nv_bfloat16, 1, 8>, 256);
    else rc = go(frontend_fwd_kernel<__nv_bfloat16, 0, 8>, 256);
    if (rc) return rc;
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

int nsd_input_noise(const float* x, float* out, int B, int T, int N, float white_noise_sd, float constant_offset_sd,
                    uint64_t seed, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(B >= 0 && T >= 0 && N > 0 && x && out, "input_noise: bad arguments");
    const size_t total = (size_t)B * T * N;
    if (total == 0) return NSD_OK;
    NSD_CHECK_ARG((N & 3) != 0 || ((((uintptr_t)x | (uintptr_t)out) & 15) == 0), "input_noise: x/out must be 16-byte aligned");
    const int blocks = (int)std::min<size_t>(cdivz(cdivz(total, 4), 256), (size_t)sm_count() * 16);
    nsd::launch_k(input_noise_kernel, blocks, 256, 0, (cudaStream_t)stream, x, out, B, T, N, white_noise_sd, constant_offset_sd, seed, seed_offset_ptr());
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

size_t nsd_frontend_bwd_workspace(int B, int N) { return sizeof(float) * (size_t)B * N * (N + 1); }

int nsd_frontend_bwd(const void* dpatches, int dpatches_dtype, const float* ys, const float* z,
                     const int64_t* day_idx, int B, int T, int N, int n_days, int kernel_len, int stride_len,
                     float* d_day_w, float* d_day_b, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(B > 0 && T >= kernel_len && N > 0 && n_days > 0, "frontend_bwd: bad sizes");
    NSD_CHECK_ARG(dpatches_dtype == NSD_F32 || dpatches_dtype == NSD_BF16, "frontend_bwd: bad dtype");
    if (workspace_bytes < nsd_frontend_bwd_workspace(B, N)) {
        set_error("frontend_bwd: workspace %zu < %zu", workspace_bytes, nsd_frontend_bwd_workspace(B, N));
        return NSD_ERR_WORKSPACE;
    }
    FrontendBwdParams p;
    p.dp = dpatches; p.ys = ys; p.z = z;
    p.partial_w = reinterpret_cast<float*>(workspace);
    p.partial_b = p.partial_w + (size_t)B * N * N;
    p.B = B; p.T = T; p.N = N; p.K = kernel_len; p.S = stride_len;
    p.Tp = (T - kernel_len) / stride_len + 1;
    p.KP = ((kernel_len + 3) / 4) * 4 + 4;
    p.ring = 1;
    while (p.ring < (FB_G - 1) * stride_len + kernel_len) p.ring <<= 1;   // power of two: ring rows are addressed with a mask
    cudaStream_t s = (cudaStream_t)stream;
    const int mt = (dpatches_dtype == NSD_BF16 && (N == 128 || N == 256)) ? N / 128 : 0;
    if (mt == 2 && kernel_len == 32 && stride_len == 4) {
        // competition shape: 16 warps, register col2im
        const size_t smem = sizeof(float) * (size_t)4 * FB_CN * 36 + sizeof(__nv_bfloat16) * (2 * 16 * (size_t)(N + 8) + 2 * 16 * (size_t)(FB_CN + 8));
        dim3 grid(B, N / FB_CN);
        NSD_CUDA(cudaFuncSetAttribute(frontend_bwd_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        nsd::launch_k(frontend_bwd_tc2_kernel, grid, FB2_THREADS, smem, s, p);
    } else if (mt) {
        // bf16 model path: per-utterance ys^T dpre on tensor cores
        size_t smem = sizeof(float) * ((((size_t)p.ring * (FB_CN + 1) + 3) & ~(size_t)3) + (size_t)FB_G * FB_CN * p.KP + FB_CN) +
                      sizeof(__nv_bfloat16) * (16 * (size_t)(N + 8) + 16 * (size_t)(FB_CN + 8));
        NSD_CHECK_ARG(smem <= 227 * 1024, "frontend_bwd: N=%d kernelLen=%d need %zu B shared memory", N, kernel_len, smem);
        dim3 grid(B, N / FB_CN);
        if (mt == 2) {
            NSD_CUDA(cudaFuncSetAttribute(frontend_bwd_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            nsd::launch_k(frontend_bwd_tc_kernel<2>, grid, FB_THREADS, smem, s, p);
        } else {
            NSD_CUDA(cudaFuncSetAttribute(frontend_bwd_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            nsd::launch_k(frontend_bwd_tc_kernel<1>, grid, FB_THREADS, smem, s, p);
        }
    } else {
    size_t smem = sizeof(float) * ((size_t)p.ring * (FB_CN + 1) + (size_t)FB_RCH * N + (size_t)FB_G * FB_CN * p.KP);
    NSD_CHECK_ARG(smem <= 227 * 1024, "frontend_bwd: N=%d kernelLen=%d need %zu B shared memory", N, kernel_len, smem);
    dim3 grid(B, cdiv(N, FB_CN));
    if (dpatches_dtype == NSD_F32) {
        NSD_CUDA(cudaFuncSetAttribute(frontend_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        nsd::launch_k(frontend_bwd_kernel<float>, grid, FB_THREADS, smem, s, p);
    } else {
        NSD_CUDA(cudaFuncSetAttribute(frontend_bwd_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        nsd::launch_k(frontend_bwd_kernel<__nv_bfloat16>, grid, FB_THREADS, smem, s, p);
    }
    }
    NSD_LAUNCH_CHECK();
    const int per = N * N + N;
    dim3 g2(min(cdiv(per, 256), 64), n_days);
    nsd::launch_k(day_segment_reduce_kernel, g2, 256, 0, s, p.partial_w, p.partial_b, day_idx, B, N * N, N, n_days, d_day_w, d_day_b);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

int nsd_frontend_bwd_input(const void* dpatches, int dpatches_dtype, const float* z, const int64_t* day_idx, const float* day_w,
                           const float* taps, int ntaps, int B, int T, int N, int n_days, int kernel_len, int stride_len,
                           float* dx, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(B > 0 && T > 0 && N > 0 && n_days > 0, "frontend_bwd_input: bad sizes B=%d T=%d N=%d", B, T, N);
    NSD_CHECK_ARG(ntaps >= 1 && ntaps <= 64, "frontend_bwd_input: ntaps=%d not in [1,64]", ntaps);
    NSD_CHECK_ARG(kernel_len >= 1 && stride_len >= 1, "frontend_bwd_input: bad kernel/stride");
    NSD_CHECK_ARG(T >= kernel_len, "frontend_bwd_input: T=%d shorter than kernelLen=%d", T, kernel_len);
    NSD_CHECK_ARG(dpatches_dtype == NSD_F32 || dpatches_dtype == NSD_BF16, "frontend_bwd_input: bad dtype");
    FrontendBwdInputParams p;
    p.dp = dpatches; p.z = z; p.day_idx = day_idx; p.day_w = day_w; p.taps = taps; p.dx = dx;
    p.ntaps = ntaps; p.B = B; p.T = T; p.N = N; p.n_days = n_days; p.K = kernel_len; p.S = stride_len;
    p.Tp = (T - kernel_len) / stride_len + 1;
    p.Tz = (p.Tp - 1) * stride_len + kernel_len;          // rows no frame covers have dz = 0
    p.ring = 1;
    while (p.ring < FI_TR + ntaps - 1) p.ring <<= 1;      // power of two: ring rows are addressed with a mask
    const bool tc = dpatches_dtype == NSD_BF16 && (N == 64 || N == 128 || N == 256);
    const size_t smem = sizeof(float) * (64 + (size_t)p.ring * ((N + 3) & ~3)) +
                        (tc ? sizeof(__nv_bfloat16) * FI_TR * (size_t)(N + 8) : sizeof(float) * FI_TR * (size_t)((N + 3) & ~3));
    NSD_CHECK_ARG(smem <= 227 * 1024, "frontend_bwd_input: N=%d ntaps=%d need %zu B shared memory", N, ntaps, smem);
    cudaStream_t s = (cudaStream_t)stream;
    auto go = [&](auto kern, int threads) -> int {
        NSD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 1;
        NSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
        // time segments: fewest waves of CTAs, each CTA paying its ntaps-1 recomputed dy rows
        const int sms = sm_count();
        int best = 1;
        double best_cost = 1e30;
        for (int n = 1; n <= 16 && n <= T; ++n) {
            const int rows = cdiv(T, n);
            const double cost = (double)cdiv(B * n, sms * std::max(per_sm, 1)) * (rows + ntaps - 1);
            if (cost < best_cost - 1e-9) { best_cost = cost; best = n; }
        }
        p.rows_per_seg = cdiv(T, best);
        nsd::launch_k(kern, dim3(B, cdiv(T, p.rows_per_seg)), threads, smem, s, p);
        return NSD_OK;
    };
    int rc;
    if (tc && N == 256) rc = go(frontend_bwd_input_kernel<__nv_bfloat16, 2, 16>, 512);
    else if (tc && N == 128) rc = go(frontend_bwd_input_kernel<__nv_bfloat16, 1, 16>, 512);
    else if (tc && N == 64) rc = go(frontend_bwd_input_kernel<__nv_bfloat16, 1, 8>, 256);
    else if (dpatches_dtype == NSD_BF16) rc = go(frontend_bwd_input_kernel<__nv_bfloat16, 0, 8>, 256);
    else rc = go(frontend_bwd_input_kernel<float, 0, 8>, 256);
    if (rc) return rc;
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

}  // extern "C"
