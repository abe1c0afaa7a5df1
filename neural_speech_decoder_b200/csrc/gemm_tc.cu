// K2 tensor-core path: C[M,N] = A[M,K] * B[N,K]^T (+bias[N]) (+beta*C), bf16 operands, fp32 accumulation.
//
// Hand-written sm_100a kernel: TMA (cp.async.bulk.tensor, 128-byte swizzle) stages K-major A / B tiles through a
// shared-memory ring, ONE elected thread issues tcgen05.mma (UMMA 128 x BN x 16, kind::f16) with the
// accumulator in tensor memory, and four epilogue warps drain TMEM with tcgen05.ld while the next tile's MMAs
// run into the second accumulator stage.  Persistent: one CTA per SM walks a grouped tile order.  Wide problems (N >= 192,
// M > 128) run the PAIR form further down: clusters of two CTAs, tcgen05.mma.cta_group::2 on 256 x 256 tiles.
// It backs the time-batched W_ih projections of nn.GRU (reference model.py:50-57, 119), their dgrad / wgrad and
// the time-batched W_hh wgrad.  Operands may be K-major or MN-major (both are native UMMA layouts).
#include <type_traits>

#include "tc_common.cuh"

namespace nsd {
namespace tc {

// SMs the persistent GEMM grids may occupy: all of them, minus the reserve set with nsd_set_gemm_sm_reserve (data-parallel
// training keeps a few SMs free for NCCL's CTAs while a gradient bucket is being all-reduced under the backward GEMMs, so
// that neither kernel has to wait for the other's CTAs to leave)
static int g_sm_reserve = 0;
static int gemm_sms() { return std::max(2, sm_count() - g_sm_reserve); }

constexpr int BM = 128;          // UMMA M (cta_group::1, all 128 TMEM lanes)
constexpr int THREADS = 256;     // warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc, warp 3 idle, warps 4-7 epilogue
constexpr int ACC_STAGES = 2;

template <int BN> struct Cfg {
    static constexpr int STAGES = (BN == 256) ? 4 : (BN == 128 ? 6 : 8);
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int TMEM_COLS = (ACC_STAGES * BN <= 32) ? 32 : (ACC_STAGES * BN <= 64 ? 64 : (ACC_STAGES * BN <= 128 ? 128 : (ACC_STAGES * BN <= 256 ? 256 : 512)));
    static constexpr int SMEM = STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 256 /*barriers*/;
};

struct TileCoord { int m_blk, n_blk; };
__device__ __forceinline__ TileCoord tile_coord(int t, int num_m, int num_n, int GROUP_M = 16) {
    // 16 m-blocks x ~9 n-blocks live at once on 148 SMs: both operands stay L2-resident
    const int per_group = GROUP_M * num_n;
    const int g = t / per_group;
    const int first_m = g * GROUP_M;
    const int gsz = min(GROUP_M, num_m - first_m);
    const int within = t - g * per_group;
    return {first_m + within % gsz, within / gsz};
}

// eight consecutive fp32 results as ONE 256-bit store (a full 32-byte sector per thread: the thread-per-row epilogue otherwise
// half-fills every sector it touches and backs up the LSU queue -- ncu: lg_throttle on the K = 2048 GEMMs)
__device__ __forceinline__ void store8_f32(float* p, const float (&v)[8]) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void store16_bf16(__nv_bfloat16* p, const uint32_t (&r)[32], int i, const float* bias_at) {
    uint32_t w[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        float lo = __uint_as_float(r[i + 2 * e]), hi = __uint_as_float(r[i + 2 * e + 1]);
        if (bias_at) { lo += __ldg(bias_at + 2 * e); hi += __ldg(bias_at + 2 * e + 1); }
        const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
        w[e] = *reinterpret_cast<const uint32_t*>(&v);
    }
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
}
template <typename OutT> __device__ __forceinline__ void store4(OutT* p, float a, float b, float c, float d);
template <> __device__ __forceinline__ void store4<float>(float* p, float a, float b, float c, float d) {
    *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
template <> __device__ __forceinline__ void store4<__nv_bfloat16>(__nv_bfloat16* p, float a, float b, float c, float d) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&lo);
    u.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(p) = u;
}

// One thread's 32 consecutive accumulator columns of row `row` (read from TMEM into r[0..31]) -> C[row, col0 .. col0+31], with the optional bias and
// beta*C terms.  Full 32-byte sectors per thread where alignment allows (256-bit fp32 / 16 x bf16 stores), element-wise at the matrix edge.
// Shared by the single-CTA and the cta_group::2 kernels.
template <typename OutT>
__device__ __forceinline__ void store_acc_row32(OutT* __restrict__ C, int ldc, int row, int col0, int M, int N, const uint32_t (&r)[32],
                                                const float* __restrict__ bias, float beta, bool vec_ok, bool vec8_ok) {
    if (row < M) {
        OutT* crow = C + (size_t)row * ldc + col0;
        if (std::is_same<OutT, float>::value && vec8_ok && beta == 0.f && col0 + 32 <= N) {
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(r[i + e]);
                if (bias) {
                    const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + col0 + i)), b1 = __ldg(reinterpret_cast<const float4*>(bias + col0 + i + 4));
                    v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w; v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
                }
                store8_f32(reinterpret_cast<float*>(crow) + i, v);
            }
        } else if (std::is_same<OutT, __nv_bfloat16>::value && vec8_ok && (ldc % 16) == 0 && beta == 0.f && col0 + 32 <= N) {
#pragma unroll
            for (int i = 0; i < 32; i += 16)
                store16_bf16(reinterpret_cast<__nv_bfloat16*>(crow) + i, r, i, bias ? bias + col0 + i : nullptr);
        } else if (vec_ok && col0 + 32 <= N) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
                float v0 = __uint_as_float(r[i]), v1 = __uint_as_float(r[i + 1]), v2 = __uint_as_float(r[i + 2]), v3 = __uint_as_float(r[i + 3]);
                if (bias) {
                    const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + col0 + i));
                    v0 += bv.x; v1 += bv.y; v2 += bv.z; v3 += bv.w;
                }
                if (beta != 0.f) {
                    v0 = fmaf(beta, to_f32<OutT>(crow[i]), v0); v1 = fmaf(beta, to_f32<OutT>(crow[i + 1]), v1);
                    v2 = fmaf(beta, to_f32<OutT>(crow[i + 2]), v2); v3 = fmaf(beta, to_f32<OutT>(crow[i + 3]), v3);
                }
                store4<OutT>(crow + i, v0, v1, v2, v3);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if (col0 + i < N) {
                    float v = __uint_as_float(r[i]);
                    if (bias) v += __ldg(bias + col0 + i);
                    if (beta != 0.f) v = fmaf(beta, to_f32<OutT>(crow[i]), v);
                    crow[i] = from_f32<OutT>(v);
                }
            }
        }
    }
}

// cluster helpers of the pair form below
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_id_x() { uint32_t r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t nclusters_x() { uint32_t r; asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
template <int BN, typename OutT, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, OutT* __restrict__ C, int ldc,
               const float* __restrict__ bias, float beta, int M, int N, int K) {
    pdl_launch_dependents();
    using cfg = Cfg<BN>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + cfg::STAGES * cfg::STAGE_BYTES);
    uint64_t* full_bar = bars;                             // [STAGES]  TMA -> MMA
    uint64_t* empty_bar = bars + cfg::STAGES;              // [STAGES]  MMA -> TMA
    uint64_t* tmem_full = bars + 2 * cfg::STAGES;          // [ACC_STAGES] MMA -> epilogue
    uint64_t* tmem_empty = tmem_full + ACC_STAGES;         // [ACC_STAGES] epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + ACC_STAGES);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int num_m = (M + BM - 1) / BM, num_n = (N + BN - 1) / BN;
    const int num_tiles = num_m * num_n;
    const int nk = (K + BK - 1) / BK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < cfg::STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < ACC_STAGES; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();                             // everything above ran under the previous kernel's tail; operands and C are touched below

    if (warp == 0) {
        // ===================== TMA producer (whole warp walks the ring, one elected lane issues) =====================
        // Warp-uniform control flow around elect.sync keeps descriptors / coordinates in uniform registers; a
        // `lane == 0` branch makes the compiler wrap every UTMALDG / UTCHMMA in an R2UR waterfall loop.
        int stage = 0; uint32_t phase = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
            const TileCoord tc = tile_coord(t, num_m, num_n);
            for (int kb = 0; kb < nk; ++kb) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                if (elect_one()) {
                    uint8_t* sa = smem + stage * cfg::STAGE_BYTES;
                    mbar_expect_tx(&full_bar[stage], cfg::STAGE_BYTES);
                    if constexpr (!A_MN) tma_load_2d(&tmA, &full_bar[stage], sa, kb * BK, tc.m_blk * BM);
                    else {
#pragma unroll
                        for (int i = 0; i < BM / 64; ++i) tma_load_2d(&tmA, &full_bar[stage], sa + i * 8192, tc.m_blk * BM + 64 * i, kb * BK);
                    }
                    if constexpr (!B_MN) tma_load_2d(&tmB, &full_bar[stage], sa + cfg::A_BYTES, kb * BK, tc.n_blk * BN);
                    else {
#pragma unroll
                        for (int i = 0; i < BN / 64; ++i) tma_load_2d(&tmB, &full_bar[stage], sa + cfg::A_BYTES + i * 8192, tc.n_blk * BN + 64 * i, kb * BK);
                    }
                }
                __syncwarp();
                if (++stage == cfg::STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (whole warp walks the ring, one elected lane issues) =====================
        constexpr uint32_t idesc = make_idesc_bf16(BM, BN, A_MN, B_MN);
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
            mbar_wait(&tmem_empty[acc], acc_phase ^ 1);          // epilogue has drained this accumulator
            tcgen05_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
            for (int kb = 0; kb < nk; ++kb) {
                mbar_wait(&full_bar[stage], phase);
                tcgen05_fence_after();
                if (elect_one()) {
                    const uint32_t sa = smem_u32(smem + stage * cfg::STAGE_BYTES);
                    const uint64_t adesc = A_MN ? make_mnmajor_sw128_desc(sa, 8192) : make_kmajor_sw128_desc(sa);
                    const uint64_t bdesc = B_MN ? make_mnmajor_sw128_desc(sa + cfg::A_BYTES, 8192) : make_kmajor_sw128_desc(sa + cfg::A_BYTES);
                    // K advance of 16 elements: 32 bytes along a K-major row, two 1024-byte k groups in an MN-major tile
                    constexpr uint64_t a_step = A_MN ? (2048 >> 4) : (32 >> 4), b_step = B_MN ? (2048 >> 4) : (32 >> 4);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k)
                        umma_bf16(d_tmem, adesc + a_step * k, bdesc + b_step * k, idesc, (kb | k) != 0);
                    umma_commit(&empty_bar[stage]);                   // smem slot reusable once these MMAs retire
                    if (kb == nk - 1) umma_commit(&tmem_full[acc]);   // accumulator complete -> epilogue
                }
                __syncwarp();
                if (++stage == cfg::STAGES) { stage = 0; phase ^= 1; }
            }
            if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
    } else if (warp >= 4) {
        // ===================== epilogue: TMEM -> registers -> global =====================
        const int q = warp & 3;                                       // TMEM lane quadrant this warp may read
        int acc = 0; uint32_t acc_phase = 0;
        const bool vec_ok = ((ldc % 4) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
        const bool vec8_ok = ((ldc % 8) == 0) && ((reinterpret_cast<uintptr_t>(C) & 31) == 0);
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
            const TileCoord tc = tile_coord(t, num_m, num_n);
            mbar_wait(&tmem_full[acc], acc_phase);
            tcgen05_fence_after();
            const int row = tc.m_blk * BM + q * 32 + lane;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                const int col0 = tc.n_blk * BN + c0;
                if (col0 >= N) break;                                 // warp-uniform
                uint32_t r[32];
                tmem_ld_32x32(taddr + (uint32_t)c0, r);
                store_acc_row32<OutT>(C, ldc, row, col0, M, N, r, bias, beta, vec_ok, vec8_ok);
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    if (warp == 2) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(cfg::TMEM_COLS) : "memory");
    }
}

// =====================================================================================================================
// Pair form (cta_group::2): the two CTAs of a cluster compute ONE 256 x 256 tile with a single stream of
// tcgen05.mma.cta_group::2 instructions issued by the leader (cluster rank 0).  Each CTA stages its own 128 rows of A and
// its own HALF of B (128 of the 256 n-rows) -- 32 KB per k-block instead of 48 KB -- so the ring is 6 stages deep instead
// of 4: with 128x256 tiles the 4-stage ring cannot cover a TMA round trip at the rate the tensor pipe drains it (measured:
// 3 stages cost 6-21 %).  Accumulator rows 0-127 live in the leader's TMEM, rows 128-255 in the peer's; each CTA's epilogue
// drains its own half.  Barriers: full[s] in the leader, completed by BOTH CTAs' TMA loads (cta_group::2 TMA form, barrier
// addressed in the leader's shared memory); empty[s] / tmem_full[a] in both CTAs (multicast commit); tmem_empty[a] in the leader (8 arrivals:
// four epilogue warps of each CTA).
// BN2 = 256 (default) or 128: the narrower tile halves the quantum of work, which pays when the 256-wide tiling leaves the
// last round of clusters mostly idle (picked per problem by pair_tile_width()).
template <int BN2> struct Cfg2 {
    static constexpr int BN = BN2, STAGES = (BN2 == 256) ? 7 : 9;
    static constexpr int A_BYTES = BM * BK * 2, B_BYTES = (BN / 2) * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int TMEM_COLS = ACC_STAGES * BN;      // 512 or 256
    static constexpr int SMEM = STAGES * STAGE_BYTES + 1024 + 512;
};
__device__ __forceinline__ uint32_t mapa_rank(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
// TMA into MY shared memory that completes a barrier which may live in the PAIR's other CTA (cluster address)
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* map, uint32_t bar_cluster_addr, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cl(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cl(uint64_t* bar, uint32_t parity) {        // barrier that a peer CTA arrives on
    if (mbar_try_wait_cl(bar, parity)) return;
    const long long t0 = clock64();
    unsigned int spins = 0;
    while (!mbar_try_wait_cl(bar, parity)) {
        if ((++spins & 0xFFFFu) == 0 && clock64() - t0 > SPIN_CYCLES) {
            printf("nsd gemm_tc2: cluster mbarrier timeout (block %d thread %d)\n", blockIdx.x, threadIdx.x);
            __trap();
        }
    }
}

// Up to TWO problems of identical shape in one launch (nprob = 2: operands tmA2 / tmB2, result C2): the two directions'
// W_hh weight gradients are 48 tile pairs each on 74 clusters -- together, with 128-wide tiles, they fill 2.6 rounds
// instead of leaving a third of the GPU idle twice.
template <typename OutT, bool A_MN, bool B_MN, int BN2>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2, OutT* __restrict__ C, OutT* __restrict__ C2,
                int ldc, const float* __restrict__ bias, float beta, int M, int N, int K, int nprob) {
    pdl_launch_dependents();
    using cfg = Cfg2<BN2>;
    constexpr int BN = cfg::BN;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + cfg::STAGES * cfg::STAGE_BYTES);
    uint64_t* full_bar = bars;                             // [STAGES]  leader only: both CTAs' TMA -> MMA
    uint64_t* empty_bar = bars + cfg::STAGES;              // [STAGES]  MMA (multicast commit) -> my TMA
    uint64_t* tmem_full = bars + 2 * cfg::STAGES;          // [ACC_STAGES] MMA (multicast commit) -> my epilogue
    uint64_t* tmem_empty = tmem_full + ACC_STAGES;         // [ACC_STAGES] leader only: both epilogues -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + ACC_STAGES);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int crank = (int)cluster_ctarank();
    const bool leader = crank == 0;
    const int num_m = (M + BM - 1) / BM, num_n = (N + BN - 1) / BN;
    const int nk = (K + BK - 1) / BK;
    const int num_mw = (num_m + 1) / 2;
    const int per_prob = num_mw * num_n;
    const int num_tiles = per_prob * nprob;
    const int w_first = (int)cluster_id_x(), w_step = (int)nclusters_x();
    auto coord_of = [&](int t) { TileCoord tc = tile_coord(t % per_prob, num_mw, num_n, 8); tc.m_blk = tc.m_blk * 2 + crank; return tc; };

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
        if (nprob > 1) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA2) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB2) : "memory");
        }
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < cfg::STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < ACC_STAGES; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();                             // everything above ran under the previous kernel's tail; operands and C are touched below

    if (warp == 0) {
        // ===================== TMA producer: my 128 rows of A, my half of B =====================
        // Both CTAs' loads complete the LEADER's full barrier (the one MMA issuer waits on one barrier per stage); the
        // leader expects the bytes of both.
        int stage = 0; uint32_t phase = 0;
        for (int t = w_first; t < num_tiles; t += w_step) {
            const TileCoord tc = coord_of(t);
            const CUtensorMap* mA = (t >= per_prob) ? &tmA2 : &tmA;
            const CUtensorMap* mB = (t >= per_prob) ? &tmB2 : &tmB;
            for (int kb = 0; kb < nk; ++kb) {
                mbar_wait_cl(&empty_bar[stage], phase ^ 1);
                if (elect_one()) {
                    uint8_t* sa = smem + stage * cfg::STAGE_BYTES;
                    const uint32_t fb = mapa_rank(smem_u32(&full_bar[stage]), 0u);
                    if (leader) mbar_expect_tx(&full_bar[stage], 2 * cfg::STAGE_BYTES);
                    if constexpr (!A_MN) tma_load_2d_pair(mA, fb, sa, kb * BK, tc.m_blk * BM);
                    else {
#pragma unroll
                        for (int i = 0; i < BM / 64; ++i) tma_load_2d_pair(mA, fb, sa + i * 8192, tc.m_blk * BM + 64 * i, kb * BK);
                    }
                    const int n0 = tc.n_blk * BN + crank * (BN / 2);
                    if constexpr (!B_MN) tma_load_2d_pair(mB, fb, sa + cfg::A_BYTES, kb * BK, n0);
                    else {
#pragma unroll
                        for (int i = 0; i < BN / 128; ++i) tma_load_2d_pair(mB, fb, sa + cfg::A_BYTES + i * 8192, n0 + 64 * i, kb * BK);
                    }
                }
                __syncwarp();
                if (++stage == cfg::STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (leader) {
            // ===================== MMA issuer (leader only): one instruction stream drives both SMs =====================
            constexpr uint32_t idesc = make_idesc_bf16(2 * BM, BN, A_MN, B_MN);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int t = w_first; t < num_tiles; t += w_step) {
                mbar_wait_cl(&tmem_empty[acc], acc_phase ^ 1);       // both epilogues have drained this accumulator
                tcgen05_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < nk; ++kb) {
                    mbar_wait_cl(&full_bar[stage], phase);
                    tcgen05_fence_after();
                    if (elect_one()) {
                        const uint32_t sa = smem_u32(smem + stage * cfg::STAGE_BYTES);
                        const uint64_t adesc = A_MN ? make_mnmajor_sw128_desc(sa, 8192) : make_kmajor_sw128_desc(sa);
                        const uint64_t bdesc = B_MN ? make_mnmajor_sw128_desc(sa + cfg::A_BYTES, 8192) : make_kmajor_sw128_desc(sa + cfg::A_BYTES);
                        constexpr uint64_t a_step = A_MN ? (2048 >> 4) : (32 >> 4), b_step = B_MN ? (2048 >> 4) : (32 >> 4);
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k)
                            umma2_bf16(d_tmem, adesc + a_step * k, bdesc + b_step * k, idesc, (kb | k) != 0);
                        umma2_commit_mc(&empty_bar[stage]);                  // both CTAs may refill this stage
                        if (kb == nk - 1) umma2_commit_mc(&tmem_full[acc]);  // both epilogues may drain
                    }
                    __syncwarp();
                    if (++stage == cfg::STAGES) { stage = 0; phase ^= 1; }
                }
                if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue: my 128 rows of the 256-row tile =====================
        const int q = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        const uintptr_t cbits = reinterpret_cast<uintptr_t>(C) | (nprob > 1 ? reinterpret_cast<uintptr_t>(C2) : 0);
        const bool vec_ok = ((ldc % 4) == 0) && ((cbits & 15) == 0);
        const bool vec8_ok = ((ldc % 8) == 0) && ((cbits & 31) == 0);
        for (int t = w_first; t < num_tiles; t += w_step) {
            const TileCoord tc = coord_of(t);
            mbar_wait_cl(&tmem_full[acc], acc_phase);
            tcgen05_fence_after();
            const int row = tc.m_blk * BM + q * 32 + lane;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                const int col0 = tc.n_blk * BN + c0;
                if (col0 >= N) break;                                 // warp-uniform
                uint32_t r[32];
                tmem_ld_32x32(taddr + (uint32_t)c0, r);
                store_acc_row32<OutT>((t >= per_prob) ? C2 : C, ldc, row, col0, M, N, r, bias, beta, vec_ok, vec8_ok);
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(mapa_rank(smem_u32(&tmem_empty[acc]), 0u));      // the leader's barrier (also for the leader itself)
            if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                 // the pair's commits / remote arrivals target each other's shared memory
    if (warp == 2) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(cfg::TMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------- host side
static PFN_cuTensorMapEncodeTiled get_encode() {
    static PFN_cuTensorMapEncodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) return nullptr;
        fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
    }
    return fn;
}

int make_bf16_map(CUtensorMap* map, const void* base, long long rows, int cols, int ld, int box_rows) {
    PFN_cuTensorMapEncodeTiled enc = get_encode();
    if (!enc) { set_error("gemm_bf16: cuTensorMapEncodeTiled entry point not available"); return NSD_ERR_CUDA; }
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%d ld=%d", (int)r, rows, cols, ld); return NSD_ERR_CUDA; }
    return NSD_OK;
}

// 3-D view [cols/64 chunks][rows][64] of the same row-major matrix: ONE box {64, box_rows, box_chunks} lands as box_chunks
// consecutive K-major 128B-swizzled [box_rows x 64] tiles, i.e. a whole multi-chunk UMMA operand per TMA instruction.
int make_bf16_map_chunked(CUtensorMap* map, const void* base, long long rows, int cols, int ld, int box_rows, int box_chunks) {
    PFN_cuTensorMapEncodeTiled enc = get_encode();
    if (!enc) { set_error("gemm_bf16: cuTensorMapEncodeTiled entry point not available"); return NSD_ERR_CUDA; }
    cuuint64_t gdim[3] = {(cuuint64_t)BK, (cuuint64_t)rows, (cuuint64_t)(cols / BK)};
    cuuint64_t gstride[2] = {(cuuint64_t)ld * 2, (cuuint64_t)BK * 2};
    cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, (cuuint32_t)box_chunks};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (chunked) failed (%d) rows=%lld cols=%d ld=%d", (int)r, rows, cols, ld); return NSD_ERR_CUDA; }
    return NSD_OK;
}

int make_bf16_map_mn(CUtensorMap* map, const void* base, long long k_rows, int mn_cols, int ld) {
    return make_bf16_map(map, base, k_rows, mn_cols, ld, BK);      // inner dim = mn (64-wide box), outer = k (64 rows)
}

template <int BN, typename OutT, bool A_MN, bool B_MN>
static int launch(const CUtensorMap& ta, const CUtensorMap& tb, void* C, int ldc, const float* bias, float beta, int M, int N, int K, cudaStream_t s) {
    using cfg = Cfg<BN>;
    auto kern = gemm_tc_kernel<BN, OutT, A_MN, B_MN>;
    static bool attr_set = false;       // per instantiation
    if (!attr_set) {
        NSD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, cfg::SMEM));
        attr_set = true;
    }
    const int tiles = cdiv(M, BM) * cdiv(N, BN);
    const int grid = std::min(tiles, gemm_sms());
    nsd::launch_k(kern, grid, THREADS, cfg::SMEM, s, ta, tb, reinterpret_cast<OutT*>(C), ldc, bias, beta, M, N, K);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

template <typename OutT, bool A_MN, bool B_MN, int BN2>
static int launch2(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& ta2, const CUtensorMap& tb2, void* C, void* C2, int ldc,
                   const float* bias, float beta, int M, int N, int K, int nprob, cudaStream_t s) {
    using cfg = Cfg2<BN2>;
    auto kern = gemm_tc2_kernel<OutT, A_MN, B_MN, BN2>;
    static bool attr_set = false;       // per instantiation
    if (!attr_set) {
        NSD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, cfg::SMEM));
        attr_set = true;
    }
    const int items = cdiv(cdiv(M, BM), 2) * cdiv(N, cfg::BN) * nprob;     // 256 x BN tiles
    const int grid = std::min(items, gemm_sms() / 2) * 2;
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(THREADS); lc.dynamicSmemBytes = cfg::SMEM; lc.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr; lc.numAttrs = 2;
    NSD_CUDA(cudaLaunchKernelEx(&lc, kern, ta, tb, ta2, tb2, reinterpret_cast<OutT*>(C), reinterpret_cast<OutT*>(C2), ldc, bias, beta, M, N, K, nprob));
    count_launch(1);
    return NSD_OK;
}

// tile width of the pair form: the one whose last round of clusters wastes less
static int pair_tile_width(int M, int N, int nprob) {
    const int clusters = std::max(1, gemm_sms() / 2);
    const long long mp = cdiv(cdiv(M, BM), 2);
    const long long c256 = cdivz((size_t)(mp * cdiv(N, 256) * nprob), (size_t)clusters) * 256;
    const long long c128 = cdivz((size_t)(mp * cdiv(N, 128) * nprob), (size_t)clusters) * 128;
    return (c128 < c256) ? 128 : 256;
}

}  // namespace tc
}  // namespace nsd

template <typename OutT, int BN2>
static int dispatch_layout2(bool a_mn, bool b_mn, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& ta2, const CUtensorMap& tb2,
                            void* C, void* C2, int ldc, const float* bias, float beta, int M, int N, int K, int nprob, cudaStream_t s) {
    using namespace nsd::tc;
    if (!a_mn && !b_mn) return launch2<OutT, false, false, BN2>(ta, tb, ta2, tb2, C, C2, ldc, bias, beta, M, N, K, nprob, s);
    if (!a_mn && b_mn) return launch2<OutT, false, true, BN2>(ta, tb, ta2, tb2, C, C2, ldc, bias, beta, M, N, K, nprob, s);
    if (a_mn && b_mn) return launch2<OutT, true, true, BN2>(ta, tb, ta2, tb2, C, C2, ldc, bias, beta, M, N, K, nprob, s);
    return launch2<OutT, true, false, BN2>(ta, tb, ta2, tb2, C, C2, ldc, bias, beta, M, N, K, nprob, s);
}
static int dispatch_pair(int bn2, bool f32, bool a_mn, bool b_mn, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& ta2, const CUtensorMap& tb2,
                         void* C, void* C2, int ldc, const float* bias, float beta, int M, int N, int K, int nprob, cudaStream_t s) {
    if (bn2 == 256) return f32 ? dispatch_layout2<float, 256>(a_mn, b_mn, ta, tb, ta2, tb2, C, C2, ldc, bias, beta, M, N, K, nprob, s)
                               : dispatch_layout2<__nv_bfloat16, 256>(a_mn, b_mn, ta, tb, ta2, tb2, C, C2, ldc, bias, beta, M, N, K, nprob, s);
    return f32 ? dispatch_layout2<float, 128>(a_mn, b_mn, ta, tb, ta2, tb2, C, C2, ldc, bias, beta, M, N, K, nprob, s)
               : dispatch_layout2<__nv_bfloat16, 128>(a_mn, b_mn, ta, tb, ta2, tb2, C, C2, ldc, bias, beta, M, N, K, nprob, s);
}

template <int BN, typename OutT>
static int dispatch_layout(bool a_mn, bool b_mn, const CUtensorMap& ta, const CUtensorMap& tb, void* C, int ldc, const float* bias, float beta,
                           int M, int N, int K, cudaStream_t s) {
    using namespace nsd::tc;
    if (!a_mn && !b_mn) return launch<BN, OutT, false, false>(ta, tb, C, ldc, bias, beta, M, N, K, s);
    if (!a_mn && b_mn) return launch<BN, OutT, false, true>(ta, tb, C, ldc, bias, beta, M, N, K, s);
    if (a_mn && b_mn) return launch<BN, OutT, true, true>(ta, tb, C, ldc, bias, beta, M, N, K, s);
    return launch<BN, OutT, true, false>(ta, tb, C, ldc, bias, beta, M, N, K, s);
}

extern "C" int nsd_set_gemm_sm_reserve(int n_sms) {
    using namespace nsd;
    NSD_CHECK_ARG(n_sms >= 0 && n_sms < sm_count(), "set_gemm_sm_reserve: %d not in [0, %d)", n_sms, sm_count());
    nsd::tc::g_sm_reserve = n_sms;
    return NSD_OK;
}

extern "C" int nsd_gemm_bf16(int transa, int transb, int M, int N, int K, const void* A, int lda, const void* B, int ldb,
                             void* C, int ldc, int c_dtype, const float* bias, float beta, void* stream) {
    using namespace nsd;
    using namespace nsd::tc;
    NSD_CHECK_ARG(M >= 0 && N >= 0 && K > 0, "gemm_bf16: bad sizes M=%d N=%d K=%d", M, N, K);
    if (M == 0 || N == 0) return NSD_OK;
    NSD_CHECK_ARG(A && B && C, "gemm_bf16: null pointer");
    // op(A) [M,K]: stored [M,K] (K-major) if !transa, [K,M] (M-major) if transa.  op(B) [K,N]: stored [N,K] (K-major) if
    // transb, [K,N] (N-major) if !transb.  Both majors are native UMMA operand layouts: no transposed copies needed.
    const bool a_mn = transa != 0, b_mn = transb == 0;
    NSD_CHECK_ARG((lda % 8) == 0 && (ldb % 8) == 0, "gemm_bf16: lda=%d / ldb=%d must be multiples of 8", lda, ldb);
    NSD_CHECK_ARG(lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K), "gemm_bf16: leading dimension smaller than the row length");
    NSD_CHECK_ARG(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0, "gemm_bf16: A and B must be 16-byte aligned");
    NSD_CHECK_ARG(c_dtype == NSD_F32 || c_dtype == NSD_BF16, "gemm_bf16: bad output dtype");
    NSD_CHECK_ARG(bias == nullptr || ((uintptr_t)bias & 15) == 0, "gemm_bf16: bias must be 16-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    const int BN = (N >= 192) ? 256 : (N >= 96 ? 128 : 64);
    CUtensorMap ta, tb;
    int rc = a_mn ? make_bf16_map_mn(&ta, A, K, M, lda) : make_bf16_map(&ta, A, M, K, lda, BM);
    if (rc) return rc;
    // wide tiles with at least one vertical pair: the cta_group::2 form (256 x 256 tile over an SM pair)
    const bool pair = (BN == 256) && (M > BM) && sm_count() >= 2;
    const int bn2 = pair ? pair_tile_width(M, N, 1) : 0;
    rc = b_mn ? make_bf16_map_mn(&tb, B, K, N, ldb) : make_bf16_map(&tb, B, N, K, ldb, pair ? bn2 / 2 : BN);
    if (rc) return rc;
    const bool f32 = c_dtype == NSD_F32;
    if (pair) return dispatch_pair(bn2, f32, a_mn, b_mn, ta, tb, ta, tb, C, C, ldc, bias, beta, M, N, K, 1, s);
    if (BN == 256) return f32 ? dispatch_layout<256, float>(a_mn, b_mn, ta, tb, C, ldc, bias, beta, M, N, K, s) : dispatch_layout<256, __nv_bfloat16>(a_mn, b_mn, ta, tb, C, ldc, bias, beta, M, N, K, s);
    if (BN == 128) return f32 ? dispatch_layout<128, float>(a_mn, b_mn, ta, tb, C, ldc, bias, beta, M, N, K, s) : dispatch_layout<128, __nv_bfloat16>(a_mn, b_mn, ta, tb, C, ldc, bias, beta, M, N, K, s);
    return f32 ? dispatch_layout<64, float>(a_mn, b_mn, ta, tb, C, ldc, bias, beta, M, N, K, s) : dispatch_layout<64, __nv_bfloat16>(a_mn, b_mn, ta, tb, C, ldc, bias, beta, M, N, K, s);
}

extern "C" int nsd_gemm_bf16_x2(int transa, int transb, int M, int N, int K, const void* A0, const void* A1, int lda, const void* B0, const void* B1,
                                int ldb, void* C0, void* C1, int ldc, int c_dtype, void* stream) {
    using namespace nsd;
    using namespace nsd::tc;
    NSD_CHECK_ARG(M >= 0 && N >= 0 && K > 0, "gemm_bf16_x2: bad sizes M=%d N=%d K=%d", M, N, K);
    if (M == 0 || N == 0) return NSD_OK;
    NSD_CHECK_ARG(A0 && A1 && B0 && B1 && C0 && C1, "gemm_bf16_x2: null pointer");
    if (N < 192 || M <= BM || sm_count() < 2) {          // shapes the pair form does not take: two plain launches
        int rc = nsd_gemm_bf16(transa, transb, M, N, K, A0, lda, B0, ldb, C0, ldc, c_dtype, nullptr, 0.f, stream);
        return rc ? rc : nsd_gemm_bf16(transa, transb, M, N, K, A1, lda, B1, ldb, C1, ldc, c_dtype, nullptr, 0.f, stream);
    }
    const bool a_mn = transa != 0, b_mn = transb == 0;
    NSD_CHECK_ARG((lda % 8) == 0 && (ldb % 8) == 0, "gemm_bf16_x2: lda=%d / ldb=%d must be multiples of 8", lda, ldb);
    NSD_CHECK_ARG(lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K), "gemm_bf16_x2: leading dimension smaller than the row length");
    NSD_CHECK_ARG((((uintptr_t)A0 | (uintptr_t)A1 | (uintptr_t)B0 | (uintptr_t)B1) & 15) == 0, "gemm_bf16_x2: operands must be 16-byte aligned");
    NSD_CHECK_ARG(c_dtype == NSD_F32 || c_dtype == NSD_BF16, "gemm_bf16_x2: bad output dtype");
    const int bn2 = pair_tile_width(M, N, 2);
    CUtensorMap ta, tb, ta2, tb2;
    int rc = a_mn ? make_bf16_map_mn(&ta, A0, K, M, lda) : make_bf16_map(&ta, A0, M, K, lda, BM);
    if (!rc) rc = a_mn ? make_bf16_map_mn(&ta2, A1, K, M, lda) : make_bf16_map(&ta2, A1, M, K, lda, BM);
    if (!rc) rc = b_mn ? make_bf16_map_mn(&tb, B0, K, N, ldb) : make_bf16_map(&tb, B0, N, K, ldb, bn2 / 2);
    if (!rc) rc = b_mn ? make_bf16_map_mn(&tb2, B1, K, N, ldb) : make_bf16_map(&tb2, B1, N, K, ldb, bn2 / 2);
    if (rc) return rc;
    return dispatch_pair(bn2, c_dtype == NSD_F32, a_mn, b_mn, ta, tb, ta2, tb2, C0, C1, ldc, nullptr, 0.f, M, N, K, 2, (cudaStream_t)stream);
}
