// Streaming inference push for small batches (BASELINE configs[3]; SURVEY.md 8f rank 3): ONE launch consumes one stride of
// new 20 ms bins and advances the whole unidirectional decoder by one output frame -- the Gaussian smoothing of the bins that
// just became computable (augmentations.py:91), their day affine and softsign (model.py:89-93), the slide of the k32/s4
// patch (model.py:96-101), every GRU layer's input and recurrent projection, gate math and state update (nn.GRU,
// model.py:50-57, 104-119, with the state CARRIED between calls, which the reference's forward cannot do), the phoneme-logit
// projection (model.py:122) and the greedy argmax (trainer:314).
//
// At batch 1..8 a push is pure weight bandwidth: 107 MB of bf16 weights (W_ih 50 MB for layer 0, 6.3 MB for each of the
// other nine matrices) against 2 x 107 M multiply-adds per batch row.  A persistent cooperative grid (one 16-warp CTA per
// SM) streams every weight element exactly once per push with 16-byte loads; the set fits the 126 MB L2, so consecutive
// pushes find it on chip.  Phases, separated by grid barriers:
//   0  front end for the new stride (a few CTAs) and, on every warp, the recurrent projections W_hh h_{t-1} of layers 1..L-1
//      (the carried states are known up front: 25 MB of weights with no dependence on this push's input);
//   1..L  layer l: one warp per hidden unit streams the unit's three gate rows of W_ih (and W_hh for layer 0) against the
//      layer input staged in shared memory and does that unit's gate math -- no partial sums leave the warp;
//   last  logits + argmax by block 0.
// The per-slot form (SLOTS = true, nsd_stream_push_slots) runs the same body with a bin counter, an active flag and a last
// frame per batch row: inactive rows are left as they are, a row still warming up (fewer than K + right bins) only moves its
// ring and patch row, and the stack writes back only the rows that emit a frame.  No row's arithmetic depends on the others
// or on BM, so a session gives the same bits in any slot of any batch size.
// A warp always has the next 512 columns' weights (2 x 3 x 16 bytes per lane) in flight while it reduces the current ones, and
// everything else a unit's gate math reads (biases, recurrent projection, previous state) is requested before the stream
// starts.  bf16 weights, bf16-rounded inputs / recurrent state, fp32 accumulation and fp32 carried state: the arithmetic of
// the time-batched tcgen05 path up to summation order.
#include <cooperative_groups.h>

#include <algorithm>
#include <stdlib.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace nsd {

constexpr int SP_MAX_LAYERS = 8;
constexpr int SP_THREADS = 512;
constexpr int SP_WARPS = SP_THREADS / 32;
constexpr int SP_KC = 512;                                // columns per weight-stream step of a warp (2 x 16 bytes per lane and row)
constexpr int SP_MAX_S = 8;
constexpr int SP_MAX_TAPS = 32;

struct StreamPushParams {
    // front end
    const float* bins_in; float* rawring; int ring_rows;          // [B][S][N] new bins; [B][ring_rows][N] raw bins by absolute index mod ring_rows
    const int64_t* day_idx; const float* day_w; const float* day_b; const float* taps; int ntaps, n_days;
    __nv_bfloat16* x0buf;                                         // [2][B][N*K]: patch row of frame j lives in half (j & 1)
    int* n_bins;                                                  // bins received before this push (device counter, += S at the end); [B] per slot
    const int* active; const int* last_frame; int* emitted;       // per-slot form only: [B] each
    int extra, N, K, S;
    // stack
    const __nv_bfloat16* w_ih[SP_MAX_LAYERS]; const __nv_bfloat16* w_hh[SP_MAX_LAYERS];   // [3H, in_l], [3H, H], gate rows r | z | n
    const float* b_ih[SP_MAX_LAYERS]; const float* b_hh[SP_MAX_LAYERS];                   // [3H]
    float* h; __nv_bfloat16* hbf;                                 // [L][B][H] carried state (fp32 master, bf16 operand copy)
    float* gh;                                                    // [L][3][H][B] recurrent projections of layers >= 1 (workspace)
    unsigned long long* trace;                                    // optional: globaltimer stamps of block 0 at the phase boundaries
    const __nv_bfloat16* fc_w; const float* fc_b;                 // [C, H], [C]
    float* logits; int* ids; int* err_flag;                       // [B, C], [B]
    int B, F0, H, L, C;
};

__device__ __forceinline__ float sp_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float sp_sigmoid(float x) { return fmaf(0.5f, sp_tanh(0.5f * x), 0.5f); }
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

__device__ __forceinline__ void bf16x8_to_f32(const uint4& u, float (&f)[8]) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 v = __bfloat1622float2(h[i]);
        f[2 * i] = v.x; f[2 * i + 1] = v.y;
    }
}
__device__ __forceinline__ float dot8(const uint4& w, const float (&x)[8], float acc) {
    float wf[8];
    bf16x8_to_f32(w, wf);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc = fmaf(wf[i], x[i], acc);
    return acc;
}
// weights: read once per push, keep them out of L1 (ld.global.nc.L1::no_allocate), 16 bytes per lane
__device__ __forceinline__ uint4 ldw(const __nv_bfloat16* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
// activations written earlier in this launch by other SMs: L2 is the point of coherence (ld.global.cg)
__device__ __forceinline__ uint4 ldx(const __nv_bfloat16* p) { return __ldcg(reinterpret_cast<const uint4*>(p)); }

__device__ __forceinline__ float gru_cell(float gir, float giz, float gin, float ghr, float ghz, float ghn, float hprev) {
    const float r = sp_sigmoid(gir + ghr);
    const float z = sp_sigmoid(giz + ghz);
    const float n = sp_tanh(fmaf(r, ghn, gin));
    return fmaf(z, hprev - n, n);                                  // (1-z)*n + z*h_prev
}

// acc[g][b] += sum_k W[(g*H + u), k] * x[b][k] over k in [0, Kdim): the warp streams the three gate rows of hidden unit u
// (16 bytes per lane per row per 256 columns, the next 256 columns' weights already in flight while the current ones are
// reduced); x is bf16 in shared memory, row stride ldx.  Not yet summed over the lanes.
template <int BM>
__device__ __forceinline__ void unit_dot(const __nv_bfloat16* __restrict__ W, int Kdim, int H, int u, const __nv_bfloat16* xs, int ldx_, int lane,
                                         float (&acc)[3][BM]) {
    const __nv_bfloat16* w0 = W + (size_t)u * Kdim + lane * 8;
    const size_t gs = (size_t)H * Kdim;
    constexpr bool DB = BM <= 2;                                   // double-buffered weight registers where the register file allows
    uint4 cur[2][3], nxt[DB ? 2 : 1][DB ? 3 : 1];
    if (DB) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int g = 0; g < 3; ++g) cur[j][g] = ldw(w0 + g * gs + j * 256);
    }
    for (int k0 = 0; k0 < Kdim; k0 += 512) {
        if constexpr (DB) {
            if (k0 + 512 < Kdim) {
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int g = 0; g < 3; ++g) nxt[j][g] = ldw(w0 + g * gs + k0 + 512 + j * 256);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int g = 0; g < 3; ++g) cur[j][g] = ldw(w0 + g * gs + k0 + j * 256);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
#pragma unroll
            for (int b = 0; b < BM; ++b) {
                float xv[8];
                bf16x8_to_f32(*reinterpret_cast<const uint4*>(xs + (size_t)b * ldx_ + k0 + j * 256 + lane * 8), xv);
#pragma unroll
                for (int g = 0; g < 3; ++g) acc[g][b] = dot8(cur[j][g], xv, acc[g][b]);
            }
        }
        if constexpr (DB) {
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int g = 0; g < 3; ++g) cur[j][g] = nxt[j][g];
        }
    }
}

// global bf16 [rows][cols] (rows >= BM and rows outside rowmask zero-filled; row b read from src + alt if bit b of altmask
// is set) -> shared memory, 16 bytes per thread; L2 is the point of coherence for activations written earlier in this
// launch by other SMs
template <int BM>
__device__ __forceinline__ void stage_x(__nv_bfloat16* dst, const __nv_bfloat16* src, int rows, int cols, int tid, unsigned rowmask = ~0u,
                                        size_t alt = 0, unsigned altmask = 0u) {
    const int per = cols / 8;
    for (int i = tid; i < BM * per; i += SP_THREADS) {
        const int b = i / per, c = i - b * per;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (b < rows && ((rowmask >> b) & 1u)) v = ldx(src + (size_t)b * cols + ((altmask >> b) & 1u) * alt + c * 8);
        reinterpret_cast<uint4*>(dst)[i] = v;
    }
}

__device__ __forceinline__ int floor_div(int a, int b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

__device__ __forceinline__ unsigned long long sp_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// The body of both kernels below (inlined into each; p lives in the kernel's parameter space)
template <int BM, bool SLOTS>
__device__ __forceinline__ void stream_push_body(const StreamPushParams& p) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) float smem[];
    const int H = p.H, B = p.B, N = p.N, K = p.K, S = p.S, L = p.L;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // warp slots interleave the SMs: consecutive slots sit on different SMs, so any prefix of the slots is spread over the chip
    const int slot = warp * gridDim.x + blockIdx.x, nslot = gridDim.x * SP_WARPS;
    const int ntaps = p.ntaps, left = (ntaps - 1) / 2, right = ntaps - 1 - left;
    // the frame a row's push completes: jn = (n0 + S - extra - K - right) / S (exact: n0 + S - extra - K - right is a multiple of S);
    // negative while the row warms up.  Rows in emitmask write back their state and logits; bit b of halfmask = jn & 1 of row b.
    unsigned actmask = ~0u, emitmask = ~0u, halfmask = 0u;
    if constexpr (SLOTS) {
        actmask = emitmask = 0u;
        for (int b = 0; b < B; ++b) {
            if (!p.active[b]) continue;
            const int j = floor_div(*reinterpret_cast<volatile int*>(p.n_bins + b) + S - p.extra - K - right, S);
            actmask |= 1u << b;
            halfmask |= (unsigned)(j & 1) << b;
            if (j >= 0 && j <= p.last_frame[b]) emitmask |= 1u << b;
        }
    } else {
        const int j = (*reinterpret_cast<volatile int*>(p.n_bins) + S - p.extra - K - right) / S;
        halfmask = (j & 1) ? ~0u : 0u;
    }
    const bool trace = p.trace != nullptr && blockIdx.x == 0 && tid == 0;
    if (trace) p.trace[0] = sp_globaltimer();

    // ---------------------------------------------------------------- phase 0a: front end, CTA = (batch row, 32 output channels)
    const int ncg = N / 32;
    if ((int)blockIdx.x < B * ncg && ((actmask >> (blockIdx.x / ncg)) & 1u)) {
        const int b = blockIdx.x / ncg, c0 = (blockIdx.x % ncg) * 32;
        const int n0 = *reinterpret_cast<volatile int*>(p.n_bins + (SLOTS ? b : 0));   // bins this row received before this push
        const int jn = floor_div(n0 + S - p.extra - K - right, S);
        __nv_bfloat16* x0_new = p.x0buf + (size_t)(jn & 1) * B * p.F0;
        const __nv_bfloat16* x0_old = p.x0buf + (size_t)((jn & 1) ^ 1) * B * p.F0;
        float* ys_s = smem;                                        // [S][N] smoothed new bins, bf16-rounded (the affine's A operand)
        float* part_s = ys_s + S * N;                              // [SP_WARPS][S][32]
        float* znew_s = part_s + SP_WARPS * S * 32;                // [S][32]
        long long day = p.day_idx[b];
        if (day < 0 || day >= p.n_days) {                          // reference: index_select raises IndexError (model.py:89)
            if (tid == 0 && p.err_flag) *p.err_flag = 1;
            day = 0;
        }
        const int s0 = n0 - p.extra - right;                       // first smoothed bin that became computable
        const float* ring = p.rawring + (size_t)b * p.ring_rows * N;
        const float* fresh = p.bins_in + (size_t)b * S * N;
        for (int i = tid; i < S * N; i += SP_THREADS) {
            const int r = i / N, d = i - r * N;
            float v[SP_MAX_TAPS];
#pragma unroll
            for (int k = 0; k < SP_MAX_TAPS; ++k) {                // all taps' loads in flight together
                const int a = s0 + r - left + k;
                v[k] = 0.f;
                if (k < ntaps) {
                    if (a >= n0) v[k] = __ldg(fresh + (size_t)(a - n0) * N + d);
                    else if (a >= 0) v[k] = ring[(size_t)(a % p.ring_rows) * N + d];
                }
            }
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < SP_MAX_TAPS; ++k)                  // same order as K1's FIR (frontend.cu): bit-identical ys
                if (k < ntaps) acc = fmaf(__ldg(p.taps + k), v[k], acc);
            ys_s[i] = bf16_round(acc);
        }
        __syncthreads();
        {   // warp = a slice of the input channels, lane = output channel: z_pre[r][c] = sum_d ys[r][d] * W[d][c]
            const int dper = (N + SP_WARPS - 1) / SP_WARPS;
            const float* W = p.day_w + (size_t)day * N * N + c0 + lane;
            float acc[SP_MAX_S];
#pragma unroll
            for (int r = 0; r < SP_MAX_S; ++r) acc[r] = 0.f;
            const int d1 = min(N, (warp + 1) * dper);
#pragma unroll 16
            for (int d = warp * dper; d < d1; ++d) {
                const float w = bf16_round(__ldg(W + (size_t)d * N));
#pragma unroll
                for (int r = 0; r < SP_MAX_S; ++r)
                    if (r < S) acc[r] = fmaf(ys_s[r * N + d], w, acc[r]);
            }
#pragma unroll
            for (int r = 0; r < SP_MAX_S; ++r)
                if (r < S) part_s[(warp * S + r) * 32 + lane] = acc[r];
        }
        __syncthreads();
        if (tid < S * 32) {
            const int r = tid >> 5;
            float a = p.day_b[(size_t)day * N + c0 + lane];
            for (int w = 0; w < SP_WARPS; ++w) a += part_s[(w * S + r) * 32 + lane];
            znew_s[tid] = a / (1.0f + fabsf(a));                   // softsign (model.py:93)
        }
        __syncthreads();
        // slide the patch: x0[c*K + k] = z[S*j + k][c]  (model.py:96-101: channel-major, tap-minor); rows before the first bin
        // (an utterance's first pushes) are zeros, whatever the buffer held
        for (int e = tid; e < 32 * K; e += SP_THREADS) {
            const int cl = e / K, k = e - cl * K;
            const size_t o = (size_t)b * p.F0 + (size_t)(c0 + cl) * K;
            __nv_bfloat16 v = __float2bfloat16_rn(0.f);
            if (S * jn + k >= 0) v = (k < K - S) ? x0_old[o + k + S] : __float2bfloat16_rn(znew_s[(k - (K - S)) * 32 + cl]);
            x0_new[o + k] = v;
        }
        if (c0 == 0) {                                             // the new raw bins join the ring (slots 64 bins behind nobody reads)
            float* ringw = p.rawring + (size_t)b * p.ring_rows * N;
            for (int i = tid; i < S * N; i += SP_THREADS) ringw[(size_t)((n0 + i / N) % p.ring_rows) * N + (i % N)] = fresh[i];
        }
        __syncthreads();
    }
    // ---------------------------------------------------------------- phase 0b: recurrent projections W_hh h_{t-1} of layers 1 .. L-1
    // (the carried states are known up front); raw sums without bias -> gh[l][g][u][b]
    __nv_bfloat16* xs = reinterpret_cast<__nv_bfloat16*>(smem);
    const bool stack = !SLOTS || emitmask != 0u;                   // a push in which no row emits leaves the stack alone
    if (stack && L > 1) {
        stage_x<BM>(xs, p.hbf + (size_t)B * H, B, H, tid, emitmask);   // layer 1's state; further layers are staged as the loop reaches them
        for (int l = 2; l < L; ++l) stage_x<BM>(xs + (size_t)(l - 1) * BM * H, p.hbf + (size_t)l * B * H, B, H, tid, emitmask);
        __syncthreads();
        for (int t = slot; t < (L - 1) * H; t += nslot) {
            const int l = 1 + t / H, u = t - (l - 1) * H;
            float acc[3][BM];
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int b = 0; b < BM; ++b) acc[g][b] = 0.f;
            unit_dot<BM>(p.w_hh[l], H, H, u, xs + (size_t)(l - 1) * BM * H, H, lane, acc);
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int b = 0; b < BM; ++b) {
                    const float v = warp_sum(acc[g][b]);
                    if (lane == 0 && b < B) p.gh[(((size_t)l * 3 + g) * H + u) * B + b] = v;
                }
        }
    }
    if (trace) p.trace[1] = sp_globaltimer();
    grid.sync();
    if (trace) p.trace[2] = sp_globaltimer();
    // ---------------------------------------------------------------- layers 0 .. L-1: one warp per hidden unit
    for (int l = 0; stack && l < L; ++l) {
        const int in_l = l == 0 ? p.F0 : H;
        __nv_bfloat16* hs = xs + (size_t)BM * in_l;                // layer 0 also needs its own previous state (bf16) for W_hh
        if (l == 0) {                                              // each row's patch row from its own half of x0buf
            stage_x<BM>(xs, p.x0buf, B, in_l, tid, emitmask, (size_t)B * p.F0, halfmask);
            stage_x<BM>(hs, p.hbf, B, H, tid, emitmask);
        } else {
            stage_x<BM>(xs, p.hbf + (size_t)(l - 1) * B * H, B, in_l, tid, emitmask);
        }
        __syncthreads();
        float* hl = p.h + (size_t)l * B * H;
        __nv_bfloat16* hbl = p.hbf + (size_t)l * B * H;
        for (int u = slot; u < H; u += nslot) {
            // everything the gate math needs besides the dot products is requested first (small batches: it arrives under the
            // weight stream; larger ones are FMA-bound and short of registers, they fetch it afterwards)
            float bi[3], bh[3], ghv[3][BM], hprev[BM];
            auto fetch_gate_inputs = [&]() {
#pragma unroll
                for (int g = 0; g < 3; ++g) {
                    bi[g] = __ldg(p.b_ih[l] + g * H + u); bh[g] = __ldg(p.b_hh[l] + g * H + u);
                    if (l > 0) {
#pragma unroll
                        for (int b = 0; b < BM; ++b) ghv[g][b] = b < B ? __ldcg(p.gh + (((size_t)l * 3 + g) * H + u) * B + b) : 0.f;
                    }
                }
#pragma unroll
                for (int b = 0; b < BM; ++b) hprev[b] = b < B ? hl[(size_t)b * H + u] : 0.f;
            };
            if constexpr (BM <= 2) fetch_gate_inputs();
            float acc[3][BM];
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int b = 0; b < BM; ++b) acc[g][b] = 0.f;
            unit_dot<BM>(p.w_ih[l], in_l, H, u, xs, in_l, lane, acc);
            if (l == 0) {
                float ah[3][BM];
#pragma unroll
                for (int g = 0; g < 3; ++g)
#pragma unroll
                    for (int b = 0; b < BM; ++b) ah[g][b] = 0.f;
                unit_dot<BM>(p.w_hh[0], H, H, u, hs, H, lane, ah);
#pragma unroll
                for (int g = 0; g < 3; ++g)
#pragma unroll
                    for (int b = 0; b < BM; ++b) ghv[g][b] = warp_sum(ah[g][b]);
            }
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int b = 0; b < BM; ++b) acc[g][b] = warp_sum(acc[g][b]);
            if constexpr (BM > 2) fetch_gate_inputs();
            if (lane == 0) {
#pragma unroll
                for (int b = 0; b < BM; ++b)
                    if (b < B && ((emitmask >> b) & 1u)) {
                        const float hn = gru_cell(acc[0][b] + bi[0], acc[1][b] + bi[1], acc[2][b] + bi[2], ghv[0][b] + bh[0], ghv[1][b] + bh[1],
                                                  ghv[2][b] + bh[2], hprev[b]);
                        hl[(size_t)b * H + u] = hn;
                        hbl[(size_t)b * H + u] = __float2bfloat16_rn(hn);
                    }
            }
        }
        if (trace) p.trace[3 + 2 * l] = sp_globaltimer();
        grid.sync();
        if (trace) p.trace[4 + 2 * l] = sp_globaltimer();
    }
    // ---------------------------------------------------------------- logits + greedy id (block 0)
    if (blockIdx.x == 0 && stack) {
        stage_x<BM>(xs, p.hbf + (size_t)(L - 1) * B * H, B, H, tid, emitmask);
        float* lg = reinterpret_cast<float*>(xs + (size_t)BM * H); // [B][C]
        __syncthreads();
        for (int c = warp; c < p.C; c += SP_WARPS) {
            float acc[BM];
#pragma unroll
            for (int b = 0; b < BM; ++b) acc[b] = 0.f;
#pragma unroll 4
            for (int k0 = lane * 8; k0 < H; k0 += 256) {
                const uint4 w = ldw(p.fc_w + (size_t)c * H + k0);
#pragma unroll
                for (int b = 0; b < BM; ++b) {
                    float xv[8];
                    bf16x8_to_f32(*reinterpret_cast<const uint4*>(xs + (size_t)b * H + k0), xv);
                    acc[b] = dot8(w, xv, acc[b]);
                }
            }
            const float fb = __ldg(p.fc_b + c);
#pragma unroll
            for (int b = 0; b < BM; ++b) {
                const float v = warp_sum(acc[b]) + fb;
                if (lane == 0 && b < B && ((emitmask >> b) & 1u)) { lg[b * p.C + c] = v; p.logits[(size_t)b * p.C + c] = v; }
            }
        }
        __syncthreads();
    }
    if (blockIdx.x == 0) {
        if (p.ids != nullptr && tid < B) {                         // argmax, ties -> lowest index (trainer:314: torch.argmax); -1: no frame
            int best = -1;
            if (stack && ((emitmask >> tid) & 1u)) {
                const float* row = reinterpret_cast<const float*>(xs + (size_t)BM * H) + tid * p.C;
                best = 0;
                for (int c = 1; c < p.C; ++c)
                    if (row[c] > row[best]) best = c;
            }
            p.ids[tid] = best;
        }
        if (tid < (SLOTS ? B : 1) && ((actmask >> tid) & 1u)) p.n_bins[tid] += S;
        if constexpr (SLOTS) {
            if (tid < B) p.emitted[tid] = (emitmask >> tid) & 1u;
        }
        if (trace) p.trace[3 + 2 * L] = sp_globaltimer();
    }
}

template <int BM>
__global__ void __launch_bounds__(SP_THREADS, 1) stream_push_kernel(const __grid_constant__ StreamPushParams p) { stream_push_body<BM, false>(p); }
template <int BM>
__global__ void __launch_bounds__(SP_THREADS, 1) stream_push_slots_kernel(const __grid_constant__ StreamPushParams p) { stream_push_body<BM, true>(p); }

// Shared host side of both entry points: argument checks, parameter block, batch-form dispatch, cooperative launch.
template <bool SLOTS>
int stream_push_launch(const float* bins_in, float* rawring, int ring_rows, const int64_t* day_idx, const float* day_w, const float* day_b,
                       int n_days, const float* taps, int ntaps, void* x0buf_bf16, int* n_bins, const int* active, const int* last_frame,
                       int* emitted, int extra, int B, int N, int K, int S, int H, int L, int C, const void* const* w_ih_bf16,
                       const void* const* w_hh_bf16, const void* const* b_ih, const void* const* b_hh, float* h, void* h_bf16,
                       const void* fc_w_bf16, const float* fc_b, float* logits, int* ids, int* err_flag, void* workspace,
                       size_t workspace_bytes, void* stream) {
    NSD_CHECK_ARG(B >= 1 && B <= 8, "stream_push: batch %d not in [1, 8] (larger batches take the time-batched path)", B);
    NSD_CHECK_ARG(L >= 1 && L <= SP_MAX_LAYERS && H > 0 && H % SP_KC == 0 && C > 0, "stream_push: bad sizes L=%d H=%d C=%d (H must be a multiple of %d)", L,
                  H, C, SP_KC);
    NSD_CHECK_ARG(N > 0 && N % 32 == 0 && S >= 1 && S <= SP_MAX_S && K > S && ((size_t)N * K) % SP_KC == 0 && ntaps >= 1 && ntaps <= SP_MAX_TAPS,
                  "stream_push: bad front-end sizes N=%d K=%d S=%d ntaps=%d (N %% 32 == 0, N*K %% %d == 0, S <= %d)", N, K, S, ntaps, SP_KC, SP_MAX_S);
    NSD_CHECK_ARG(extra >= 0 && extra < S && ring_rows >= ntaps - 1 + 2 * S, "stream_push: extra=%d must be in [0, S) and the raw ring (%d rows) must cover the smoothing window",
                  extra, ring_rows);
    NSD_CHECK_ARG(bins_in && rawring && day_idx && day_w && day_b && taps && x0buf_bf16 && n_bins && w_ih_bf16 && w_hh_bf16 && b_ih && b_hh && h && h_bf16 &&
                      fc_w_bf16 && fc_b && logits && workspace, "stream_push: null pointer");
    const int F0 = N * K;
    if (workspace_bytes < nsd_stream_push_workspace(B, F0, H, L)) { set_error("stream_push: workspace too small"); return NSD_ERR_WORKSPACE; }
    StreamPushParams p;
    p.bins_in = bins_in; p.rawring = rawring; p.ring_rows = ring_rows; p.day_idx = day_idx; p.day_w = day_w; p.day_b = day_b; p.taps = taps;
    p.ntaps = ntaps; p.n_days = n_days; p.x0buf = reinterpret_cast<__nv_bfloat16*>(x0buf_bf16); p.n_bins = n_bins; p.extra = extra;
    p.active = active; p.last_frame = last_frame; p.emitted = emitted;
    p.N = N; p.K = K; p.S = S;
    for (int l = 0; l < L; ++l) {
        NSD_CHECK_ARG(w_ih_bf16[l] && w_hh_bf16[l] && b_ih[l] && b_hh[l], "stream_push: null weight pointer for layer %d", l);
        p.w_ih[l] = reinterpret_cast<const __nv_bfloat16*>(w_ih_bf16[l]); p.w_hh[l] = reinterpret_cast<const __nv_bfloat16*>(w_hh_bf16[l]);
        p.b_ih[l] = reinterpret_cast<const float*>(b_ih[l]); p.b_hh[l] = reinterpret_cast<const float*>(b_hh[l]);
    }
    p.h = h; p.hbf = reinterpret_cast<__nv_bfloat16*>(h_bf16);
    p.gh = reinterpret_cast<float*>(workspace);
    {   // NSD_STREAM_TRACE=1: block 0 stamps the phase boundaries into the tail of the workspace (read by scratch/stream_trace.py)
        static const bool tr = getenv("NSD_STREAM_TRACE") != nullptr && atoi(getenv("NSD_STREAM_TRACE")) != 0;
        const size_t off = (sizeof(float) * (size_t)L * 3 * H * B + 255) / 256 * 256;
        p.trace = tr ? reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(workspace) + off) : nullptr;
    }
    p.fc_w = reinterpret_cast<const __nv_bfloat16*>(fc_w_bf16); p.fc_b = fc_b; p.logits = logits; p.ids = ids; p.err_flag = err_flag;
    p.B = B; p.F0 = F0; p.H = H; p.L = L; p.C = C;
    auto go = [&](auto kern, int BM) -> int {
        // front end scratch | staged layer input (layer 0: patch row + own state; phase 0b: L-1 states) | logits
        const size_t smem = std::max<size_t>(sizeof(float) * ((size_t)S * N + (size_t)SP_WARPS * S * 32 + (size_t)S * 32),
                                        std::max<size_t>(2 * (size_t)BM * ((size_t)F0 + H), 2 * (size_t)BM * H * std::max(1, L - 1)) +
                                            sizeof(float) * (size_t)B * C);
        if (smem > 48 * 1024) NSD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        NSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SP_THREADS, smem));
        if (per_sm < 1) { set_error("stream_push: kernel does not fit an SM"); return NSD_ERR_INVALID; }
        const int grid = sm_count();                                       // one CTA per SM, all co-resident (grid barriers between phases)
        if (grid < B * (N / 32)) { set_error("stream_push: %d front-end CTAs needed, %d SMs", B * (N / 32), grid); return NSD_ERR_INVALID; }
        void* args[] = {(void*)&p};
        NSD_CUDA(cudaLaunchCooperativeKernel((const void*)kern, dim3(grid), dim3(SP_THREADS), args, smem, (cudaStream_t)stream));
        count_launch(1);
        return NSD_OK;
    };
    if (B == 1) return go(SLOTS ? stream_push_slots_kernel<1> : stream_push_kernel<1>, 1);
    if (B == 2) return go(SLOTS ? stream_push_slots_kernel<2> : stream_push_kernel<2>, 2);
    if (B <= 4) return go(SLOTS ? stream_push_slots_kernel<4> : stream_push_kernel<4>, 4);
    return go(SLOTS ? stream_push_slots_kernel<8> : stream_push_kernel<8>, 8);
}

}  // namespace nsd

extern "C" {

size_t nsd_stream_push_workspace(int B, int F0, int H, int L) {
    if (B < 1 || F0 < 1 || H < 1 || L < 1) return 0;
    (void)F0;
    return sizeof(float) * (size_t)L * 3 * H * B + 32 * sizeof(unsigned long long) + 256;
}

int nsd_stream_push(const float* bins_in, float* rawring, int ring_rows, const int64_t* day_idx, const float* day_w, const float* day_b,
                    int n_days, const float* taps, int ntaps, void* x0buf_bf16, int* n_bins, int extra, int B, int N, int K, int S, int H,
                    int L, int C, const void* const* w_ih_bf16, const void* const* w_hh_bf16, const void* const* b_ih,
                    const void* const* b_hh, float* h, void* h_bf16, const void* fc_w_bf16, const float* fc_b, float* logits, int* ids,
                    int* err_flag, void* workspace, size_t workspace_bytes, void* stream) {
    return nsd::stream_push_launch<false>(bins_in, rawring, ring_rows, day_idx, day_w, day_b, n_days, taps, ntaps, x0buf_bf16, n_bins, nullptr,
                                          nullptr, nullptr, extra, B, N, K, S, H, L, C, w_ih_bf16, w_hh_bf16, b_ih, b_hh, h, h_bf16, fc_w_bf16,
                                          fc_b, logits, ids, err_flag, workspace, workspace_bytes, stream);
}

int nsd_stream_push_slots(const float* bins_in, float* rawring, int ring_rows, const int64_t* day_idx, const float* day_w, const float* day_b,
                          int n_days, const float* taps, int ntaps, void* x0buf_bf16, int* n_bins, const int* active, const int* last_frame,
                          int* emitted, int B, int N, int K, int S, int H, int L, int C, const void* const* w_ih_bf16,
                          const void* const* w_hh_bf16, const void* const* b_ih, const void* const* b_hh, float* h, void* h_bf16,
                          const void* fc_w_bf16, const float* fc_b, float* logits, int* ids, int* err_flag, void* workspace,
                          size_t workspace_bytes, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(active && last_frame && emitted, "stream_push_slots: null pointer");
    NSD_CHECK_ARG(S >= 1 && ntaps >= 1, "stream_push_slots: bad sizes S=%d ntaps=%d", S, ntaps);
    // every utterance starts at bin 0 and moves one stride per push: bins past the newest frame's look-ahead are one constant
    const int right = ntaps - 1 - (ntaps - 1) / 2, extra = ((-(K + right)) % S + S) % S;
    return nsd::stream_push_launch<true>(bins_in, rawring, ring_rows, day_idx, day_w, day_b, n_days, taps, ntaps, x0buf_bf16, n_bins, active,
                                         last_frame, emitted, extra, B, N, K, S, H, L, C, w_ih_bf16, w_hh_bf16, b_ih, b_hh, h, h_bf16,
                                         fc_w_bf16, fc_b, logits, ids, err_flag, workspace, workspace_bytes, stream);
}

}  // extern "C"
