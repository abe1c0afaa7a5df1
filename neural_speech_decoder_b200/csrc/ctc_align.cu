// K5c: CTC forced alignment -- the Viterbi (max-product) form of K4's alpha recursion over the same blank-extended lattice, plus a
// backtrace, for a whole batch in one launch.  Semantics: include/nsd_b200.h.
//
// One CTA per utterance, ALIGN_THREADS threads.  The frames are consumed in chunks of ALIGN_F: warps 1..7 load (and, for logits,
// log-softmax with the arithmetic of log_softmax_kernel) the rows of chunk k+1 into a shared ring while warp 0 runs the recursion over
// chunk k, so the recursion reads its emissions from shared memory.  Warp 0 walks the actual 2L+1 states (lane + 32 j), keeps two delta
// rows in shared memory with -inf guard cells in front (as K4's alpha warp does) and records each state's choice as a 2-bit code: two
// ballots per 32 states, one uint2 per (frame, group) in the workspace.  The backtrace (warp 0) fetches the codes of 32 frames at once --
// lane i holds frame t-i's words for the three groups the path can reach in 32 steps -- and walks them with shuffles.  A last pass over
// frames (all warps) writes labels / frame_logp / span ends, then one over tokens writes spans / token_logp.
#include <math.h>

#include "common.cuh"

namespace nsd {

constexpr int ALIGN_THREADS = 256;
constexpr int ALIGN_F = 32;                        // frames per chunk of the emission ring
constexpr int ALIGN_PRODUCERS = ALIGN_THREADS / 32 - 1;
constexpr int ALIGN_ROWS_PER_PRODUCER = (ALIGN_F + ALIGN_PRODUCERS - 1) / ALIGN_PRODUCERS;
constexpr int ALIGN_MAX_C = 128;
constexpr int ALIGN_MAX_T = 8192;
constexpr int ALIGN_MAX_TGT = 1024;
constexpr int ALIGN_SKIP = 1 << 30;                // ext[] flag: the s-2 predecessor counts

struct AlignParams {
    const float* act; int64_t st, sb, sc; int is_logits;
    const int32_t* targets; int tgt_stride; const int32_t* in_lens; const int32_t* tgt_lens;
    int T, C, blank, max_tgt, SP, NJ;              // SP = 2*max_tgt+1, NJ = ceil(SP/32): groups per frame of the code table
    int32_t* labels; float* frame_logp; int32_t* spans; float* token_logp; float* score; int* err_flag;
    uint2* codes;                                  // [B][T][NJ]: bit (s & 31) of .x / .y = bit 0 / 1 of state s's code
};

// Rows t in [t0, t0+ALIGN_F) ∩ [0, il) of this warp's share -> ybuf (log-softmaxed if is_logits), and (m, lz) of each row -> mlz.
__device__ __forceinline__ void align_produce(const AlignParams& p, int b, int il, int t0, int pw, int lane, float* ybuf, float2* mlz) {
    const int C = p.C;
    float v[ALIGN_ROWS_PER_PRODUCER][4];
#pragma unroll
    for (int i = 0; i < ALIGN_ROWS_PER_PRODUCER; ++i) {          // every load of the share in flight at once
        const int f = pw + ALIGN_PRODUCERS * i, t = t0 + f;
        const float* a = p.act + (int64_t)t * p.st + (int64_t)b * p.sb;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int c = lane + 32 * q;
            v[i][q] = (f < ALIGN_F && t < il && c < C) ? a[(int64_t)c * p.sc] : 0.f;
        }
    }
#pragma unroll
    for (int i = 0; i < ALIGN_ROWS_PER_PRODUCER; ++i) {
        const int f = pw + ALIGN_PRODUCERS * i, t = t0 + f;
        if (f >= ALIGN_F || t >= il) continue;
        float* y = ybuf + (size_t)(t % (2 * ALIGN_F)) * C;
        if (p.is_logits) {                                       // log_softmax_kernel's arithmetic, bit for bit
            float m = -INFINITY;
#pragma unroll
            for (int q = 0; q < 4; ++q) if (lane + 32 * q < C) m = fmaxf(m, v[i][q]);
            m = warp_max(m);
            float s = 0.f;
#pragma unroll
            for (int q = 0; q < 4; ++q) if (lane + 32 * q < C) s += expf(v[i][q] - m);
            s = warp_sum(s);
            const float lz = logf(s);
#pragma unroll
            for (int q = 0; q < 4; ++q) if (lane + 32 * q < C) y[lane + 32 * q] = v[i][q] - m - lz;
            if (lane == 0) mlz[t] = make_float2(m, lz);
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) if (lane + 32 * q < C) y[lane + 32 * q] = v[i][q];
        }
    }
}

__global__ void __launch_bounds__(ALIGN_THREADS) ctc_align_kernel(AlignParams p) {
    pdl_enter();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_rep, s_bad;
    __shared__ float s_score;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int T = p.T, C = p.C, SP = p.SP;
    const int il = min(max(p.in_lens[b], 0), T);
    const int L = min(max(p.tgt_lens[b], 0), p.max_tgt);
    const int S = 2 * L + 1;

    float* ybuf = reinterpret_cast<float*>(smem_raw);                       // [2*ALIGN_F][C]   emission ring
    float* rows = ybuf + 2 * ALIGN_F * C;                                    // [2][SP+2]        delta ping-pong; later span ends
    int* ext = reinterpret_cast<int*>(rows + 2 * (SP + 2));                  // [SP]             label | ALIGN_SKIP
    float2* mlz = reinterpret_cast<float2*>(ext + SP + (SP & 1));            // [T]              (m, lz) per row; later frame_logp
    short* path = reinterpret_cast<short*>(mlz + T);                         // [T]              state of every frame
    uint2* codes = p.codes + (size_t)b * T * p.NJ;

    if (tid == 0) { s_rep = 0; s_bad = 0; }
    __syncthreads();
    for (int s = tid; s < S; s += ALIGN_THREADS) {
        int v = p.blank, skip = 0;
        if (s & 1) {
            const int32_t* tg = p.targets + (size_t)b * p.tgt_stride;
            const int k = s >> 1;
            v = tg[k];
            if (v == p.blank || v < 0 || v >= C) { atomicOr(&s_bad, 1); v = p.blank; }
            if (k > 0) {
                const int u = tg[k - 1];
                if (u == v) atomicAdd(&s_rep, 1);
                else if (s >= 3) skip = ALIGN_SKIP;
            }
        }
        ext[s] = v | skip;
    }
    __syncthreads();
    if (s_bad && tid == 0 && p.err_flag != nullptr) *p.err_flag = 1;
    // feasible: every target valid and enough frames for L labels plus a blank between each adjacent equal pair
    const bool feasible = !s_bad && il >= L + s_rep;

    if (feasible && il > 0) {
        const int nch = (il + ALIGN_F - 1) / ALIGN_F;
        const int NJ = (S + 31) >> 5;
        float* prev = rows + 2;
        float* cur = rows + (SP + 2) + 2;
        if (warp > 0) align_produce(p, b, il, 0, warp - 1, lane, ybuf, mlz);
        __syncthreads();
        for (int k = 0; k < nch; ++k) {
            if (warp == 0) {
                int t = k * ALIGN_F;
                if (k == 0) {                                                // delta_0
                    if (lane == 0) { rows[0] = rows[1] = -INFINITY; rows[SP + 2] = rows[SP + 3] = -INFINITY; }
                    for (int s = lane; s < S; s += 32) prev[s] = s < 2 ? ybuf[ext[s] & (ALIGN_SKIP - 1)] : -INFINITY;
                    __syncwarp();
                    t = 1;
                }
                const int t1 = min(il, (k + 1) * ALIGN_F);
                for (; t < t1; ++t) {
                    const float* y = ybuf + (size_t)(t % (2 * ALIGN_F)) * C;
                    uint2* row_codes = codes + (size_t)t * p.NJ;
                    for (int j = 0; j < NJ; ++j) {
                        const int s = lane + 32 * j;
                        int code = 0;
                        if (s < S) {
                            const int e = ext[s];
                            float best = prev[s];
                            const float a1 = prev[s - 1];
                            if (a1 > best) { best = a1; code = 1; }             // ties stay: s, then s-1, then s-2
                            if (e & ALIGN_SKIP) {
                                const float a2 = prev[s - 2];
                                if (a2 > best) { best = a2; code = 2; }
                            }
                            cur[s] = best + y[e & (ALIGN_SKIP - 1)];
                        }
                        const unsigned b0 = __ballot_sync(0xffffffffu, code & 1), b1 = __ballot_sync(0xffffffffu, code >> 1);
                        if (lane == 0) row_codes[j] = make_uint2(b0, b1);
                    }
                    __syncwarp();
                    float* tmp = prev; prev = cur; cur = tmp;
                }
            } else if (k + 1 < nch) {
                align_produce(p, b, il, (k + 1) * ALIGN_F, warp - 1, lane, ybuf, mlz);
            }
            __syncthreads();
        }
        if (warp == 0) {
            // end state: argmax(delta(S-1), delta(S-2)), ties -> S-1
            int s = S - 1;
            if (S > 1 && prev[S - 2] > prev[S - 1]) s = S - 2;
            if (lane == 0) s_score = prev[s];
            // backtrace, 32 frames per round: lane i holds the code words of frame t-i for groups j0, j0-1, j0-2 (the path drops at most
            // 2 states a frame, so from state s at frame t it stays within s-62 .. s for the next 31 frames)
            int t = il - 1;
            while (t >= 1) {
                const int j0 = s >> 5, tl = t - lane;
                uint2 w0 = make_uint2(0u, 0u), w1 = w0, w2 = w0;
                if (tl >= 1) {
                    const uint2* rc = codes + (size_t)tl * p.NJ;
                    w0 = rc[j0];
                    if (j0 >= 1) w1 = rc[j0 - 1];
                    if (j0 >= 2) w2 = rc[j0 - 2];
                }
                const int n = min(32, t);
                for (int i = 0; i < n; ++i) {
                    const int d = j0 - (s >> 5);
                    const uint2 w = d == 0 ? w0 : (d == 1 ? w1 : w2);
                    const unsigned x = __shfl_sync(0xffffffffu, w.x, i), y = __shfl_sync(0xffffffffu, w.y, i);
                    const int bit = s & 31;
                    if (lane == 0) path[t - i] = (short)s;
                    s -= (int)((x >> bit) & 1u) | (int)(((y >> bit) & 1u) << 1);
                }
                t -= n;
            }
            if (lane == 0) path[0] = (short)s;
        }
    } else if (tid == 0) {
        s_score = feasible ? 0.f : -INFINITY;                                // il == 0, L == 0: the empty path
    }
    __syncthreads();

    // outputs.  ok: a path exists (a feasible utterance whose best final delta is above -inf; NaN inputs can make it NaN)
    const float score = s_score;
    const bool ok = feasible && il > 0 && score > -INFINITY;
    if (tid == 0) p.score[b] = score;
    int* span0 = reinterpret_cast<int*>(rows);                               // [max_tgt] first frame of token k
    int* span1 = span0 + p.max_tgt;                                          // [max_tgt] last frame
    float* flp = reinterpret_cast<float*>(mlz);                              // frame_logp[t] in slot 2t (after (m, lz) of row t is read)
    for (int t = tid; t < T; t += ALIGN_THREADS) {
        int lab = -1;
        float v = 0.f;
        if (ok && t < il) {
            const int s = path[t];
            lab = ext[s] & (ALIGN_SKIP - 1);
            const float a = p.act[(int64_t)t * p.st + (int64_t)b * p.sb + (int64_t)lab * p.sc];
            if (p.is_logits) {
                const float2 ml = mlz[t];
                v = a - ml.x - ml.y;
            } else {
                v = a;
            }
            flp[2 * t] = v;
            if (s & 1) {
                if (t == 0 || path[t - 1] != s) span0[s >> 1] = t;
                if (t == il - 1 || path[t + 1] != s) span1[s >> 1] = t;
            }
        }
        p.labels[(size_t)b * T + t] = lab;
        p.frame_logp[(size_t)b * T + t] = v;
    }
    __syncthreads();
    for (int k = tid; k < p.max_tgt; k += ALIGN_THREADS) {
        int f0 = -1, f1 = -1;
        float acc = 0.f;
        if (ok && k < L) {
            f0 = span0[k]; f1 = span1[k];
            acc = flp[2 * f0];
            for (int t = f0 + 1; t <= f1; ++t) acc += flp[2 * t];
        }
        p.spans[((size_t)b * p.max_tgt + k) * 2] = f0;
        p.spans[((size_t)b * p.max_tgt + k) * 2 + 1] = f1;
        p.token_logp[(size_t)b * p.max_tgt + k] = acc;
    }
}

static size_t align_smem(int T, int C, int max_tgt) {
    const size_t SP = 2 * (size_t)max_tgt + 1;
    return sizeof(float) * (2 * (size_t)ALIGN_F * C + 2 * (SP + 2)) + sizeof(int) * (SP + (SP & 1)) + sizeof(float2) * (size_t)T +
           sizeof(short) * (size_t)T;
}

}  // namespace nsd

extern "C" {

size_t nsd_ctc_align_workspace(int T, int B, int C, int max_tgt) {
    (void)C;
    const size_t NJ = (2 * (size_t)(max_tgt > 0 ? max_tgt : 0) + 1 + 31) / 32;
    return sizeof(uint2) * (size_t)(B > 0 ? B : 0) * (size_t)(T > 0 ? T : 0) * NJ;
}

int nsd_ctc_align(const float* act, int64_t st, int64_t sb, int64_t sc, int is_logits, const int32_t* targets, int tgt_stride,
                  const int32_t* in_lens, const int32_t* tgt_lens, int T, int B, int C, int blank, int max_tgt, int32_t* labels,
                  float* frame_logp, int32_t* spans, float* token_logp, float* score, int* err_flag, void* workspace,
                  size_t workspace_bytes, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(T >= 1 && T <= ALIGN_MAX_T && B >= 1 && C >= 1 && C <= ALIGN_MAX_C,
                  "ctc_align: bad sizes T=%d B=%d C=%d (1 <= T <= %d, C <= %d)", T, B, C, ALIGN_MAX_T, ALIGN_MAX_C);
    NSD_CHECK_ARG(max_tgt >= 0 && max_tgt <= ALIGN_MAX_TGT, "ctc_align: max_tgt=%d outside [0, %d]", max_tgt, ALIGN_MAX_TGT);
    NSD_CHECK_ARG(blank >= 0 && blank < C, "ctc_align: blank=%d out of range", blank);
    NSD_CHECK_ARG(max_tgt == 0 || tgt_stride >= max_tgt, "ctc_align: tgt_stride=%d < max_tgt=%d", tgt_stride, max_tgt);
    if (workspace_bytes < nsd_ctc_align_workspace(T, B, C, max_tgt)) { set_error("ctc_align: workspace too small"); return NSD_ERR_WORKSPACE; }
    AlignParams p;
    p.act = act; p.st = st; p.sb = sb; p.sc = sc; p.is_logits = is_logits;
    p.targets = targets; p.tgt_stride = tgt_stride; p.in_lens = in_lens; p.tgt_lens = tgt_lens;
    p.T = T; p.C = C; p.blank = blank; p.max_tgt = max_tgt; p.SP = 2 * max_tgt + 1; p.NJ = (p.SP + 31) / 32;
    p.labels = labels; p.frame_logp = frame_logp; p.spans = spans; p.token_logp = token_logp; p.score = score; p.err_flag = err_flag;
    p.codes = reinterpret_cast<uint2*>(workspace);
    const size_t smem = align_smem(T, C, max_tgt);
    if (smem > 48 * 1024) NSD_CUDA(cudaFuncSetAttribute(ctc_align_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nsd::launch_k(ctc_align_kernel, B, ALIGN_THREADS, smem, (cudaStream_t)stream, p);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

}  // extern "C"
