// K5b: CTC prefix beam search with an optional phoneme-bigram prior, state resumable on the device.
//
// No counterpart in the reference: its evaluation decodes greedily (trainer:313-320).  This produces the N-best lists with
// scores that a downstream rescorer consumes.  Semantics (log space, a (+) b = logaddexp):
//   beam entry l: (Pb, Pnb, prior); start {empty: Pb = 0, Pnb = -inf, prior = 0}
//   stay        Pb'(l)  = (Pb (+) Pnb) + y[blank];   Pnb'(l) = Pnb + y[last(l)]   (l non-empty)
//   extend      Pnb'(l.c) = (c == last(l) ? Pb : Pb (+) Pnb) + y[c],  c != blank,  prior(l.c) = prior(l) + a*lm[last(l)|blank, c] + b
//   merge       l.c already in the beam: Pnb'(l.c) = (Pnb(l.c) + y[c]) (+) extension from l, and the extension is not a candidate
//   rank        total = (Pb' (+) Pnb') + prior, keep the best W, ties -> smaller key (stay of slot i: i*(C+1), extension by c:
//               i*(C+1)+c+1), candidates at -inf (or NaN) are never kept; the new beam is stored in rank order.
// One CTA per utterance runs the frames in order (a latency-bound serial chain like K4).  Per frame:
//   1. warp 0 log-softmaxes the row (arithmetic of log_softmax_kernel) while the next row's load is already in flight;
//      every slot finds its parent among the other slots (the merge map);
//   2. one thread per candidate computes its total and an order-preserving 32-bit key;
//   3. an MSD radix select over the unique 64-bit (key, ~candidate index) finds the W-th best exactly;
//   4. the survivors are ranked among themselves (<= W^2 comparisons) and the extensions among them take trie nodes by a
//      prefix sum in rank order.
// Every decision is an integer comparison or an exact count, so the result does not depend on thread scheduling: one call
// and any chunking of the same frames give the same bits.
#include <math.h>

#include "common.cuh"

namespace nsd {

constexpr int BEAM_THREADS = 256;
constexpr int BEAM_MAX_W = 128;
constexpr int BEAM_MAX_C = 128;
constexpr unsigned long long BEAM_HASH_MUL = 0x9E3779B97F4A7C15ull;
constexpr unsigned long long BEAM_KEY_BITS = 0x7FFFull;    // candidate index < 128 * 129 < 2^15
static_assert(BEAM_THREADS == 256, "one radix-select bin per thread");
static_assert(BEAM_MAX_W * (BEAM_MAX_C + 1) <= (int)BEAM_KEY_BITS + 1, "candidate index must fit the composite's low bits");

__host__ __device__ inline size_t al16(size_t x) { return (x + 15) & ~(size_t)15; }

// Byte offsets inside one utterance's block of the state.  Header: int32 {frames_done, nodes, size, 0}; then the W slots
// (prefix hash, parent's hash, Pb, Pnb, prior, trie node, parent node, last token, length); then the trie of
// 1 + W*max_frames nodes int2 {parent node, token}, node 0 = the empty prefix.
struct BeamLayout {
    size_t hash, phash, pb, pnb, prior, node, pnode, last, len, trie, bytes;
};

__host__ __device__ inline BeamLayout beam_layout(int W, int max_frames) {
    BeamLayout L;
    size_t o = 16;
    L.hash = o; o += 8 * (size_t)W;
    L.phash = o; o += 8 * (size_t)W;
    L.pb = o; o += 4 * (size_t)W;
    L.pnb = o; o += 4 * (size_t)W;
    L.prior = o; o += 4 * (size_t)W;
    L.node = o; o += 4 * (size_t)W;
    L.pnode = o; o += 4 * (size_t)W;
    L.last = o; o += 4 * (size_t)W;
    L.len = o; o += 4 * (size_t)W;
    L.trie = al16(o);
    L.bytes = al16(L.trie + 8 * (1 + (size_t)W * max_frames));
    return L;
}

// One beam in shared memory (structure of arrays).  par: slot of the parent prefix in the same beam, or -1.
struct Beam {
    unsigned long long *hash, *phash;
    float *pb, *pnb, *prior;
    int *node, *pnode, *last, *len, *par;
};

__device__ __forceinline__ Beam carve_beam(unsigned char* p, int W) {
    Beam b;
    b.hash = reinterpret_cast<unsigned long long*>(p); p += 8 * W;
    b.phash = reinterpret_cast<unsigned long long*>(p); p += 8 * W;
    b.pb = reinterpret_cast<float*>(p); p += 4 * W;
    b.pnb = reinterpret_cast<float*>(p); p += 4 * W;
    b.prior = reinterpret_cast<float*>(p); p += 4 * W;
    b.node = reinterpret_cast<int*>(p); p += 4 * W;
    b.pnode = reinterpret_cast<int*>(p); p += 4 * W;
    b.last = reinterpret_cast<int*>(p); p += 4 * W;
    b.len = reinterpret_cast<int*>(p); p += 4 * W;
    b.par = reinterpret_cast<int*>(p);
    return b;
}
constexpr int BEAM_SLOT_SMEM = 8 + 8 + 4 * 3 + 4 * 5;

__device__ __forceinline__ float lse2(float a, float b) {
    const float m = fmaxf(a, b);
    if (m == -INFINITY) return -INFINITY;
    return m + logf(expf(a - m) + expf(b - m));
}

// Larger float -> larger key; -inf and NaN -> 0 (never kept), every other value > 0.
__device__ __forceinline__ unsigned int order_key(float v) {
    if (!(v > -INFINITY)) return 0u;
    const unsigned int u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ unsigned long long composite(unsigned int u, int k) {
    return ((unsigned long long)u << 32) | (BEAM_KEY_BITS - (unsigned long long)k);
}

// true iff trie nodes a and b (prefixes of the same length) spell the same prefix
__device__ bool same_prefix(const int2* trie, int a, int b) {
    while (a != b) {
        const int2 ea = trie[a], eb = trie[b];
        if (ea.y != eb.y) return false;
        a = ea.x;
        b = eb.x;
    }
    return true;
}

struct BeamParams {
    const float* act; int64_t st, sb, sc; int is_logits; const int32_t* lens;
    int T, C, blank; const float* lm; float alpha, beta;
    int W, max_frames; unsigned char* state; BeamLayout L; int* err_flag;
};

// Candidate (slot i, r): r == 0 is the stay of slot i, r = c + 1 its extension by c.  Returns the ranking total.
__device__ __forceinline__ float candidate(const Beam& bm, int i, int r, const float* y, const BeamParams& p, float& opb, float& opnb,
                                           float& oprior) {
    const float pb = bm.pb[i], pnb = bm.pnb[i];
    const int last = bm.last[i];
    if (r == 0) {
        opb = lse2(pb, pnb) + y[p.blank];
        float v = last >= 0 ? pnb + y[last] : -INFINITY;
        const int q = bm.par[i];
        if (q >= 0) v = lse2(v, (bm.last[q] == last ? bm.pb[q] : lse2(bm.pb[q], bm.pnb[q])) + y[last]);
        opnb = v;
        oprior = bm.prior[i];
    } else {
        const int c = r - 1;
        opb = -INFINITY;
        opnb = (c == last ? pb : lse2(pb, pnb)) + y[c];
        const int ctx = last >= 0 ? last : p.blank;
        oprior = bm.prior[i] + (p.lm != nullptr ? fmaf(p.alpha, p.lm[ctx * p.C + c], p.beta) : p.beta);
    }
    return lse2(opb, opnb) + oprior;
}

__global__ void __launch_bounds__(BEAM_THREADS) ctc_beam_advance_kernel(BeamParams p) {
    pdl_enter();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ float s_y[BEAM_MAX_C];
    __shared__ unsigned int s_merged[BEAM_MAX_W * 4];      // bit c of row i: the extension of slot i by c is already a slot
    __shared__ int s_hist[256];
    __shared__ int s_sel[4];                               // radix select: digit, count above it, count in it, all-valid flag
    __shared__ int s_wext[BEAM_MAX_W / 32];
    __shared__ int s_cnt;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int W = p.W, C = p.C, C1 = p.C + 1;

    unsigned char* g = p.state + (size_t)b * p.L.bytes;
    int* hdr = reinterpret_cast<int*>(g);
    int2* trie = reinterpret_cast<int2*>(g + p.L.trie);
    const int n = p.lens != nullptr ? min(max(p.lens[b], 0), p.T) : p.T;
    const int frames_done = hdr[0];
    if (n == 0) return;
    if (frames_done + n > p.max_frames) {                  // the trie could overflow: leave this utterance untouched
        if (tid == 0 && p.err_flag != nullptr) *p.err_flag = 1;
        return;
    }
    const int cap = 1 + W * p.max_frames;
    int nodes = hdr[1], size = hdr[2];

    unsigned char* sp = smem_raw;
    unsigned long long* surv = reinterpret_cast<unsigned long long*>(sp); sp += 8 * W;
    unsigned long long* ranked = reinterpret_cast<unsigned long long*>(sp); sp += 8 * W;
    unsigned char* beam_buf[2] = {sp, sp + BEAM_SLOT_SMEM * W};      // ping-pong: frame t reads buffer t & 1
    unsigned int* ukey = reinterpret_cast<unsigned int*>(sp + 2 * BEAM_SLOT_SMEM * W);   // [W*(C+1)]

    if (tid < size) {
        const Beam d = carve_beam(beam_buf[0], W);
        d.hash[tid] = reinterpret_cast<const unsigned long long*>(g + p.L.hash)[tid];
        d.phash[tid] = reinterpret_cast<const unsigned long long*>(g + p.L.phash)[tid];
        d.pb[tid] = reinterpret_cast<const float*>(g + p.L.pb)[tid];
        d.pnb[tid] = reinterpret_cast<const float*>(g + p.L.pnb)[tid];
        d.prior[tid] = reinterpret_cast<const float*>(g + p.L.prior)[tid];
        d.node[tid] = reinterpret_cast<const int*>(g + p.L.node)[tid];
        d.pnode[tid] = reinterpret_cast<const int*>(g + p.L.pnode)[tid];
        d.last[tid] = reinterpret_cast<const int*>(g + p.L.last)[tid];
        d.len[tid] = reinterpret_cast<const int*>(g + p.L.len)[tid];
    }
    // warp 0 keeps the next row in flight: lane holds classes lane, lane+32, lane+64, lane+96
    float nxt_row[4];
    if (warp == 0) {
        const float* a = p.act + (int64_t)b * p.sb;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = lane + 32 * k;
            nxt_row[k] = c < C ? a[(int64_t)c * p.sc] : 0.f;
        }
    }

    int t = 0;
    for (; t < n; ++t) {
        const Beam cur = carve_beam((t & 1) ? beam_buf[1] : beam_buf[0], W);
        const Beam nb = carve_beam((t & 1) ? beam_buf[0] : beam_buf[1], W);
        // ---- 1. row, merge map, cleared counters
        if (warp == 0) {
            float a[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) a[k] = nxt_row[k];
            if (t + 1 < n) {
                const float* an = p.act + (int64_t)(t + 1) * p.st + (int64_t)b * p.sb;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = lane + 32 * k;
                    if (c < C) nxt_row[k] = an[(int64_t)c * p.sc];
                }
            }
            if (p.is_logits) {
                float m = -INFINITY;
#pragma unroll
                for (int k = 0; k < 4; ++k) if (lane + 32 * k < C) m = fmaxf(m, a[k]);
                m = warp_max(m);
                float s = 0.f;
#pragma unroll
                for (int k = 0; k < 4; ++k) if (lane + 32 * k < C) s += expf(a[k] - m);
                s = warp_sum(s);
                const float lz = logf(s);
#pragma unroll
                for (int k = 0; k < 4; ++k) if (lane + 32 * k < C) s_y[lane + 32 * k] = a[k] - m - lz;
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) if (lane + 32 * k < C) s_y[lane + 32 * k] = a[k];
            }
        }
        for (int i = tid; i < size * 4; i += BEAM_THREADS) s_merged[i] = 0u;
        s_hist[tid] = 0;                                   // BEAM_THREADS == 256 bins
        if (tid == 0) s_cnt = 0;
        if (tid < size) {
            int q = -1;
            const int lj = cur.len[tid];
            if (lj > 0) {
                const int pn = cur.pnode[tid];
                const unsigned long long ph = cur.phash[tid];
                for (int i = 0; i < size; ++i) {
                    if (cur.len[i] != lj - 1) continue;
                    if (cur.node[i] == pn || (cur.hash[i] == ph && same_prefix(trie, cur.node[i], pn))) { q = i; break; }
                }
            }
            cur.par[tid] = q;
        }
        __syncthreads();
        if (tid < size && cur.par[tid] >= 0) {
            const int c = cur.last[tid];
            atomicOr(&s_merged[cur.par[tid] * 4 + (c >> 5)], 1u << (c & 31));
        }
        __syncthreads();

        // ---- 2. every candidate's key, histogram of the top byte
        const int N = size * C1;
        for (int k = tid; k < N; k += BEAM_THREADS) {
            const int i = k / C1, r = k - i * C1;
            unsigned int u = 0u;
            if (r == 0 || (r - 1 != p.blank && !((s_merged[i * 4 + ((r - 1) >> 5)] >> ((r - 1) & 31)) & 1u))) {
                float a0, a1, a2;
                u = order_key(candidate(cur, i, r, s_y, p, a0, a1, a2));
            }
            ukey[k] = u;
            if (u != 0u) atomicAdd(&s_hist[u >> 24], 1);
        }
        __syncthreads();

        // ---- 3. radix select of the W-th best over the unique composite (key << 32 | ~index)
        unsigned long long prefix = 0ull, mask = 0ull, thr = 0ull;
        int need = W;
        for (int pass = 0; pass < 6; ++pass) {
            const int sh = pass < 4 ? 56 - 8 * pass : (pass == 4 ? 8 : 0);
            if (pass > 0) {
                for (int k = tid; k < N; k += BEAM_THREADS) {
                    const unsigned int u = ukey[k];
                    if (u == 0u) continue;
                    const unsigned long long cv = composite(u, k);
                    if ((cv & mask) == prefix) atomicAdd(&s_hist[(int)((cv >> sh) & 255ull)], 1);
                }
                __syncthreads();
            }
            if (warp == 0) {
                int cnt[8], tot = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) { cnt[j] = s_hist[255 - 8 * lane - j]; tot += cnt[j]; }
                int incl = tot;                            // inclusive scan, lane 0 = the highest bins
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += v;
                }
                const int excl = incl - tot;
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                if (pass == 0 && total <= need) {
                    if (lane == 0) s_sel[3] = 1;
                } else {
                    if (excl < need && need <= incl) {
                        int run = excl;
                        for (int j = 0; j < 8; ++j) {
                            if (run + cnt[j] >= need) {
                                s_sel[0] = 255 - 8 * lane - j; s_sel[1] = run; s_sel[2] = cnt[j];
                                break;
                            }
                            run += cnt[j];
                        }
                    }
                    if (lane == 0) s_sel[3] = 0;
                }
            }
            __syncthreads();
            if (s_sel[3]) { thr = 1ull << 32; break; }     // no more valid candidates than slots: keep every one
            prefix |= (unsigned long long)s_sel[0] << sh;
            mask |= 255ull << sh;
            need -= s_sel[1];
            const bool done = s_sel[2] == need;            // the whole bin is kept
            __syncthreads();
            s_hist[tid] = 0;
            __syncthreads();
            if (done) { thr = prefix; break; }
        }

        // ---- 4. survivors, their rank, trie nodes for the extensions
        for (int k = tid; k < N; k += BEAM_THREADS) {
            const unsigned int u = ukey[k];
            if (u == 0u) continue;
            const unsigned long long cv = composite(u, k);
            if (cv >= thr) surv[atomicAdd(&s_cnt, 1)] = cv;
        }
        __syncthreads();
        const int ns = s_cnt;
        if (tid < ns) {
            const unsigned long long cv = surv[tid];
            int rank = 0;
            for (int q = 0; q < ns; ++q) rank += surv[q] > cv;
            ranked[rank] = cv;
        }
        __syncthreads();
        int i = 0, r = 0;
        if (tid < ns) {
            const int k = (int)(BEAM_KEY_BITS - (ranked[tid] & BEAM_KEY_BITS));
            i = k / C1;
            r = k - i * C1;
        }
        const unsigned int em = __ballot_sync(0xffffffffu, tid < ns && r > 0);
        if (lane == 0 && warp < BEAM_MAX_W / 32) s_wext[warp] = __popc(em);
        __syncthreads();
        int off = nodes, n_ext = 0;
#pragma unroll
        for (int w = 0; w < BEAM_MAX_W / 32; ++w) {
            off += w < warp ? s_wext[w] : 0;
            n_ext += s_wext[w];
        }
        if (nodes + n_ext > cap) {                         // unreachable while frames_done <= max_frames; a backstop
            if (tid == 0 && p.err_flag != nullptr) *p.err_flag = 1;
            break;
        }
        if (tid < ns) {
            off += __popc(em & ((1u << lane) - 1u));
            float npb, npnb, nprior;
            candidate(cur, i, r, s_y, p, npb, npnb, nprior);
            nb.pb[tid] = npb;
            nb.pnb[tid] = npnb;
            nb.prior[tid] = nprior;
            if (r == 0) {
                nb.hash[tid] = cur.hash[i];
                nb.phash[tid] = cur.phash[i];
                nb.node[tid] = cur.node[i];
                nb.pnode[tid] = cur.pnode[i];
                nb.last[tid] = cur.last[i];
                nb.len[tid] = cur.len[i];
            } else {
                const int c = r - 1;
                nb.hash[tid] = cur.hash[i] * BEAM_HASH_MUL + (unsigned long long)(c + 1);
                nb.phash[tid] = cur.hash[i];
                nb.node[tid] = off;
                nb.pnode[tid] = cur.node[i];
                nb.last[tid] = c;
                nb.len[tid] = cur.len[i] + 1;
                trie[off] = make_int2(cur.node[i], c);
            }
        }
        nodes += n_ext;
        size = ns;
        __syncthreads();
    }

    // ---- write the beam back (t frames were applied)
    const Beam fin = carve_beam((t & 1) ? beam_buf[1] : beam_buf[0], W);
    if (tid < size) {
        reinterpret_cast<unsigned long long*>(g + p.L.hash)[tid] = fin.hash[tid];
        reinterpret_cast<unsigned long long*>(g + p.L.phash)[tid] = fin.phash[tid];
        reinterpret_cast<float*>(g + p.L.pb)[tid] = fin.pb[tid];
        reinterpret_cast<float*>(g + p.L.pnb)[tid] = fin.pnb[tid];
        reinterpret_cast<float*>(g + p.L.prior)[tid] = fin.prior[tid];
        reinterpret_cast<int*>(g + p.L.node)[tid] = fin.node[tid];
        reinterpret_cast<int*>(g + p.L.pnode)[tid] = fin.pnode[tid];
        reinterpret_cast<int*>(g + p.L.last)[tid] = fin.last[tid];
        reinterpret_cast<int*>(g + p.L.len)[tid] = fin.len[tid];
    }
    if (tid == 0) {
        hdr[0] = frames_done + t;
        hdr[1] = nodes;
        hdr[2] = size;
    }
}

// mask == nullptr: every utterance; otherwise only those with mask[b] != 0 (the others keep every byte)
__global__ void ctc_beam_init_kernel(unsigned char* state, BeamLayout L, const int32_t* mask) {
    pdl_enter();
    if (threadIdx.x != 0 || (mask != nullptr && mask[blockIdx.x] == 0)) return;
    unsigned char* g = state + (size_t)blockIdx.x * L.bytes;
    int* hdr = reinterpret_cast<int*>(g);
    hdr[0] = 0; hdr[1] = 1; hdr[2] = 1; hdr[3] = 0;
    reinterpret_cast<unsigned long long*>(g + L.hash)[0] = 0ull;
    reinterpret_cast<unsigned long long*>(g + L.phash)[0] = 0ull;
    reinterpret_cast<float*>(g + L.pb)[0] = 0.f;
    reinterpret_cast<float*>(g + L.pnb)[0] = -INFINITY;
    reinterpret_cast<float*>(g + L.prior)[0] = 0.f;
    reinterpret_cast<int*>(g + L.node)[0] = 0;
    reinterpret_cast<int*>(g + L.pnode)[0] = -1;
    reinterpret_cast<int*>(g + L.last)[0] = -1;
    reinterpret_cast<int*>(g + L.len)[0] = 0;
    reinterpret_cast<int2*>(g + L.trie)[0] = make_int2(-1, -1);
}

// One CTA per utterance: thread k walks hypothesis k's trie path backwards; then the block pads every row with -1.
__global__ void ctc_beam_nbest_kernel(const unsigned char* state, BeamLayout L, int nbest, int64_t* hyps, int hyp_stride,
                                      int32_t* hyp_len, float* score, float* acoustic) {
    pdl_enter();
    __shared__ int s_len[BEAM_MAX_W];
    const int b = blockIdx.x, k = threadIdx.x;
    const unsigned char* g = state + (size_t)b * L.bytes;
    const int size = reinterpret_cast<const int*>(g)[2];
    const int2* trie = reinterpret_cast<const int2*>(g + L.trie);
    int64_t* out = hyps + (size_t)b * nbest * hyp_stride;
    if (k < nbest) {
        const size_t o = (size_t)b * nbest + k;
        int len = 0;
        if (k < size) {
            len = reinterpret_cast<const int*>(g + L.len)[k];
            const float a = lse2(reinterpret_cast<const float*>(g + L.pb)[k], reinterpret_cast<const float*>(g + L.pnb)[k]);
            score[o] = a + reinterpret_cast<const float*>(g + L.prior)[k];
            acoustic[o] = a;
            int node = reinterpret_cast<const int*>(g + L.node)[k];
            for (int pos = len - 1; pos >= 0; --pos) {
                const int2 e = trie[node];
                out[(size_t)k * hyp_stride + pos] = e.y;
                node = e.x;
            }
        } else {
            score[o] = -INFINITY;
            acoustic[o] = -INFINITY;
        }
        hyp_len[o] = len;
        s_len[k] = len;
    }
    __syncthreads();
    for (size_t e = k; e < (size_t)nbest * hyp_stride; e += blockDim.x) {
        const int h = (int)(e / hyp_stride), pos = (int)(e - (size_t)h * hyp_stride);
        if (pos >= s_len[h]) out[e] = -1;
    }
}

}  // namespace nsd

extern "C" {

size_t nsd_ctc_beam_state_bytes(int B, int W, int max_frames) {
    if (B <= 0 || W <= 0 || max_frames <= 0) return 0;
    return (size_t)B * nsd::beam_layout(W, max_frames).bytes;
}

static int beam_check(int B, int W, int max_frames, size_t state_bytes) {
    using namespace nsd;
    NSD_CHECK_ARG(B > 0, "ctc_beam: bad batch %d", B);
    NSD_CHECK_ARG(W >= 1 && W <= BEAM_MAX_W, "ctc_beam: beam width %d outside [1, %d]", W, BEAM_MAX_W);
    NSD_CHECK_ARG(max_frames >= 1 && (long long)W * max_frames < (1ll << 30), "ctc_beam: max_frames=%d out of range for W=%d", max_frames, W);
    if (state_bytes < nsd_ctc_beam_state_bytes(B, W, max_frames)) {
        set_error("ctc_beam: state buffer too small (%zu < %zu bytes)", state_bytes, nsd_ctc_beam_state_bytes(B, W, max_frames));
        return NSD_ERR_WORKSPACE;
    }
    return NSD_OK;
}

int nsd_ctc_beam_init(void* state, size_t state_bytes, int B, int W, int max_frames, void* stream) {
    using namespace nsd;
    const int st = beam_check(B, W, max_frames, state_bytes);
    if (st != NSD_OK) return st;
    nsd::launch_k(ctc_beam_init_kernel, B, 32, 0, (cudaStream_t)stream, (unsigned char*)state, beam_layout(W, max_frames), (const int32_t*)nullptr);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

int nsd_ctc_beam_reset(void* state, size_t state_bytes, int B, int W, int max_frames, const int32_t* mask, void* stream) {
    using namespace nsd;
    const int st = beam_check(B, W, max_frames, state_bytes);
    if (st != NSD_OK) return st;
    NSD_CHECK_ARG(mask != nullptr, "ctc_beam_reset: null mask");
    nsd::launch_k(ctc_beam_init_kernel, B, 32, 0, (cudaStream_t)stream, (unsigned char*)state, beam_layout(W, max_frames), mask);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

int nsd_ctc_beam_advance(const float* act, int64_t st, int64_t sb, int64_t sc, int is_logits, const int32_t* lens, int T, int B,
                         int C, int blank, const float* lm_logp, float lm_weight, float insertion_bonus, int W, int max_frames,
                         void* state, size_t state_bytes, int* err_flag, void* stream) {
    using namespace nsd;
    const int s0 = beam_check(B, W, max_frames, state_bytes);
    if (s0 != NSD_OK) return s0;
    NSD_CHECK_ARG(T >= 0 && C >= 1 && C <= BEAM_MAX_C, "ctc_beam: bad sizes T=%d C=%d (C <= %d)", T, C, BEAM_MAX_C);
    NSD_CHECK_ARG(blank >= 0 && blank < C, "ctc_beam: blank=%d out of range", blank);
    if (T == 0) return NSD_OK;
    BeamParams p;
    p.act = act; p.st = st; p.sb = sb; p.sc = sc; p.is_logits = is_logits; p.lens = lens;
    p.T = T; p.C = C; p.blank = blank; p.lm = lm_logp; p.alpha = lm_weight; p.beta = insertion_bonus;
    p.W = W; p.max_frames = max_frames; p.state = (unsigned char*)state; p.L = beam_layout(W, max_frames); p.err_flag = err_flag;
    const size_t smem = 2 * 8 * (size_t)W + 2 * (size_t)BEAM_SLOT_SMEM * W + 4 * (size_t)W * (C + 1);
    if (smem > 48 * 1024) NSD_CUDA(cudaFuncSetAttribute(ctc_beam_advance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nsd::launch_k(ctc_beam_advance_kernel, B, BEAM_THREADS, smem, (cudaStream_t)stream, p);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

int nsd_ctc_beam_nbest(const void* state, int B, int W, int max_frames, int nbest, int64_t* hyps, int hyp_stride, int32_t* hyp_len,
                       float* score, float* acoustic, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(B > 0 && W >= 1 && W <= BEAM_MAX_W && max_frames >= 1, "ctc_beam_nbest: bad sizes B=%d W=%d max_frames=%d", B, W, max_frames);
    NSD_CHECK_ARG(nbest >= 1 && nbest <= W, "ctc_beam_nbest: nbest=%d outside [1, W=%d]", nbest, W);
    NSD_CHECK_ARG(hyp_stride >= max_frames, "ctc_beam_nbest: hyp_stride=%d < max_frames=%d", hyp_stride, max_frames);
    nsd::launch_k(ctc_beam_nbest_kernel, B, BEAM_MAX_W, 0, (cudaStream_t)stream, (const unsigned char*)state, beam_layout(W, max_frames),
                  nbest, hyps, hyp_stride, hyp_len, score, acoustic);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

}  // extern "C"
