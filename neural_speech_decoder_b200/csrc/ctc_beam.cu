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
//
// K5d (ctc_word_beam_advance_kernel) is the same body with LEX = true: each slot also carries a pronunciation-lexicon node, a
// word-LM history (h2, h1), a word count and a node of a word trie, all functions of its phoneme prefix, so the merge rule and
// the select carry over unchanged.  In phase 1 one thread per slot stages its lexicon node (128-bit child mask, first child)
// and computes the slot's separator increment (best homophone under the LM, <= W LM lookups per frame); phase 2 admits an
// extension by c != sep only if c is a child, by sep only at a word-final non-root node.  Only a separator changes the prior.
// ctc_word_beam_live_kernel reads a K5d state while it streams: the words every live hypothesis agrees on (committed) and the
// top hypothesis's words past them (tentative).
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

// K5d: K5b's block, then per slot (lexicon node, LM history h2, h1, word count, word-trie node), then the word trie of
// 1 + W*max_frames nodes int2 {parent node, word id}, node 0 = no word.  Header word 3 counts the word-trie nodes.
// b.bytes is the whole utterance block, so the K5b body strides over it unchanged.
struct WordLayout {
    BeamLayout b;
    size_t lex, h2, h1, nw, wnode, wtrie;
};

__host__ __device__ inline WordLayout word_layout(int W, int max_frames) {
    WordLayout L;
    L.b = beam_layout(W, max_frames);
    size_t o = L.b.bytes;
    L.lex = o; o += 4 * (size_t)W;
    L.h2 = o; o += 4 * (size_t)W;
    L.h1 = o; o += 4 * (size_t)W;
    L.nw = o; o += 4 * (size_t)W;
    L.wnode = o; o += 4 * (size_t)W;
    L.wtrie = al16(o);
    L.b.bytes = al16(L.wtrie + 8 * (1 + (size_t)W * max_frames));
    return L;
}

// Lexicon and word LM, read from global memory / L2.
//   lex_nodes int4 x2 per node: {child mask bits 0-31, 32-63, 64-95, 96-127}, {first child, first homophone entry, homophone
//             count, 0}; the children of a node are consecutive, in class order, so child(c) = first + popcount(mask below c).
//   lex_words int2 per homophone entry: {word id, LM id}, ascending word id within a node.
//   lm_idx    NULL (no LM) or b_off[V+1] | b_word[n2] | t_off[n2+1] | t_word[n3]: bigrams (a, w) at b_off[a]..b_off[a+1]
//             sorted by w, trigrams (a, b, w) of bigram j = (a, b) at t_off[j]..t_off[j+1] sorted by w (KenLM-style trie).
//   lm_val    p1[V] | bo1[V] | p2[n2] | bo2[n2] | p3[n3], natural log.
struct WordModel {
    const int4* lex_nodes; const int2* lex_words; const int* lm_idx; const float* lm_val;
    int V, n2, n3, sep; float lm_weight, word_bonus; WordLayout WL;
};

__device__ __forceinline__ int find_sorted(const int* a, int lo, int hi, int key) {
    const int end = hi;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo < end && a[lo] == key ? lo : -1;
}

// lm(w | a, b) with ARPA backoff; a < 0: no second word of history
__device__ float lm_logp(const WordModel& m, int a, int b, int w) {
    const int* b_off = m.lm_idx;
    const int* b_word = b_off + m.V + 1;
    const int* t_off = b_word + m.n2;
    const int* t_word = t_off + m.n2 + 1;
    const float* p1 = m.lm_val;
    const float* bo1 = p1 + m.V;
    const float* p2 = bo1 + m.V;
    const float* bo2 = p2 + m.n2;
    const float* p3 = bo2 + m.n2;
    float bo = 0.f;
    if (a >= 0) {
        const int j = find_sorted(b_word, b_off[a], b_off[a + 1], b);
        if (j >= 0) {
            const int k = find_sorted(t_word, t_off[j], t_off[j + 1], w);
            if (k >= 0) return p3[k];
            bo = bo2[j];
        }
    }
    const int j = find_sorted(b_word, b_off[b], b_off[b + 1], w);
    return bo + (j >= 0 ? p2[j] : bo1[b] + p1[w]);
}

// The word a separator completes at lexicon node rec (homophones at rec[1].y.., count rec[1].z > 0): the best under the LM
// (ties -> smaller word id), or the smallest id without an LM.  Returns the entry; *inc = lm_weight * lm + word_bonus.
__device__ int2 best_homophone(const WordModel& m, int4 rec1, int h2, int h1, float* inc) {
    int2 best = m.lex_words[rec1.y];
    if (m.lm_idx == nullptr) { *inc = m.word_bonus; return best; }
    float bv = lm_logp(m, h2, h1, best.y);
    for (int j = 1; j < rec1.z; ++j) {
        const int2 e = m.lex_words[rec1.y + j];
        const float v = lm_logp(m, h2, h1, e.y);
        if (v > bv) { bv = v; best = e; }
    }
    *inc = fmaf(m.lm_weight, bv, m.word_bonus);
    return best;
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
// LEX: only an extension by sep changes the prior, by the slot's staged increment sep_inc[i].
template <bool LEX>
__device__ __forceinline__ float candidate(const Beam& bm, int i, int r, const float* y, const BeamParams& p, float& opb, float& opnb,
                                           float& oprior, int sep = -1, const float* sep_inc = nullptr) {
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
        if constexpr (LEX) {
            oprior = c == sep ? bm.prior[i] + sep_inc[i] : bm.prior[i];
        } else {
            const int ctx = last >= 0 ? last : p.blank;
            oprior = bm.prior[i] + (p.lm != nullptr ? fmaf(p.alpha, p.lm[ctx * p.C + c], p.beta) : p.beta);
        }
    }
    return lse2(opb, opnb) + oprior;
}

// The word fields of one beam in shared memory (LEX only), beside its Beam.
struct WordSlots {
    int *lex, *h2, *h1, *nw, *wnode;
};

__device__ __forceinline__ WordSlots carve_words(unsigned char* p, int W) {
    WordSlots s;
    s.lex = reinterpret_cast<int*>(p); p += 4 * W;
    s.h2 = reinterpret_cast<int*>(p); p += 4 * W;
    s.h1 = reinterpret_cast<int*>(p); p += 4 * W;
    s.nw = reinterpret_cast<int*>(p); p += 4 * W;
    s.wnode = reinterpret_cast<int*>(p);
    return s;
}
constexpr int WORD_SLOT_SMEM = 4 * 5;
// per slot: two WordSlots, then the staged child mask, first child, separator increment, word id and LM id
constexpr int WORD_STAGE_SMEM = 2 * WORD_SLOT_SMEM + 16 + 4 * 4;

static size_t beam_smem(int W, int C, bool lex) {
    return 2 * 8 * (size_t)W + 2 * (size_t)BEAM_SLOT_SMEM * W + 4 * (size_t)W * (C + 1) + (lex ? (size_t)WORD_STAGE_SMEM * W + 16 : 0);
}

template <bool LEX>
__device__ __forceinline__ void beam_advance_body(const BeamParams& p, const WordModel& wm) {
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

    // LEX: word fields (ping-pong like the beam), the lexicon node and separator staged per slot for the current frame
    WordSlots wbuf[2];
    unsigned int* s_lmask = nullptr;
    int *s_child = nullptr, *s_sepw = nullptr, *s_seplm = nullptr, *s_wsep = nullptr;
    float* s_sepinc = nullptr;
    int2* wtrie = nullptr;
    int wnodes = 0;
    if constexpr (LEX) {
        unsigned char* q = reinterpret_cast<unsigned char*>(ukey + (size_t)W * C1);
        wbuf[0] = carve_words(q, W);
        wbuf[1] = carve_words(q + WORD_SLOT_SMEM * W, W);
        q += 2 * WORD_SLOT_SMEM * W;
        s_lmask = reinterpret_cast<unsigned int*>(q); q += 16 * W;
        s_child = reinterpret_cast<int*>(q); q += 4 * W;
        s_sepinc = reinterpret_cast<float*>(q); q += 4 * W;
        s_sepw = reinterpret_cast<int*>(q); q += 4 * W;
        s_seplm = reinterpret_cast<int*>(q); q += 4 * W;
        s_wsep = reinterpret_cast<int*>(q);
        wtrie = reinterpret_cast<int2*>(g + wm.WL.wtrie);
        wnodes = hdr[3];
    }

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
        if constexpr (LEX) {
            wbuf[0].lex[tid] = reinterpret_cast<const int*>(g + wm.WL.lex)[tid];
            wbuf[0].h2[tid] = reinterpret_cast<const int*>(g + wm.WL.h2)[tid];
            wbuf[0].h1[tid] = reinterpret_cast<const int*>(g + wm.WL.h1)[tid];
            wbuf[0].nw[tid] = reinterpret_cast<const int*>(g + wm.WL.nw)[tid];
            wbuf[0].wnode[tid] = reinterpret_cast<const int*>(g + wm.WL.wnode)[tid];
        }
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
    // frame 0's merge map reads every slot: a resumed beam (size > 1) must be in shared memory first
    __syncthreads();

    int t = 0;
    for (; t < n; ++t) {
        const Beam cur = carve_beam((t & 1) ? beam_buf[1] : beam_buf[0], W);
        const Beam nb = carve_beam((t & 1) ? beam_buf[0] : beam_buf[1], W);
        // ---- 1. row, merge map, cleared counters (LEX: staged lexicon nodes and separators)
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
            if constexpr (LEX) {
                const WordSlots cw = (t & 1) ? wbuf[1] : wbuf[0];
                const int u = cw.lex[tid];
                const int4 r0 = wm.lex_nodes[2 * u], r1 = wm.lex_nodes[2 * u + 1];
                s_lmask[4 * tid] = (unsigned int)r0.x;
                s_lmask[4 * tid + 1] = (unsigned int)r0.y;
                s_lmask[4 * tid + 2] = (unsigned int)r0.z;
                s_lmask[4 * tid + 3] = (unsigned int)r0.w;
                s_child[tid] = r1.x;
                int2 e = make_int2(-1, -1);                // no separator: the root, or not word-final
                float inc = 0.f;
                if (u != 0 && r1.z > 0) e = best_homophone(wm, r1, cw.h2[tid], cw.h1[tid], &inc);
                s_sepw[tid] = e.x;
                s_seplm[tid] = e.y;
                s_sepinc[tid] = inc;
            }
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
            bool ok = r == 0 || (r - 1 != p.blank && !((s_merged[i * 4 + ((r - 1) >> 5)] >> ((r - 1) & 31)) & 1u));
            if constexpr (LEX) {
                if (ok && r > 0) {
                    const int c = r - 1;
                    ok = c == wm.sep ? s_sepw[i] >= 0 : ((s_lmask[i * 4 + (c >> 5)] >> (c & 31)) & 1u) != 0u;
                }
            }
            if (ok) {
                float a0, a1, a2;
                u = order_key(candidate<LEX>(cur, i, r, s_y, p, a0, a1, a2, wm.sep, s_sepinc));
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

        // ---- 4. survivors, their rank, trie nodes for the extensions (LEX: word-trie nodes for the separators)
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
        unsigned int es = 0u;
        if constexpr (LEX) {
            es = __ballot_sync(0xffffffffu, tid < ns && r > 0 && r - 1 == wm.sep);
            if (lane == 0 && warp < BEAM_MAX_W / 32) s_wsep[warp] = __popc(es);
        }
        __syncthreads();
        int off = nodes, n_ext = 0;
#pragma unroll
        for (int w = 0; w < BEAM_MAX_W / 32; ++w) {
            off += w < warp ? s_wext[w] : 0;
            n_ext += s_wext[w];
        }
        int woff = wnodes, n_sep = 0;
        if constexpr (LEX) {
#pragma unroll
            for (int w = 0; w < BEAM_MAX_W / 32; ++w) {
                woff += w < warp ? s_wsep[w] : 0;
                n_sep += s_wsep[w];
            }
        }
        if (nodes + n_ext > cap) {                         // unreachable while frames_done <= max_frames; a backstop
            if (tid == 0 && p.err_flag != nullptr) *p.err_flag = 1;
            break;                                         // (LEX: wnodes <= nodes and n_sep <= n_ext, so the word trie fits)
        }
        if (tid < ns) {
            off += __popc(em & ((1u << lane) - 1u));
            float npb, npnb, nprior;
            candidate<LEX>(cur, i, r, s_y, p, npb, npnb, nprior, wm.sep, s_sepinc);
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
            if constexpr (LEX) {
                const WordSlots cw = (t & 1) ? wbuf[1] : wbuf[0];
                const WordSlots nw = (t & 1) ? wbuf[0] : wbuf[1];
                const int c = r - 1;
                if (r > 0 && c == wm.sep) {                // a word ends: back to the root, the history shifts
                    woff += __popc(es & ((1u << lane) - 1u));
                    nw.lex[tid] = 0;
                    nw.h2[tid] = cw.h1[i];
                    nw.h1[tid] = s_seplm[i];
                    nw.nw[tid] = cw.nw[i] + 1;
                    nw.wnode[tid] = woff;
                    wtrie[woff] = make_int2(cw.wnode[i], s_sepw[i]);
                } else {
                    int u = cw.lex[i];
                    if (r > 0) {                           // child by c: rank of c among the node's children
                        int rank = __popc(s_lmask[4 * i + (c >> 5)] & ((1u << (c & 31)) - 1u));
                        for (int w = 0; w < (c >> 5); ++w) rank += __popc(s_lmask[4 * i + w]);
                        u = s_child[i] + rank;
                    }
                    nw.lex[tid] = u;
                    nw.h2[tid] = cw.h2[i];
                    nw.h1[tid] = cw.h1[i];
                    nw.nw[tid] = cw.nw[i];
                    nw.wnode[tid] = cw.wnode[i];
                }
            }
        }
        nodes += n_ext;
        wnodes += n_sep;
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
        if constexpr (LEX) {
            const WordSlots fw = (t & 1) ? wbuf[1] : wbuf[0];
            reinterpret_cast<int*>(g + wm.WL.lex)[tid] = fw.lex[tid];
            reinterpret_cast<int*>(g + wm.WL.h2)[tid] = fw.h2[tid];
            reinterpret_cast<int*>(g + wm.WL.h1)[tid] = fw.h1[tid];
            reinterpret_cast<int*>(g + wm.WL.nw)[tid] = fw.nw[tid];
            reinterpret_cast<int*>(g + wm.WL.wnode)[tid] = fw.wnode[tid];
        }
    }
    if (tid == 0) {
        hdr[0] = frames_done + t;
        hdr[1] = nodes;
        hdr[2] = size;
        if constexpr (LEX) hdr[3] = wnodes;
    }
}

__global__ void __launch_bounds__(BEAM_THREADS) ctc_beam_advance_kernel(BeamParams p) {
    beam_advance_body<false>(p, WordModel{});
}

__global__ void __launch_bounds__(BEAM_THREADS) ctc_word_beam_advance_kernel(BeamParams p, WordModel wm) {
    beam_advance_body<true>(p, wm);
}

// Utterance block g back to the empty hypothesis (K5b's part).
__device__ __forceinline__ void beam_init_block(unsigned char* g, const BeamLayout& L) {
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

// mask == nullptr: every utterance; otherwise only those with mask[b] != 0 (the others keep every byte)
__global__ void ctc_beam_init_kernel(unsigned char* state, BeamLayout L, const int32_t* mask) {
    pdl_enter();
    if (threadIdx.x != 0 || (mask != nullptr && mask[blockIdx.x] == 0)) return;
    beam_init_block(state + (size_t)blockIdx.x * L.bytes, L);
}

// K5d: K5b's empty hypothesis at the lexicon root with history (-, bos) and no words.
__global__ void ctc_word_beam_init_kernel(unsigned char* state, WordLayout L, int bos, const int32_t* mask) {
    pdl_enter();
    if (threadIdx.x != 0 || (mask != nullptr && mask[blockIdx.x] == 0)) return;
    unsigned char* g = state + (size_t)blockIdx.x * L.b.bytes;
    beam_init_block(g, L.b);
    reinterpret_cast<int*>(g)[3] = 1;
    reinterpret_cast<int*>(g + L.lex)[0] = 0;
    reinterpret_cast<int*>(g + L.h2)[0] = -1;
    reinterpret_cast<int*>(g + L.h1)[0] = bos;
    reinterpret_cast<int*>(g + L.nw)[0] = 0;
    reinterpret_cast<int*>(g + L.wnode)[0] = 0;
    reinterpret_cast<int2*>(g + L.wtrie)[0] = make_int2(-1, -1);
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

// K5d read-out, one CTA of BEAM_MAX_W threads per utterance; thread k owns beam slot k.  final: the end term is added (at the
// root lm_weight * lm(eos | h2, h1); at a word-final node the pending word's separator increment, then lm(eos) after it; at any
// other node the slot is no hypothesis: score and acoustic -inf, lengths 0) and the slots are re-ranked by (total, slot).
// Slots past the beam's size rank last, as in K5b.
__global__ void ctc_word_beam_nbest_kernel(const unsigned char* state, WordModel wm, int eos, int final, int nbest, int64_t* hyps,
                                           int hyp_stride, int32_t* hyp_len, int64_t* words, int word_stride, int32_t* word_len,
                                           float* score, float* acoustic) {
    pdl_enter();
    __shared__ unsigned int s_key[BEAM_MAX_W];
    __shared__ int s_len[BEAM_MAX_W], s_wlen[BEAM_MAX_W];
    const int b = blockIdx.x, k = threadIdx.x;
    const WordLayout& WL = wm.WL;
    const unsigned char* g = state + (size_t)b * WL.b.bytes;
    const int size = reinterpret_cast<const int*>(g)[2];
    float tot = -INFINITY, ac = -INFINITY;
    int2 pend = make_int2(-1, -1);
    bool valid = k < size;
    if (valid) {
        ac = lse2(reinterpret_cast<const float*>(g + WL.b.pb)[k], reinterpret_cast<const float*>(g + WL.b.pnb)[k]);
        tot = ac + reinterpret_cast<const float*>(g + WL.b.prior)[k];
        if (final) {
            const int u = reinterpret_cast<const int*>(g + WL.lex)[k];
            int h2 = reinterpret_cast<const int*>(g + WL.h2)[k], h1 = reinterpret_cast<const int*>(g + WL.h1)[k];
            const int4 r1 = wm.lex_nodes[2 * u + 1];
            if (u != 0 && r1.z > 0) {
                float inc;
                pend = best_homophone(wm, r1, h2, h1, &inc);
                tot += inc;
                h2 = h1;
                h1 = pend.y;
            } else if (u != 0) {
                valid = false;
                tot = ac = -INFINITY;
            }
            if (valid && wm.lm_idx != nullptr) tot += wm.lm_weight * lm_logp(wm, h2, h1, eos);
        }
    }
    s_key[k] = valid ? order_key(tot) : 0u;
    __syncthreads();
    int rank = k;
    if (final) {
        const unsigned int kk = s_key[k];
        rank = 0;
        for (int q = 0; q < BEAM_MAX_W; ++q) rank += s_key[q] > kk || (s_key[q] == kk && q < k);
    }
    int len = 0, wlen = 0;
    if (rank < nbest) {
        const size_t o = (size_t)b * nbest + rank;
        int64_t* out = hyps + o * hyp_stride;
        int64_t* wout = words + o * word_stride;
        if (valid) {
            len = reinterpret_cast<const int*>(g + WL.b.len)[k];
            int node = reinterpret_cast<const int*>(g + WL.b.node)[k];
            const int2* trie = reinterpret_cast<const int2*>(g + WL.b.trie);
            for (int pos = len - 1; pos >= 0; --pos) {
                const int2 e = trie[node];
                out[pos] = e.y;
                node = e.x;
            }
            wlen = reinterpret_cast<const int*>(g + WL.nw)[k];
            node = reinterpret_cast<const int*>(g + WL.wnode)[k];
            const int2* wtrie = reinterpret_cast<const int2*>(g + WL.wtrie);
            for (int pos = wlen - 1; pos >= 0; --pos) {
                const int2 e = wtrie[node];
                wout[pos] = e.y;
                node = e.x;
            }
            if (pend.x >= 0) wout[wlen++] = pend.x;
        }
        score[o] = tot;
        acoustic[o] = ac;
        hyp_len[o] = len;
        word_len[o] = wlen;
        s_len[rank] = len;
        s_wlen[rank] = wlen;
    }
    __syncthreads();
    int64_t* out = hyps + (size_t)b * nbest * hyp_stride;
    for (size_t e = k; e < (size_t)nbest * hyp_stride; e += blockDim.x) {
        const int h = (int)(e / hyp_stride), pos = (int)(e - (size_t)h * hyp_stride);
        if (pos >= s_len[h]) out[e] = -1;
    }
    int64_t* wout = words + (size_t)b * nbest * word_stride;
    for (size_t e = k; e < (size_t)nbest * word_stride; e += blockDim.x) {
        const int h = (int)(e / word_stride), pos = (int)(e - (size_t)h * word_stride);
        if (pos >= s_wlen[h]) wout[e] = -1;
    }
}

constexpr int LIVE_HDR = 4;      // live read-out row: {committed, first, top word count, overflow}, then cap word ids

// K5d live read-out, one CTA of 32 * ceil(W / 32) threads per utterance; thread k owns beam slot k; the state is only read.
// Every later beam extends one of the live slots (finite total), so the longest common prefix of their word sequences is
// final.  Positions below first = reported[b] are already known to agree, so each live slot walks its word trie up to the
// least word count m, then the slots compare one column per step from m down to first: one word trie node for every slot
// means the same words above it and ends the walk; any differing word id moves the prefix end up to that column.  Two
// slots can spell the same words on different nodes (two pronunciations, a prefix dropped and spelled again), so the
// content is compared, and the node test only stops the walk.  The cost is in the words past first, not in the utterance.
__global__ void ctc_word_beam_live_kernel(const unsigned char* state, WordLayout WL, int32_t* reported, int cap, int32_t* out) {
    pdl_enter();
    __shared__ unsigned int s_live[BEAM_MAX_W / 32];
    __shared__ int s_min[BEAM_MAX_W / 32];
    __shared__ int2 s_ref;
    const int b = blockIdx.x, k = threadIdx.x, lane = k & 31, warp = k >> 5, nwarp = blockDim.x >> 5;
    const unsigned char* g = state + (size_t)b * WL.b.bytes;
    const int size = reinterpret_cast<const int*>(g)[2];
    const int* nw_of = reinterpret_cast<const int*>(g + WL.nw);
    const int2* wtrie = reinterpret_cast<const int2*>(g + WL.wtrie);
    const int first = reported[b];
    int32_t* o = out + (size_t)b * (LIVE_HDR + cap);
    bool live = false;
    int nw = 0, node = 0;
    if (k < size) {
        const float tot = lse2(reinterpret_cast<const float*>(g + WL.b.pb)[k], reinterpret_cast<const float*>(g + WL.b.pnb)[k]) +
                          reinterpret_cast<const float*>(g + WL.b.prior)[k];
        live = tot > -INFINITY && tot < INFINITY;
        nw = nw_of[k];
        node = reinterpret_cast<const int*>(g + WL.wnode)[k];
    }
    const unsigned int lb = __ballot_sync(0xffffffffu, live);
    const int wmin = __reduce_min_sync(0xffffffffu, live ? (unsigned int)nw : 0x7fffffffu);
    if (lane == 0) { s_live[warp] = lb; s_min[warp] = wmin; }
    __syncthreads();
    int top = -1, m = 0x7fffffff;                           // top: the best live slot (slot 0: the beam is in rank order)
    for (int w = 0; w < nwarp; ++w) {
        if (top < 0 && s_live[w] != 0u) top = 32 * w + __ffs(s_live[w]) - 1;
        m = min(m, s_min[w]);
    }
    if (top < 0) {                                          // no live slot: nothing new, the counter stays
        if (k == 0) { o[0] = first; o[1] = first; o[2] = first; o[3] = 0; }
        for (int e = k; e < cap; e += blockDim.x) o[LIVE_HDR + e] = -1;
        return;
    }
    const int top_nw = nw_of[top];
    if (k == top) {                                         // the top slot's words first .. top_nw - 1
        int n = node;
        for (int pos = top_nw - 1; pos >= first; --pos) {
            const int2 e = wtrie[n];
            if (pos - first < cap) o[LIVE_HDR + pos - first] = e.y;
            n = e.x;
        }
    }
    for (int e = k; e < cap; e += blockDim.x)
        if (first + e >= top_nw) o[LIVE_HDR + e] = -1;
    if (live)
        for (int d = nw; d > m; --d) node = wtrie[node].x;
    int lcp = m;
    for (int d = m; d > first; --d) {                       // every live slot's node holds d words; its word d - 1 is compared
        const int2 e = live ? wtrie[node] : make_int2(0, 0);
        if (k == top) s_ref = make_int2(node, e.y);
        __syncthreads();
        const int2 r = s_ref;
        if (!__syncthreads_or(live && node != r.x)) break;
        if (__syncthreads_or(live && e.y != r.y)) lcp = d - 1;
        node = e.x;
    }
    lcp = max(lcp, first);                                  // the beam only extends: lcp < first cannot occur
    if (k == 0) {
        o[0] = lcp;
        o[1] = first;
        o[2] = top_nw;
        o[3] = top_nw - first > cap;                        // (lcp <= top_nw: committed words past cap overflow too)
        reported[b] = min(lcp, first + cap);
    }
}

}  // namespace nsd

extern "C" {

size_t nsd_ctc_beam_state_bytes(int B, int W, int max_frames) {
    if (B <= 0 || W <= 0 || max_frames <= 0) return 0;
    return (size_t)B * nsd::beam_layout(W, max_frames).bytes;
}

// need: the state size the caller's layout requires (K5b or K5d)
static int beam_check(int B, int W, int max_frames, size_t state_bytes, size_t (*need)(int, int, int) = nsd_ctc_beam_state_bytes) {
    using namespace nsd;
    NSD_CHECK_ARG(B > 0, "ctc_beam: bad batch %d", B);
    NSD_CHECK_ARG(W >= 1 && W <= BEAM_MAX_W, "ctc_beam: beam width %d outside [1, %d]", W, BEAM_MAX_W);
    NSD_CHECK_ARG(max_frames >= 1 && (long long)W * max_frames < (1ll << 30), "ctc_beam: max_frames=%d out of range for W=%d", max_frames, W);
    if (state_bytes < need(B, W, max_frames)) {
        set_error("ctc_beam: state buffer too small (%zu < %zu bytes)", state_bytes, need(B, W, max_frames));
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
    const size_t smem = beam_smem(W, C, false);
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

// ---- K5d
size_t nsd_ctc_word_beam_state_bytes(int B, int W, int max_frames) {
    if (B <= 0 || W <= 0 || max_frames <= 0) return 0;
    return (size_t)B * nsd::word_layout(W, max_frames).b.bytes;
}

int nsd_ctc_word_beam_init(void* state, size_t state_bytes, int B, int W, int max_frames, int lm_bos, void* stream) {
    using namespace nsd;
    const int st = beam_check(B, W, max_frames, state_bytes, nsd_ctc_word_beam_state_bytes);
    if (st != NSD_OK) return st;
    nsd::launch_k(ctc_word_beam_init_kernel, B, 32, 0, (cudaStream_t)stream, (unsigned char*)state, word_layout(W, max_frames), lm_bos,
                  (const int32_t*)nullptr);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

int nsd_ctc_word_beam_reset(void* state, size_t state_bytes, int B, int W, int max_frames, int lm_bos, const int32_t* mask, void* stream) {
    using namespace nsd;
    const int st = beam_check(B, W, max_frames, state_bytes, nsd_ctc_word_beam_state_bytes);
    if (st != NSD_OK) return st;
    NSD_CHECK_ARG(mask != nullptr, "ctc_word_beam_reset: null mask");
    nsd::launch_k(ctc_word_beam_init_kernel, B, 32, 0, (cudaStream_t)stream, (unsigned char*)state, word_layout(W, max_frames), lm_bos, mask);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

static int word_model(nsd::WordModel& m, const int32_t* lex_nodes, int n_nodes, const int32_t* lex_words, int n_entries,
                      const int32_t* lm_idx, const float* lm_val, int lm_vocab, int lm_n2, int lm_n3, float lm_weight, float word_bonus,
                      int W, int max_frames) {
    using namespace nsd;
    NSD_CHECK_ARG(lex_nodes != nullptr && lex_words != nullptr && n_nodes >= 1 && n_entries >= 0,
                  "ctc_word_beam: bad lexicon (nodes %d, homophone entries %d)", n_nodes, n_entries);
    NSD_CHECK_ARG(((uintptr_t)lex_nodes & 15) == 0 && ((uintptr_t)lex_words & 7) == 0, "ctc_word_beam: lexicon arrays misaligned");
    if (lm_idx != nullptr)
        NSD_CHECK_ARG(lm_val != nullptr && lm_vocab >= 1 && lm_n2 >= 0 && lm_n3 >= 0 && (lm_n3 == 0 || lm_n2 > 0),
                      "ctc_word_beam: bad LM sizes (V=%d, bigrams %d, trigrams %d)", lm_vocab, lm_n2, lm_n3);
    m.lex_nodes = reinterpret_cast<const int4*>(lex_nodes);
    m.lex_words = reinterpret_cast<const int2*>(lex_words);
    m.lm_idx = lm_idx; m.lm_val = lm_val; m.V = lm_vocab; m.n2 = lm_n2; m.n3 = lm_n3;
    m.sep = -1; m.lm_weight = lm_weight; m.word_bonus = word_bonus; m.WL = word_layout(W, max_frames);
    return NSD_OK;
}

int nsd_ctc_word_beam_advance(const float* act, int64_t st, int64_t sb, int64_t sc, int is_logits, const int32_t* lens, int T, int B,
                              int C, int blank, int sep, const int32_t* lex_nodes, int n_nodes, const int32_t* lex_words, int n_entries,
                              const int32_t* lm_idx, const float* lm_val, int lm_vocab, int lm_n2, int lm_n3, float lm_weight,
                              float word_bonus, int W, int max_frames, void* state, size_t state_bytes, int* err_flag, void* stream) {
    using namespace nsd;
    const int s0 = beam_check(B, W, max_frames, state_bytes, nsd_ctc_word_beam_state_bytes);
    if (s0 != NSD_OK) return s0;
    NSD_CHECK_ARG(T >= 0 && C >= 1 && C <= BEAM_MAX_C, "ctc_word_beam: bad sizes T=%d C=%d (C <= %d)", T, C, BEAM_MAX_C);
    NSD_CHECK_ARG(blank >= 0 && blank < C, "ctc_word_beam: blank=%d out of range", blank);
    NSD_CHECK_ARG(sep >= 0 && sep < C && sep != blank, "ctc_word_beam: sep=%d must lie in [0, %d) and differ from blank=%d", sep, C, blank);
    WordModel m;
    const int s1 = word_model(m, lex_nodes, n_nodes, lex_words, n_entries, lm_idx, lm_val, lm_vocab, lm_n2, lm_n3, lm_weight, word_bonus,
                              W, max_frames);
    if (s1 != NSD_OK) return s1;
    m.sep = sep;
    if (T == 0) return NSD_OK;
    BeamParams p;
    p.act = act; p.st = st; p.sb = sb; p.sc = sc; p.is_logits = is_logits; p.lens = lens;
    p.T = T; p.C = C; p.blank = blank; p.lm = nullptr; p.alpha = lm_weight; p.beta = word_bonus;
    p.W = W; p.max_frames = max_frames; p.state = (unsigned char*)state; p.L = m.WL.b; p.err_flag = err_flag;
    const size_t smem = beam_smem(W, C, true);
    if (smem > 48 * 1024) NSD_CUDA(cudaFuncSetAttribute(ctc_word_beam_advance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nsd::launch_k(ctc_word_beam_advance_kernel, B, BEAM_THREADS, smem, (cudaStream_t)stream, p, m);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

int nsd_ctc_word_beam_nbest(const void* state, int B, int W, int max_frames, const int32_t* lex_nodes, int n_nodes,
                            const int32_t* lex_words, int n_entries, const int32_t* lm_idx, const float* lm_val, int lm_vocab, int lm_n2,
                            int lm_n3, int lm_eos, float lm_weight, float word_bonus, int final, int nbest, int64_t* hyps, int hyp_stride,
                            int32_t* hyp_len, int64_t* words, int word_stride, int32_t* word_len, float* score, float* acoustic,
                            void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(B > 0 && W >= 1 && W <= BEAM_MAX_W && max_frames >= 1, "ctc_word_beam_nbest: bad sizes B=%d W=%d max_frames=%d", B, W, max_frames);
    NSD_CHECK_ARG(nbest >= 1 && nbest <= W, "ctc_word_beam_nbest: nbest=%d outside [1, W=%d]", nbest, W);
    NSD_CHECK_ARG(hyp_stride >= max_frames, "ctc_word_beam_nbest: hyp_stride=%d < max_frames=%d", hyp_stride, max_frames);
    NSD_CHECK_ARG(word_stride >= max_frames / 2 + 1, "ctc_word_beam_nbest: word_stride=%d < max_frames / 2 + 1", word_stride);
    NSD_CHECK_ARG(lm_idx == nullptr || (lm_eos >= 0 && lm_eos < lm_vocab), "ctc_word_beam_nbest: eos=%d outside [0, %d)", lm_eos, lm_vocab);
    WordModel m;
    const int s1 = word_model(m, lex_nodes, n_nodes, lex_words, n_entries, lm_idx, lm_val, lm_vocab, lm_n2, lm_n3, lm_weight, word_bonus,
                              W, max_frames);
    if (s1 != NSD_OK) return s1;
    nsd::launch_k(ctc_word_beam_nbest_kernel, B, BEAM_MAX_W, 0, (cudaStream_t)stream, (const unsigned char*)state, m, lm_eos, final, nbest,
                  hyps, hyp_stride, hyp_len, words, word_stride, word_len, score, acoustic);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

int nsd_ctc_word_beam_live(const void* state, int B, int W, int max_frames, int32_t* reported, int cap, int32_t* out, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(B > 0 && W >= 1 && W <= BEAM_MAX_W && max_frames >= 1, "ctc_word_beam_live: bad sizes B=%d W=%d max_frames=%d", B, W, max_frames);
    NSD_CHECK_ARG(cap >= 1, "ctc_word_beam_live: cap=%d must be positive", cap);
    NSD_CHECK_ARG(state != nullptr && reported != nullptr && out != nullptr, "ctc_word_beam_live: null buffer");
    nsd::launch_k(ctc_word_beam_live_kernel, B, 32 * cdiv(W, 32), 0, (cudaStream_t)stream, (const unsigned char*)state,
                  word_layout(W, max_frames), reported, cap, out);
    NSD_LAUNCH_CHECK();
    return NSD_OK;
}

}  // extern "C"
