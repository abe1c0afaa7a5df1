// K3 tensor-core path: persistent GRU recurrence (forward and BPTT) on tcgen05 with the recurrent weights
// STATIONARY IN TENSOR MEMORY (reference nn.GRU, model.py:50-57, 104-119).
//
// One cooperative launch walks all timesteps of one layer, both directions at once.  Measured on B200
// (scratch/umma_ts_bench.cu): one tcgen05.mma (M=128, K=16) costs max(46, N/2) cycles, with the A operand read from
// tensor memory at no extra cost.  So the weights are the A operand (M = gate rows, loaded once into TMEM with
// tcgen05.st), the batch is N, and the only per-step operand traffic is the previous state (B operand, TMA -> smem):
//
//   * forward: a cluster of 4 CTAs owns 64 hidden units of one direction.  CTA j holds in TMEM, for all 64 units x
//     3 gates (two M tiles of 96 rows), the columns of W_hh that multiply ITS QUARTER of h_{t-1} (K split, 16 MMAs per
//     tile per step at H = 1024).  BPTT: a cluster of 4 owns 128 units; CTA j holds W_hh^T[128 units, its quarter of
//     the 3H gate index] (one full M tile, 48 MMAs per step; 16 clusters of 8 CTAs are not co-resident on a B200).
//   * the partial sums D[gate row, batch] meet through distributed shared memory: each epilogue thread owns one TMEM
//     lane (= one gate row), converts its row to bf16 and stages it in the outbox of the CTA that finalises that unit;
//     one cp.async.bulk per peer completes the peer's inbox mbarrier.  Each CTA finalises 16 (BPTT: 32) units: gate math
//     for (batch row, 4 units) per thread and pass, bf16 state stored first and published, fp32 state / saved gates after.
//   * steps are separated by per-cluster ("zone") step counters in global memory (release add / acquire polls).
//   * OPERAND RING: the previous state of a chain arrives as one multi-chunk TMA box into a two-stage shared-memory ring
//     with full / empty mbarriers.  The lanes of the TMA warp poll, in parallel, only the
//     zones that PRODUCE this CTA's K share (plus the CTA's own cluster); one fence, one TMA per stage.  (Tried and
//     rejected, profiles/r02_k3_ring_experiment.log: one TMA per 64-column box issued by its own lane as soon as that
//     box's zone had published -- the zones publish within a few hundred cycles of each other, while a per-lane
//     fence.proxy.async + per-box barrier hand-offs cost 0.5 us per step forward and 2 us per step in the BPTT.)
//   * LATENCY HIDING: independent batch chains are in flight per CTA, each with its own TMEM accumulator and in/outbox, so
//     the barrier + exchange latency of one chain runs under the MMAs and gate math of the others ("Chains in flight" below).
//     B <= 64: two chains of 32 batch rows (UMMA N = 32), one epilogue warpgroup each.  B > 64: FOUR 32-row chains, two per
//     warpgroup (the accumulators beside the stationary weights fill the tensor memory exactly).
//   * The kernels signal griddepcontrol.launch_dependents at their top: a launch placed directly behind them with the
//     programmatic-serialization attribute gets the ~20 SMs the recurrence leaves free (the optimizer update of the
//     previous layer's gradient bucket runs there, elementwise.cu: adam_kernel late_wait).
#include <stdlib.h>

#include "tc_common.cuh"

namespace nsd {
namespace rts {
using namespace nsd::tc;

constexpr int NG = 32;                  // batch rows per epilogue warpgroup pass (one TMEM column block)
constexpr int CTRL_THREADS = 128;       // warp 0: zone polls + TMA, warp 1: MMA issue, warps 2 / 3: publishers of warpgroups 0 / 1 (warp 2 also allocates TMEM)
constexpr int WG_THREADS = 128;         // epilogue warpgroup
constexpr int THREADS = CTRL_THREADS + 2 * WG_THREADS;
constexpr int TMEM_COLS = 512;
constexpr int CNT_STRIDE = 32;          // uint32 slots between two step counters (128 B apart)
constexpr int MAX_STAGES = 2;
constexpr int TRACE_STEPS = 16;

__device__ __forceinline__ float fast_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fast_sigmoid(float x) { return fmaf(0.5f, fast_tanh(0.5f * x), 0.5f); }

__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait_cluster(bar, parity)) return;
    const long long t0 = clock64();
    unsigned int spins = 0;
    while (!mbar_try_wait_cluster(bar, parity)) {
        if ((++spins & 0xFFFFu) == 0 && clock64() - t0 > SPIN_CYCLES) {
            printf("nsd gru_ts: inbox timeout (block %d thread %d)\n", blockIdx.x, threadIdx.x);
            __trap();
        }
    }
}
__device__ __forceinline__ void grid_wait(const unsigned int* counter, unsigned int target) {
    if (ld_acquire_u32(counter) >= target) return;
    const long long t0 = clock64();
    unsigned int spins = 0;
    while (ld_acquire_u32(counter) < target) {
        if ((++spins & 0x3FFFu) == 0 && clock64() - t0 > SPIN_CYCLES) {
            printf("nsd gru_ts: zone barrier timeout (block %d, have %u want %u)\n", blockIdx.x, ld_acquire_u32(counter), target);
            __trap();
        }
    }
}
__device__ __forceinline__ void red_release_add(unsigned int* p) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p) : "memory");
}
// publish hand-off: the 128 epilogue threads of warpgroup w ARRIVE (no wait) once their state stores are issued; the warpgroup's
// publisher warp (control warp 2 + w) syncs on the same barrier and performs the release fence + counter add.  The fence
// (~0.7 us: it waits for the stores' L2 acknowledgements) then stalls an otherwise idle warp instead of warp 0 of the
// warpgroup, which can go on to its deferred stores and -- with two chains per warpgroup -- to the other chain's exchange.
// Two barrier ids alternate per warpgroup, so a thread can never arrive twice on a barrier whose phase is still open.
constexpr int PUB_THREADS = WG_THREADS + 32;
__device__ __forceinline__ void pub_arrive(int w, uint32_t n) { asm volatile("bar.arrive %0, %1;" ::"r"(3 + 2 * w + (int)(n & 1u)), "n"(PUB_THREADS) : "memory"); }
__device__ __forceinline__ void pub_sync(int w, uint32_t n) { asm volatile("bar.sync %0, %1;" ::"r"(3 + 2 * w + (int)(n & 1u)), "n"(PUB_THREADS) : "memory"); }
// "fence done" hand-back (one chain per warpgroup only): the publisher ARRIVES once its release fence + counter add have been issued, the
// epilogue threads SYNC on it before they issue their deferred stores.  MEMBAR.GPU waits for every store the SM has in flight, so deferred
// stores issued between pub_arrive and the publisher's fence (which the early-arriving threads otherwise do) lengthen the critical publish
// by 0.2-0.3 us per step (profiles/r02_k3_bounds.log).  The epilogue threads have nothing else to do until the next step's accumulator.
// With two chains per warpgroup (B > 64) the wait would hold up the other chain's exchange, so it is not used there (measured with
// two 64-row chains per warpgroup: slower in the forward, 12.0 -> 13.1 us).
__device__ __forceinline__ void done_arrive(int w, uint32_t n) { asm volatile("bar.arrive %0, %1;" ::"r"(7 + 2 * w + (int)(n & 1u)), "n"(PUB_THREADS) : "memory"); }
__device__ __forceinline__ void done_sync(int w, uint32_t n) { asm volatile("bar.sync %0, %1;" ::"r"(7 + 2 * w + (int)(n & 1u)), "n"(PUB_THREADS) : "memory"); }
// Chains in flight.  A chain is 32 batch rows (one TMEM accumulator, one message slot); NCH chains of a chain group are in flight
// per CTA, and warpgroup w finalises chains w + 2k, k < NCH / 2.
//   NCH = 2  B <= 64: warpgroup w owns chain w.
//   NCH = 4  B > 64: warpgroup w owns chains w and w + 2 -- the short per-chain critical path of NCH = 2 with twice the rows in
//            flight: the tensor memory (4 accumulators beside the stationary weights) is exactly full.
__device__ __forceinline__ void wg_bar_sync(int w) { asm volatile("bar.sync %0, %1;" ::"r"(1 + w), "n"(WG_THREADS) : "memory"); }

// D[tmem] (+)= A[tmem] * B[smem]: A = stationary weights, lane = row, two bf16 of consecutive k per 32-bit column
__device__ __forceinline__ void umma_ts_bf16(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}

struct Common {
    int Tp, B, H, D, reverse0;
    int nper;                               // CTAs per direction
    int nchain;                             // batch chains of 32 rows
    int ktot, kper;                         // reduction length (H forward, 3H BPTT) and its share per CTA (multiple of 16)
    int s0, row_off;                        // first step with a recurrent term (0 when an initial state is given, else 1); rows the
                                            // exchanged-state tensor is shifted by (B when its first B rows hold the initial state)
    int bps, chunked;                       // boxes per ring stage (two stages; a stage holds a step's whole K share); 1: the K shares are
                                            // whole 64-wide chunks -> one 3-D TMA box per stage
    int cs, upz, nzone;                     // CTAs per cluster, units per zone (= per cluster), zones per direction
    unsigned int* counters;                 // [D][nchain][nzone] step counters, CNT_STRIDE apart: cs arrivals per step
    long long* trace;                       // debug (NSD_GRU_TRACE=1)
};
// Debug stamps go to shared memory (a global store here would sit in front of the next fence) and are dumped at exit.
__device__ __forceinline__ void stamp(const Common& c, long long* tsm, int s, int ev) {
    if (c.trace == nullptr) return;
    if (blockIdx.x == 0 && s < TRACE_STEPS) tsm[s * 8 + ev] = clock64();
    if (s == 8) {                           // every block, one step, global nanosecond timer: skew across CTAs
        unsigned long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        tsm[TRACE_STEPS * 8 + ev] = (long long)g;
    }
}
__device__ __forceinline__ void trace_dump(const Common& c, const long long* tsm) {      // after a __syncthreads
    if (c.trace == nullptr) return;
    for (int i = threadIdx.x; i < 8; i += blockDim.x) c.trace[TRACE_STEPS * 8 + blockIdx.x * 8 + i] = tsm[TRACE_STEPS * 8 + i];
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < TRACE_STEPS * 8; i += blockDim.x) c.trace[i] = tsm[i];
}
__device__ __forceinline__ unsigned int* zone_counter(const Common& c, int d, int chain, int zone) {
    return c.counters + (size_t)((d * c.nchain + chain) * c.nzone + zone) * CNT_STRIDE;
}

// Exchange rows are [gate][unit 0..UU-1][batch 0..31]; the batch index is rotated per unit so that both the row-wise
// writers (lane = unit, 16-byte stores) and the column-wise readers (lane = (batch, unit/4), scalar loads) are
// bank-conflict free.
__device__ __forceinline__ int rot_f32(int u) { return ((4 * ((u >> 2) & 1) + 2 * ((u >> 3) & 1) + 2 * ((u >> 1) & 1) + (u & 1)) & 7) * 4; }
__device__ __forceinline__ int rot_bf16(int u) { return (((u >> 1) & 3) ^ ((u >> 3) & 1)) * 8; }

// Shared memory: [operand ring: 2 stages of bps boxes][inbox: nslot x (CS-1) messages][outbox: same][self: 2 x fp32 rows][barriers]
// nslot = NCH message slots: one per chain in flight.
struct Smem {
    uint8_t* ring; uint8_t* inbox; uint8_t* outbox; float* self;
    uint64_t* full; uint64_t* empty;                               // [MAX_STAGES] each
    uint64_t* tmem_full;                                           // [4] one per chain in flight
    uint64_t* inbox_bar;                                           // [4] one per message slot
    uint32_t* tmem_slot;
    long long* trace;
    float* bsum;                                                   // BPTT: [2 warpgroups][32 values][128 threads] bias-gradient partial sums
};
constexpr int BAR_WORDS = 2 * MAX_STAGES + 4 + 4 + 2;             // uint64 slots in the barrier block
__device__ __forceinline__ Smem carve(uint8_t* raw, int ring_bytes, int nslot, int msgs_bytes, int self_bytes) {
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~uintptr_t(1023));
    Smem s;
    s.ring = base;
    s.inbox = base + ring_bytes;
    s.outbox = s.inbox + nslot * msgs_bytes;
    s.self = reinterpret_cast<float*>(s.outbox + nslot * msgs_bytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s.self) + 2 * self_bytes);
    s.full = bars; s.empty = bars + MAX_STAGES; s.tmem_full = bars + 2 * MAX_STAGES; s.inbox_bar = bars + 2 * MAX_STAGES + 4;
    s.tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 8);
    s.trace = reinterpret_cast<long long*>(bars + BAR_WORDS);
    s.bsum = reinterpret_cast<float*>(s.trace + (TRACE_STEPS + 1) * 8);
    return s;
}
static size_t smem_bytes(int ring_bytes, int nslot, int msgs_bytes, int self_bytes, size_t extra = 0) {
    return extra + (size_t)ring_bytes + 2 * (size_t)nslot * msgs_bytes + 2 * (size_t)self_bytes + BAR_WORDS * 8 + (TRACE_STEPS + 1) * 64 + 1024 + 64;
}

__device__ __forceinline__ uint32_t setup(const Smem& sm, int warp, int lane) {
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < MAX_STAGES; ++i) { mbar_init(&sm.full[i], 1); mbar_init(&sm.empty[i], 1); }
        for (int i = 0; i < 4; ++i) mbar_init(&sm.tmem_full[i], 1);
        for (int i = 0; i < 4; ++i) mbar_init(&sm.inbox_bar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sm.tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    __syncwarp();
    cluster_sync_all();                 // every CTA's barriers exist before any peer pushes into its inbox
    tcgen05_fence_after();
    return *sm.tmem_slot;
}
__device__ __forceinline__ void teardown(int warp, uint32_t tmem_base, const Common& c, const Smem& sm) {
    tcgen05_fence_before();
    __syncthreads();
    trace_dump(c, sm.trace);
    __syncwarp();
    cluster_sync_all();                 // nobody leaves while a peer may still push into its shared memory
    if (warp == 2) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

// One row of the stationary operand into this thread's TMEM lane: k in [k_lo, k_lo + 2*kc) of `src_row` (nullptr or
// beyond k_hi -> zeros), columns [col0, col0 + kc), 8 columns (= 16 bf16 = 32 bytes) per step, steps c0 = first, first+stride, ..
__device__ __forceinline__ void load_a_row(uint32_t taddr_row, const __nv_bfloat16* src_row, int k_lo, int k_hi, int kc, int first, int stride) {
    for (int c0 = first * 8; c0 < kc; c0 += stride * 8) {
        uint32_t v[8];
        if (src_row != nullptr && k_lo + 2 * c0 < k_hi) {
            const uint4 a = __ldg(reinterpret_cast<const uint4*>(src_row + k_lo + 2 * c0));
            const uint4 b = __ldg(reinterpret_cast<const uint4*>(src_row + k_lo + 2 * c0 + 8));
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = 0u;
        }
        tmem_st_32x8(taddr_row + (uint32_t)c0, v);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// Control warps of both kernels.  Item (s, ch): step s >= s0 of the chain `ch` of the current chain group consumes the rows
// the direction produced in step s-1 of that chain: nbox boxes of 64 columns, loaded into one ring stage.
//   warp 0: lane i < nbox polls the zone(s) that produce box i (a 64-wide box touches at most two); lane 31 polls this
//     CTA's own cluster: once it has published step s-1 of the chain, my MMAs and epilogue of that step are finished and my
//     peers have drained their inboxes, so the chain's TMEM accumulator and message buffers are free.  Then lane 0 fences
//     once and issues the stage.  A CTA without a K share still paces its epilogue with an empty stage.
//   warp 1: waits for each stage in order and issues its MMAs; a tcgen05.commit per item wakes the chain's epilogue (and,
//     with four chains, frees the stage).
// Control warps 2 and 3: publisher of warpgroup w = warp - 2.  Walks the (chain group, step, chain) items in the order the
// warpgroup finalises them.
template <int NCH>
__device__ __forceinline__ void publisher_warp(const Smem& sm, const Common& c, int d, int my_zone, int w, int lane) {
    const int npair = (c.nchain + NCH - 1) / NCH;
    uint32_t n = 0;
    for (int pr = 0; pr < npair; ++pr)
        for (int s = 0; s < c.Tp; ++s)
            for (int k = 0; k < NCH / 2; ++k) {
                const int chain = NCH * pr + w + 2 * k;
                if (chain >= c.nchain) continue;
                pub_sync(w, n);
                if (lane == 0) {
                    red_release_add(zone_counter(c, d, chain, my_zone));
                    if (chain == 0 && w == 0) stamp(c, sm.trace, s, 7);
                }
                __syncwarp();
                if (NCH == 2) done_arrive(w, n);
                ++n;
            }
}

template <int NT, int NCH>
__device__ __forceinline__ void control_warps(const Smem& sm, const CUtensorMap* tmB, const CUtensorMap* tmB3, int warp, int lane, uint32_t tmem_base,
                                              const Common& c, int d, int my_zone, int k_lo, int k_hi, int nslab, int nbox,
                                              int b_col0, bool bptt) {
    constexpr int BOXB = NG * 128;
    constexpr uint32_t A_COL0 = NCH * NT * NG;
    constexpr bool HANDSHAKE = NCH > 2;              // the ring stage an item reuses was last read by ANOTHER chain's MMAs: explicit empty wait
    const bool rev = (d == 1) || (c.reverse0 != 0);
    const int kc = c.kper / 2;
    const size_t stage_bytes = (size_t)c.bps * BOXB;
    const int npair = (c.nchain + NCH - 1) / NCH;
    if (warp == 0) {
        int z0 = my_zone, z1 = my_zone;
        if (lane < nbox) {
            const int c0 = k_lo + lane * BK, c1 = min(c0 + BK, k_hi) - 1;
            z0 = (c0 % c.H) / c.upz; z1 = (c1 % c.H) / c.upz;
        }
        const bool poller = lane < nbox || lane == 31;
        uint32_t seq = 0;
        for (int pr = 0; pr < npair; ++pr) {
            for (int s = c.s0; s < c.Tp; ++s) {
                int t_src;
                if (!bptt) { const int t = rev ? (c.Tp - 1 - s) : s; t_src = rev ? t + 1 : t - 1; }
                else { const int t = rev ? s : (c.Tp - 1 - s); t_src = rev ? t - 1 : t + 1; }
                for (int ch = 0; ch < NCH && NCH * pr + ch < c.nchain; ++ch) {
                    const int chain = NCH * pr + ch;
                    const unsigned int want = (unsigned int)(s * c.cs);
                    if (poller) {
                        grid_wait(zone_counter(c, d, chain, z0), want);
                        if (z1 != z0) grid_wait(zone_counter(c, d, chain, z1), want);
                    }
                    __syncwarp();
                    if (lane == 0 && chain == 0) stamp(c, sm.trace, s, 0);
                    if (lane == 0) asm volatile("fence.proxy.async.global;" ::: "memory");      // generic-proxy writes (acquired above) -> TMA reads
                    const int row = t_src * c.B + chain * NG + c.row_off;
                    const uint32_t stage = seq & 1u, use = seq >> 1;
                    ++seq;
                    if (HANDSHAKE) {
                        // wait until the MMAs that read this stage last have completed.  (With two chains the stage was last read by
                        // an earlier step of this chain, which the own-cluster wait above already shows finished.)
                        if (lane == 0) mbar_wait(&sm.empty[stage], (use & 1u) ^ 1u);
                        __syncwarp();
                    }
                    uint8_t* dst = sm.ring + stage * stage_bytes;
                    if (nbox == 0) {
                        if (lane == 0) mbar_arrive(&sm.full[stage]);
                    } else if (c.chunked) {
                        // K share aligned to 64-wide chunks: the whole stage (nbox swizzled tiles) in one TMA instruction
                        if (lane == 0) {
                            mbar_expect_tx(&sm.full[stage], (uint32_t)(nbox * BOXB));
                            tma_load_3d(tmB3, &sm.full[stage], dst, 0, row, (b_col0 + k_lo) / BK);
                        }
                    } else {
                        if (lane == 0) mbar_expect_tx(&sm.full[stage], (uint32_t)(nbox * BOXB));
                        __syncwarp();
                        if (lane < nbox) tma_load_2d(tmB, &sm.full[stage], dst + (size_t)lane * BOXB, b_col0 + k_lo + lane * BK, row);
                    }
                    if (lane == 0 && chain == 0) stamp(c, sm.trace, s, 1);
                }
            }
        }
    } else if (warp == 1) {
        // The whole warp walks the items; one elected lane issues the MMAs (the compiler then keeps the operands in
        // uniform registers instead of emitting a per-instruction R2UR waterfall, which made the issue rate the bound).
        constexpr uint32_t idesc = make_idesc_bf16(128, NG);
        uint32_t seq = 0;
        for (int pr = 0; pr < npair; ++pr) {
            for (int s = c.s0; s < c.Tp; ++s) {
                for (int ch = 0; ch < NCH && NCH * pr + ch < c.nchain; ++ch) {
                    const uint32_t stage = seq & 1u, use = seq >> 1;
                    ++seq;
                    mbar_wait(&sm.full[stage], use & 1u);
                    if (lane == 0 && NCH * pr + ch == 0) stamp(c, sm.trace, s, 2);
                    tcgen05_fence_after();
                    if (elect_one()) {
                        if (nslab > 0) {
#pragma unroll
                            for (int t = 0; t < NT; ++t) {
                                const uint32_t dcol = tmem_base + (uint32_t)((ch * NT + t) * NG);
                                uint32_t acol = tmem_base + A_COL0 + (uint32_t)(t * kc);
                                uint64_t bdesc = make_kmajor_sw128_desc(smem_u32(sm.ring + stage * stage_bytes));
                                for (int sl = 0; sl < nslab; sl += 4, acol += 32u, bdesc += (uint64_t)(BOXB >> 4)) {   // one box = 4 slabs
                                    const int ns = nslab - sl;
                                    umma_ts_bf16(dcol, acol, bdesc, idesc, sl != 0);
                                    if (ns > 1) umma_ts_bf16(dcol, acol + 8u, bdesc + 2u, idesc, 1u);
                                    if (ns > 2) umma_ts_bf16(dcol, acol + 16u, bdesc + 4u, idesc, 1u);
                                    if (ns > 3) umma_ts_bf16(dcol, acol + 24u, bdesc + 6u, idesc, 1u);
                                }
                            }
                            if (HANDSHAKE) umma_commit(&sm.empty[stage]);
                            umma_commit(&sm.tmem_full[ch]);
                        } else {
                            if (HANDSHAKE) mbar_arrive(&sm.empty[stage]);
                            mbar_arrive(&sm.tmem_full[ch]);
                        }
                    }
                    __syncwarp();
                    if (lane == 0 && NCH * pr + ch == 0) stamp(c, sm.trace, s, 3);
                }
            }
        }
    } else {
        publisher_warp<NCH>(sm, c, d, my_zone, warp - 2, lane);
    }
}

__device__ __forceinline__ void ld4g(const float* p, float (&v)[4]) {    // read-only for the whole launch
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
}
__device__ __forceinline__ void st4(float* p, const float (&v)[4]) { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&a);
}
__device__ __forceinline__ void st4_bf16(__nv_bfloat16* p, const float (&v)[4]) {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]));
}

// Phase A of the exchange: this thread's TMEM lane of accumulator tile `taddr` is gate row (gate, cluster unit ul) with
// 32 batch columns.  The CTA that finalises unit ul is rank ul / UU: keep the row (fp32) if that is me, else stage it as
// bf16 in the outbox slot of that peer (slot = (peer - me - 1) mod CS).
template <int CS, int NGATE, int UU>
__device__ __forceinline__ void stage_row(uint32_t taddr, bool have, int gate, int ul, int me, float* self, uint8_t* outbox) {
    uint32_t raw[32];
    if (have) {
        tmem_ld_32x32(taddr, raw);
    } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) raw[i] = 0u;
    }
    const int owner = ul / UU, uo = ul % UU;
    if (owner == me) {
        float* dst = self + (gate * UU + uo) * NG;
        const int rot = rot_f32(uo);
#pragma unroll
        for (int cq = 0; cq < 8; ++cq)
            *reinterpret_cast<uint4*>(dst + ((4 * cq + rot) & (NG - 1))) = make_uint4(raw[4 * cq], raw[4 * cq + 1], raw[4 * cq + 2], raw[4 * cq + 3]);
    } else if (owner < CS) {
        const int slot = (owner - me - 1 + CS) % CS;
        __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(outbox) + ((slot * NGATE + gate) * UU + uo) * NG;
        const int rot = rot_bf16(uo);
#pragma unroll
        for (int cq = 0; cq < 4; ++cq) {
            uint4 u;
            u.x = pack_bf16(__uint_as_float(raw[8 * cq]), __uint_as_float(raw[8 * cq + 1]));
            u.y = pack_bf16(__uint_as_float(raw[8 * cq + 2]), __uint_as_float(raw[8 * cq + 3]));
            u.z = pack_bf16(__uint_as_float(raw[8 * cq + 4]), __uint_as_float(raw[8 * cq + 5]));
            u.w = pack_bf16(__uint_as_float(raw[8 * cq + 6]), __uint_as_float(raw[8 * cq + 7]));
            *reinterpret_cast<uint4*>(dst + ((8 * cq + rot) & (NG - 1))) = u;
        }
    }
}
// One bulk shared->distributed-shared copy per peer: my outbox slot for peer p lands in p's inbox slot for me
// ((me - p - 1) mod CS) and completes p's inbox mbarrier with the byte count.  Thread i < CS-1 serves peer (me+1+i) mod CS.
template <int CS, int NGATE, int UU>
__device__ __forceinline__ void send_message(uint8_t* outbox, uint8_t* inbox, uint64_t* inbox_bar, int me, int i) {
    constexpr uint32_t MSG = NGATE * UU * NG * 2;
    const int p = (me + 1 + i) % CS;
    const int out_slot = i, in_slot = (me - p - 1 + CS) % CS;
    const uint32_t src = smem_u32(outbox + (size_t)out_slot * MSG);
    const uint32_t dst = map_to_cta(smem_u32(inbox + (size_t)in_slot * MSG), (uint32_t)p);
    const uint32_t bar = map_to_cta(smem_u32(inbox_bar), (uint32_t)p);
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "r"(src), "r"(MSG), "r"(bar) : "memory");
}
// Phase B: sum of my fp32 partial and the CS-1 bf16 partials for (gate, units u0 .. u0+3, batch row bl)
template <int CS, int NGATE, int UU>
__device__ __forceinline__ void gather(const float* self, const uint8_t* inbox, int gate, int u0, int bl, float (&acc)[4]) {
    const __nv_bfloat16* in = reinterpret_cast<const __nv_bfloat16*>(inbox);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int u = u0 + i;
        float a = self[(gate * UU + u) * NG + ((bl + rot_f32(u)) & (NG - 1))];
        const int cb = (bl + rot_bf16(u)) & (NG - 1);
#pragma unroll
        for (int slot = 0; slot < CS - 1; ++slot) a += __bfloat162float(in[((slot * NGATE + gate) * UU + u) * NG + cb]);
        acc[i] = a;
    }
}

// =============================================================================================== forward
struct FwdParams {
    Common c;
    const __nv_bfloat16* w;               // [D*3H, H] bf16 W_hh, gate rows r | z | n per direction
    const float* gi; int ldgi;            // [Tp*B, D*3H] = x W_ih^T + b_ih
    const float* b_hh;                    // [D*3H]
    float* hseq; __nv_bfloat16* hseq_bf; int ldh;    // [Tp*B, D*H]; the bf16 copy is what the other CTAs TMA-load
    float* r; float* z; float* n; float* hn;         // [D][Tp*B][H] or null
    const float* h0;                                 // [B, ldh] initial state (fp32) or null; its bf16 copy = first B rows of hseq_bf
    __nv_bfloat16* hdrop; uint32_t drop_thresh; float inv_keep; uint64_t seed;   // fused inter-layer dropout output (or null)
};

template <int NCH>
__global__ void __launch_bounds__(THREADS, 1)
gru_fwd_ts_kernel(const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmH3, const FwdParams p) {
    // a kernel launched behind this one with the programmatic-serialization attribute may take the ~20 SMs the recurrence leaves free
    // once all of its CTAs are resident (the optimizer of the previous layer's bucket does, elementwise.cu: adam_kernel late_wait)
    pdl_launch_dependents();
    constexpr int CS = 4, NT = 2, NGATE = 3, U = 16, CPW = NCH / 2;
    constexpr int MSG = NGATE * U * NG * 2, MSGS = (CS - 1) * MSG, SELF = NGATE * U * NG * 4;
    constexpr uint32_t A_COL0 = NCH * NT * NG;
    extern __shared__ uint8_t smem_raw[];
    const Common& c = p.c;
    const int H = c.H, B = c.B;
    const int me = (int)cluster_rank();
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int d = blockIdx.x / c.nper;
    const int my_zone = (blockIdx.x - d * c.nper) / CS;
    const int uc0 = my_zone * (CS * U);                                  // first unit of the cluster
    const bool rev = (d == 1) || (c.reverse0 != 0);
    const int k_lo = min(me * c.kper, c.ktot), k_hi = min(k_lo + c.kper, c.ktot);
    const int nslab = (k_hi - k_lo) / UMMA_K, nbox = (k_hi - k_lo + BK - 1) / BK;
    const int kc = c.kper / 2;
    const Smem sm = carve(smem_raw, 2 * c.bps * NG * 128, NCH, MSGS, SELF);
    if (c.trace != nullptr)
        for (int i = threadIdx.x; i < (TRACE_STEPS + 1) * 8; i += blockDim.x) sm.trace[i] = 0;
    const uint32_t tmem_base = setup(sm, warp, lane);

    if (warp >= 4) {
        // stationary weights: tile t = units uc0 + 32t .. +32, lanes [r | z | n | unused] x 32 units, my quarter of K
        const int e = warp - 4, w4 = e & 3, t = e >> 2;
        const int unit = uc0 + 32 * t + lane;
        const __nv_bfloat16* row = (w4 < 3 && unit < H) ? p.w + (size_t)(d * 3 * H + w4 * H + unit) * H : nullptr;
        load_a_row(tmem_base + ((uint32_t)(w4 * 32) << 16) + A_COL0 + (uint32_t)(t * kc), row, k_lo, k_hi, kc, 0, 1);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();

    if (warp < 4) {
        control_warps<NT, NCH>(sm, &tmH, &tmH3, warp, lane, tmem_base, c, d, my_zone, k_lo, k_hi, nslab, nbox, d * H, false);
    } else {
        // ------------------------------------------------------------ epilogue warpgroup w: chains w + 2k of every chain group
        const int e = warp - 4, w4 = e & 3, w = e >> 2, te = w4 * 32 + lane;
        const int bl = te >> 2, uo4 = te & 3;
        const int ub = uc0 + me * U + 4 * uo4;             // first of this thread's 4 units
        float* self = sm.self + w * (SELF / 4);
        float bh[3][4];
#pragma unroll
        for (int g = 0; g < 3; ++g) ld4g(p.b_hh + d * 3 * H + g * H + ub, bh[g]);
        uint32_t it[CPW], npub = 0;
#pragma unroll
        for (int k = 0; k < CPW; ++k) it[k] = 0;
        const int npair = (c.nchain + NCH - 1) / NCH;
        for (int pr = 0; pr < npair; ++pr) {
            float k_h[CPW][4];                             // h_{t-1} of this thread's (row, 4 units) per chain, fp32, in registers
#pragma unroll
            for (int k = 0; k < CPW; ++k) {
                const int ch = w + 2 * k;
                const int b = (NCH * pr + ch) * NG + bl;
#pragma unroll
                for (int i = 0; i < 4; ++i) k_h[k][i] = 0.f;
                if (p.h0 != nullptr && NCH * pr + ch < c.nchain && b < B) ld4g(p.h0 + (size_t)b * p.ldh + d * H + ub, k_h[k]);
            }
            for (int s = 0; s < c.Tp; ++s) {
                const int t = rev ? (c.Tp - 1 - s) : s;
#pragma unroll
                for (int k = 0; k < CPW; ++k) {
                    const int ch = w + 2 * k;
                    const int chain = NCH * pr + ch;
                    if (chain >= c.nchain) continue;
                    uint8_t* inbox = sm.inbox + ch * MSGS;
                    uint8_t* outbox = sm.outbox + ch * MSGS;
                    const int b = chain * NG + bl;
                    const bool row_ok = b < B;
                    const size_t m = (size_t)t * B + b;
                    float gi[3][4];
                    if (row_ok) {
#pragma unroll
                        for (int g = 0; g < 3; ++g) {
                            ld4g(p.gi + m * p.ldgi + d * 3 * H + g * H + ub, gi[g]);
                            if (g < 2) {
#pragma unroll
                                for (int i = 0; i < 4; ++i) gi[g][i] += bh[g][i];
                            }
                        }
                    }
                    float acc[3][4];
#pragma unroll
                    for (int g = 0; g < 3; ++g)
#pragma unroll
                        for (int i = 0; i < 4; ++i) acc[g][i] = 0.f;
                    if (s >= c.s0) {
                        if (te == 0) mbar_expect_tx(&sm.inbox_bar[ch], (uint32_t)MSGS);
                        mbar_wait(&sm.tmem_full[ch], it[k] & 1);
                        tcgen05_fence_after();
                        if (te == 0 && chain == 0 && w == 0) stamp(c, sm.trace, s, 4);
                        if (w4 < 3) {
#pragma unroll
                            for (int t2 = 0; t2 < NT; ++t2)
                                stage_row<CS, NGATE, U>(tmem_base + ((uint32_t)(w4 * 32) << 16) + (uint32_t)((ch * NT + t2) * NG),
                                                        nslab > 0, w4, 32 * t2 + lane, me, self, outbox);
                        }
                        tcgen05_fence_before();
                        fence_proxy_async_smem();
                        wg_bar_sync(w);
                        if (te < CS - 1) send_message<CS, NGATE, U>(outbox, inbox, &sm.inbox_bar[ch], me, te);
                        mbar_wait_cluster(&sm.inbox_bar[ch], it[k] & 1);
                        if (te == 0 && chain == 0 && w == 0) stamp(c, sm.trace, s, 5);
#pragma unroll
                        for (int g = 0; g < 3; ++g) gather<CS, NGATE, U>(self, inbox, g, 4 * uo4, bl, acc[g]);
                        ++it[k];
                    }
                    float rr[4], zz[4], nn[4], gn[4];
                    if (row_ok) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            rr[i] = fast_sigmoid(gi[0][i] + acc[0][i]);
                            zz[i] = fast_sigmoid(gi[1][i] + acc[1][i]);
                            gn[i] = acc[2][i] + bh[2][i];
                            nn[i] = fast_tanh(fmaf(rr[i], gn[i], gi[2][i]));
                            k_h[k][i] = fmaf(zz[i], k_h[k][i] - nn[i], nn[i]);        // (1-z)*n + z*h_prev
                        }
                        // the bf16 state is what the other CTAs wait for: store it first, publish, then write the rest
                        st4_bf16(p.hseq_bf + (m + c.row_off) * p.ldh + d * H + ub, k_h[k]);
                    }
                    if (te == 0 && chain == 0 && w == 0) stamp(c, sm.trace, s, 6);
                    pub_arrive(w, npub);                         // the publisher warp releases the counter (the consumer fences generic->async proxy after its acquire)
                    if (CPW == 1) done_sync(w, npub);            // deferred stores only after the publisher's fence has been issued
                    ++npub;
                    if (CPW > 1) wg_bar_sync(w);                 // the other chain's stage_row reuses `self`: every thread's gather must be done
                    if (row_ok) {                                // off the critical path: nobody else reads these during the launch
                        st4(p.hseq + m * p.ldh + d * H + ub, k_h[k]);
                        if (p.r) {
                            const size_t o = ((size_t)d * c.Tp * B + m) * H + ub;
                            st4(p.r + o, rr); st4(p.z + o, zz); st4(p.n + o, nn); st4(p.hn + o, gn);
                        }
                        if (p.hdrop) {                           // same mask and rounding as nsd_dropout on the bf16 [Tp*B, ldh] tensor
                            const size_t el = m * p.ldh + d * H + ub;
                            const uint4 bits = dropout_bits(el >> 2, p.seed);
                            const uint32_t bw[4] = {bits.x, bits.y, bits.z, bits.w};
                            float o[4];
#pragma unroll
                            for (int i = 0; i < 4; ++i)
                                o[i] = bw[i] >= p.drop_thresh ? __bfloat162float(__float2bfloat16_rn(k_h[k][i])) * p.inv_keep : 0.f;
                            st4_bf16(p.hdrop + el, o);
                        }
                    }
                }
            }
        }
    }
    teardown(warp, tmem_base, c, sm);
}

// =============================================================================================== BPTT
struct BwdParams {
    Common c;
    const __nv_bfloat16* wT;              // [D*H, 3H] bf16 transpose of W_hh per direction
    const float* dhseq; int lddh;         // [Tp*B, D*H] gradient w.r.t. every emitted h_t
    const float* hseq; int ldh;           // forward hidden states (f32)
    const float* r; const float* z; const float* n; const float* hn;   // [D][Tp*B][H]
    __nv_bfloat16* dgi; __nv_bfloat16* dgh; int ldg;    // [Tp*B, D*3H]: [dr~,dz~,dn~] and [dr~,dz~,dn~*r]
    uint32_t drop_thresh; float inv_keep; uint64_t seed;   // dropout mask of this layer's output, applied to dhseq (thresh 0 = none)
    float* db_ih; float* db_hh;                          // [D*3H] column sums of dgi / dgh over all rows (or null), pre-zeroed
};

template <int NCH>
__global__ void __launch_bounds__(THREADS, 1)
gru_bwd_ts_kernel(const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmG3, const BwdParams p) {
    // a kernel launched behind this one with the programmatic-serialization attribute may take the ~20 SMs the recurrence leaves free
    // once all of its CTAs are resident (the optimizer of the previous layer's bucket does, elementwise.cu: adam_kernel late_wait)
    pdl_launch_dependents();
    constexpr int CS = 4, NT = 1, NGATE = 1, U = 32, NP = U / 16, CPW = NCH / 2;       // NP passes of (batch row, 4 units) per thread
    constexpr int MSG = NGATE * U * NG * 2, MSGS = (CS - 1) * MSG, SELF = NGATE * U * NG * 4;
    constexpr uint32_t A_COL0 = NCH * NT * NG;
    extern __shared__ uint8_t smem_raw[];
    const Common& c = p.c;
    const int H = c.H, B = c.B;
    const int me = (int)cluster_rank();
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int d = blockIdx.x / c.nper;
    const int my_zone = (blockIdx.x - d * c.nper) / CS;
    const int uc0 = my_zone * (CS * U);
    const bool rev = (d == 1) || (c.reverse0 != 0);
    const int k_lo = min(me * c.kper, c.ktot), k_hi = min(k_lo + c.kper, c.ktot);
    const int nslab = (k_hi - k_lo) / UMMA_K, nbox = (k_hi - k_lo + BK - 1) / BK;
    const int kc = c.kper / 2;
    const Smem sm = carve(smem_raw, 2 * c.bps * NG * 128, NCH, MSGS, SELF);
    if (c.trace != nullptr)
        for (int i = threadIdx.x; i < (TRACE_STEPS + 1) * 8; i += blockDim.x) sm.trace[i] = 0;
    const uint32_t tmem_base = setup(sm, warp, lane);

    if (warp >= 4) {
        // stationary weights: lane = unit uc0 + lane of W_hh^T [H, 3H], my quarter of the gate index; the two warpgroups
        // interleave the column chunks
        const int e = warp - 4, w4 = e & 3, half = e >> 2;
        const int unit = uc0 + w4 * 32 + lane;
        const __nv_bfloat16* row = unit < H ? p.wT + (size_t)(d * H + unit) * (3 * H) : nullptr;
        load_a_row(tmem_base + ((uint32_t)(w4 * 32) << 16) + A_COL0, row, k_lo, k_hi, kc, half, 2);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();

    if (warp < 4) {
        control_warps<NT, NCH>(sm, &tmG, &tmG3, warp, lane, tmem_base, c, d, my_zone, k_lo, k_hi, nslab, nbox, d * 3 * H, true);
    } else {
        const int e = warp - 4, w4 = e & 3, w = e >> 2, te = w4 * 32 + lane;
        const int bl = te >> 2, uo4 = te & 3;
        const int ub0 = uc0 + me * U + 4 * uo4;             // pass q handles units ub0 + 16q .. +3
        float* self = sm.self + w * (SELF / 4);
        float* bsum = sm.bsum + (size_t)w * 16 * NP * WG_THREADS + te;
        if (p.db_ih)
            for (int v = 0; v < 16 * NP; ++v) bsum[v * WG_THREADS] = 0.f;
        uint32_t it[CPW], npub = 0;
#pragma unroll
        for (int k = 0; k < CPW; ++k) it[k] = 0;
        const int npair = (c.nchain + NCH - 1) / NCH;
        for (int pr = 0; pr < npair; ++pr) {
            float cr[CPW][NP][4];                            // dh_t * z_t carried to the next step, in registers
#pragma unroll
            for (int k = 0; k < CPW; ++k)
#pragma unroll
                for (int q = 0; q < NP; ++q)
#pragma unroll
                    for (int i = 0; i < 4; ++i) cr[k][q][i] = 0.f;
            for (int s = 0; s < c.Tp; ++s) {
                const int t = rev ? s : (c.Tp - 1 - s);              // BPTT visits time in the opposite order of the forward pass
                const int tprev = rev ? t + 1 : t - 1;               // forward-time predecessor (source of h_{t-1})
                const bool has_prev = rev ? (t + 1 < c.Tp) : (t > 0);
#pragma unroll
                for (int k = 0; k < CPW; ++k) {
                    const int ch = w + 2 * k;
                    const int chain = NCH * pr + ch;
                    if (chain >= c.nchain) continue;
                    uint8_t* inbox = sm.inbox + ch * MSGS;
                    uint8_t* outbox = sm.outbox + ch * MSGS;
                    const int b = chain * NG + bl;
                    const size_t m = (size_t)t * B + b;
                    float dh[NP][4], rr[NP][4], zz[NP][4], nn[NP][4], gn[NP][4], hp[NP][4];
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        const int ub = ub0 + 16 * q;
#pragma unroll
                        for (int i = 0; i < 4; ++i) hp[q][i] = 0.f;
                        if (b < B && ub < H) {                   // H % 64 == 0: a pass's 16 units are all inside or all outside
                            const size_t o = ((size_t)d * c.Tp * B + m) * H + ub;
                            ld4g(p.dhseq + m * p.lddh + d * H + ub, dh[q]);
                            if (p.drop_thresh != 0u) {           // gradient through this layer's output dropout (mask of nsd_dropout)
                                const uint4 bits = dropout_bits((m * p.lddh + d * H + ub) >> 2, p.seed);
                                const uint32_t bw[4] = {bits.x, bits.y, bits.z, bits.w};
#pragma unroll
                                for (int i = 0; i < 4; ++i) dh[q][i] = bw[i] >= p.drop_thresh ? dh[q][i] * p.inv_keep : 0.f;
                            }
                            ld4g(p.r + o, rr[q]); ld4g(p.z + o, zz[q]); ld4g(p.n + o, nn[q]); ld4g(p.hn + o, gn[q]);
                            if (has_prev) ld4g(p.hseq + ((size_t)tprev * B + b) * p.ldh + d * H + ub, hp[q]);
                        }
                    }
                    float acc[NP][4];
#pragma unroll
                    for (int q = 0; q < NP; ++q)
#pragma unroll
                        for (int i = 0; i < 4; ++i) acc[q][i] = 0.f;
                    if (s > 0) {
                        if (te == 0) mbar_expect_tx(&sm.inbox_bar[ch], (uint32_t)MSGS);
                        mbar_wait(&sm.tmem_full[ch], it[k] & 1);
                        tcgen05_fence_after();
                        if (te == 0 && chain == 0 && w == 0) stamp(c, sm.trace, s, 4);
                        stage_row<CS, NGATE, U>(tmem_base + ((uint32_t)(w4 * 32) << 16) + (uint32_t)(ch * NT * NG), nslab > 0, 0,
                                                w4 * 32 + lane, me, self, outbox);
                        tcgen05_fence_before();
                        fence_proxy_async_smem();
                        wg_bar_sync(w);
                        if (te < CS - 1) send_message<CS, NGATE, U>(outbox, inbox, &sm.inbox_bar[ch], me, te);
                        mbar_wait_cluster(&sm.inbox_bar[ch], it[k] & 1);
                        if (te == 0 && chain == 0 && w == 0) stamp(c, sm.trace, s, 5);
#pragma unroll
                        for (int q = 0; q < NP; ++q) gather<CS, NGATE, U>(self, inbox, 0, 16 * q + 4 * uo4, bl, acc[q]);
                        ++it[k];
                    }
                    float drt[NP][4], dzt[NP][4], dnt[NP][4];
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        const int ub = ub0 + 16 * q;
                        if (b < B && ub < H) {
                            float dgn[4];
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float dht = dh[q][i] + cr[k][q][i] + acc[q][i];
                                const float dn = dht * (1.0f - zz[q][i]);
                                const float dz = dht * (hp[q][i] - nn[q][i]);
                                dnt[q][i] = dn * (1.0f - nn[q][i] * nn[q][i]);
                                dzt[q][i] = dz * zz[q][i] * (1.0f - zz[q][i]);
                                drt[q][i] = dnt[q][i] * gn[q][i] * rr[q][i] * (1.0f - rr[q][i]);
                                dgn[i] = dnt[q][i] * rr[q][i];
                                cr[k][q][i] = dht * zz[q][i];
                            }
                            __nv_bfloat16* gh_row = p.dgh + m * p.ldg + d * 3 * H + ub;
                            st4_bf16(gh_row, drt[q]); st4_bf16(gh_row + H, dzt[q]); st4_bf16(gh_row + 2 * H, dgn);   // what the other CTAs wait for
                        }
                    }
                    if (te == 0 && chain == 0 && w == 0) stamp(c, sm.trace, s, 6);
                    pub_arrive(w, npub);                         // the publisher warp releases the counter (the consumer fences generic->async proxy after its acquire)
                    if (CPW == 1) done_sync(w, npub);            // deferred stores only after the publisher's fence has been issued
                    ++npub;
                    if (CPW > 1) wg_bar_sync(w);                 // the other chain's stage_row reuses `self`: every thread's gather must be done
#pragma unroll
                    for (int q = 0; q < NP; ++q) {               // off the critical path
                        const int ub = ub0 + 16 * q;
                        if (b < B && ub < H) {
                            __nv_bfloat16* gi_row = p.dgi + m * p.ldg + d * 3 * H + ub;
                            st4_bf16(gi_row, drt[q]); st4_bf16(gi_row + H, dzt[q]); st4_bf16(gi_row + 2 * H, dnt[q]);
                            if (p.db_ih) {                       // bias gradients: fp32 sums over (t, b) of dgi and dgh, this thread's cells
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                    bsum[((0 * NP + q) * 4 + i) * WG_THREADS] += drt[q][i];
                                    bsum[((1 * NP + q) * 4 + i) * WG_THREADS] += dzt[q][i];
                                    bsum[((2 * NP + q) * 4 + i) * WG_THREADS] += dnt[q][i];
                                    bsum[((3 * NP + q) * 4 + i) * WG_THREADS] += dnt[q][i] * rr[q][i];
                                }
                            }
                        }
                    }
                }
            }
        }
        if (p.db_ih) {
            // fold the 32 batch rows of this warpgroup; the two warpgroups then add into the zero-initialised outputs
            // (two commutative additions per element: the result does not depend on their order)
            wg_bar_sync(w);
            const int v = te >> 2, gate4 = v / (4 * NP), q = (v >> 2) % NP, i = v & 3;
            const float* col = sm.bsum + (size_t)w * 16 * NP * WG_THREADS + (size_t)v * WG_THREADS + uo4;
            float sum = 0.f;
            for (int r = 0; r < NG; ++r) sum += col[4 * r];
            const int unit = uc0 + me * U + 4 * uo4 + 16 * q + i;
            if (unit < H) {
                if (gate4 < 3) atomicAdd(p.db_ih + d * 3 * H + gate4 * H + unit, sum);
                if (gate4 != 2) atomicAdd(p.db_hh + d * 3 * H + min(gate4, 2) * H + unit, sum);
            }
        }
    }
    teardown(warp, tmem_base, c, sm);
}

// ---------------------------------------------------------------- host side
template <typename Kern, typename P>
static int launch_cluster_coop(Kern kern, int grid, int cs, size_t smem, const CUtensorMap& m0, const CUtensorMap& m1, const P& p, cudaStream_t s) {
    NSD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attrs[2];
    attrs[0].id = cudaLaunchAttributeClusterDimension;
    attrs[0].val.clusterDim.x = cs; attrs[0].val.clusterDim.y = 1; attrs[0].val.clusterDim.z = 1;
    attrs[1].id = cudaLaunchAttributeCooperative;      // the CTAs spin on each other's step counters: the whole grid must be co-resident
    attrs[1].val.cooperative = 1;
    cfg.attrs = attrs; cfg.numAttrs = 2;
    int max_clusters = 0;
    NSD_CUDA(cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg));
    if (max_clusters * cs < grid) { set_error("gru_ts: %d CTAs in clusters of %d cannot be co-resident (max %d clusters)", grid, cs, max_clusters); return NSD_ERR_INVALID; }
    NSD_CUDA(cudaLaunchKernelEx(&cfg, kern, m0, m1, p));
    count_launch(1);
    return NSD_OK;
}

// Debug aid: NSD_GRU_TRACE=1 prints block 0's per-step event times of batch chain 0 (SM cycles relative to the step's barrier pass).
static long long* trace_begin() {
    const char* e = getenv("NSD_GRU_TRACE");
    if (!e || e[0] != '1') return nullptr;
    long long* d = nullptr;
    if (cudaMalloc(&d, sizeof(long long) * (TRACE_STEPS + 160) * 8) != cudaSuccess) return nullptr;
    cudaMemset(d, 0, sizeof(long long) * (TRACE_STEPS + 160) * 8);
    return d;
}
static void trace_end(const char* who, long long* d, cudaStream_t s, int grid = 0) {
    if (!d) return;
    static long long h[(TRACE_STEPS + 160) * 8];
    cudaStreamSynchronize(s);
    cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(d);
    fprintf(stderr, "[%s trace, chain 0, cycles] step: box0 zones seen->tma_issued first_box_landed mma_committed epi_wake inbox_complete state_stored published | step period\n", who);
    for (int st = 1; st < TRACE_STEPS; ++st) {
        const long long* r = h + st * 8;
        if (r[0] == 0) break;
        fprintf(stderr, "  s=%2d: %6lld %6lld %6lld %6lld %6lld %6lld %6lld | %6lld\n", st, r[1] - r[0], r[2] - r[0], r[3] - r[0], r[4] - r[0],
                r[5] - r[0], r[6] - r[0], r[7] - r[0], st > 1 ? r[0] - h[(st - 1) * 8] : 0LL);
    }
    long long t0 = -1;
    for (int b = 0; b < grid && b < 160; ++b) { const long long v = h[(TRACE_STEPS + b) * 8]; if (v > 0 && (t0 < 0 || v < t0)) t0 = v; }
    if (t0 > 0) {
        fprintf(stderr, "  step 8 per block [ns after first barrier pass]: pass / mma_committed / epi_wake / inbox / stored / published\n");
        for (int b = 0; b < grid && b < 160; ++b) {
            const long long* r = h + (TRACE_STEPS + b) * 8;
            fprintf(stderr, "   blk %3d: %6lld %6lld %6lld %6lld %6lld %6lld\n", b, r[0] - t0, r[3] - t0, r[4] - t0, r[5] - t0, r[6] - t0, r[7] - t0);
        }
    }
}

static int round_up(int a, int b) { return (a + b - 1) / b * b; }
// two chains of 32 rows (one per warpgroup) up to B = 64, four beyond (two per warpgroup)
static int chains_in_flight(int B) { return B > 2 * NG ? 4 : 2; }
static int n_chains(int B) { return (B + NG - 1) / NG; }

constexpr int MAX_H = 1024;             // largest hidden size of the tensor-core path
// A ring stage holds a step's whole K share: nbox boxes of 32 rows x 128 B.  The largest share, the BPTT's at H = MAX_H
// (3H / 4 = 768 columns = 12 boxes), keeps the two stages within 96 KB.
static_assert(2 * ((3 * MAX_H / 4 + BK - 1) / BK) * NG * 128 <= 96 * 1024, "two operand ring stages exceed 96 KB");

static int check_shape(const char* who, int Tp, int B, int H, int D, int cs, int u) {
    if (!(Tp > 0 && B > 0 && H > 0 && (D == 1 || D == 2))) { set_error("%s: bad sizes Tp=%d B=%d H=%d D=%d", who, Tp, B, H, D); return NSD_ERR_INVALID; }
    if (H % 64 != 0 || H > MAX_H) { set_error("%s: hidden size %d must be a multiple of 64 and at most %d on the tensor-core path", who, H, MAX_H); return NSD_ERR_INVALID; }
    const int grid = D * cdiv(H, cs * u) * cs;
    if (grid > sm_count()) { set_error("%s: hidden size %d x %d directions needs %d co-resident CTAs", who, H, D, grid); return NSD_ERR_INVALID; }
    return NSD_OK;
}

}  // namespace rts
}  // namespace nsd

extern "C" {

size_t nsd_gru_tc_workspace(int B, int H, int D) {
    return 256 + (size_t)D * nsd::rts::n_chains(B) * nsd::cdiv(H, 64) * nsd::rts::CNT_STRIDE * sizeof(unsigned int);
}

int nsd_gru_fwd_bf16(const float* gi, int ldgi, const void* w_hh_bf16, const float* b_hh, int Tp, int B, int H, int D,
                     int reverse0, float* hseq, void* hseq_bf16, int ldh, float* r, float* z, float* n, float* hn,
                     void* hdrop_bf16, float p_drop, uint64_t seed, const float* h0, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace nsd;
    using namespace nsd::rts;
    constexpr int CS = 4, U = 16;
    NSD_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "gru_fwd_bf16: p_drop=%f not in [0,1)", (double)p_drop);
    int rc = check_shape("gru_fwd_bf16", Tp, B, H, D, CS, U);
    if (rc) return rc;
    NSD_CHECK_ARG((r && z && n && hn) || (!r && !z && !n && !hn), "gru_fwd_bf16: save pointers must be all set or all NULL");
    NSD_CHECK_ARG((ldgi % 4) == 0 && (ldh % 8) == 0, "gru_fwd_bf16: ldgi must be a multiple of 4 and ldh of 8");
    if (workspace_bytes < nsd_gru_tc_workspace(B, H, D)) { set_error("gru_fwd_bf16: workspace too small"); return NSD_ERR_WORKSPACE; }
    cudaStream_t s = (cudaStream_t)stream;
    NSD_CUDA(cudaMemsetAsync(workspace, 0, nsd_gru_tc_workspace(B, H, D), s));
    CUtensorMap tmH;
    const int row_off = h0 ? B : 0;       // with an initial state, hseq_bf16 has Tp*B + B rows: [bf16(h0) | h_0 .. h_{Tp-1}]
    rc = make_bf16_map(&tmH, hseq_bf16, (long long)Tp * B + row_off, D * H, ldh, NG);
    if (rc) return rc;
    FwdParams p;
    long long* tr = trace_begin();
    const int nper = cdiv(H, CS * U) * CS;
    const int kper = round_up(cdiv(H, CS), UMMA_K);
    const int nbox = cdiv(kper, BK);      // boxes per ring stage
    const int chunked = (kper % BK == 0 && H % BK == 0) ? 1 : 0;
    CUtensorMap tmH3 = tmH;
    if (chunked) { rc = make_bf16_map_chunked(&tmH3, hseq_bf16, (long long)Tp * B + row_off, D * H, ldh, NG, nbox); if (rc) return rc; }
    p.c = {Tp, B, H, D, reverse0, nper, n_chains(B), H, kper, h0 ? 0 : 1, row_off, nbox, chunked, CS, CS * U, nper / CS, reinterpret_cast<unsigned int*>(workspace), tr};
    p.h0 = h0;
    p.w = reinterpret_cast<const __nv_bfloat16*>(w_hh_bf16);
    p.gi = gi; p.ldgi = ldgi; p.b_hh = b_hh; p.hseq = hseq; p.hseq_bf = reinterpret_cast<__nv_bfloat16*>(hseq_bf16); p.ldh = ldh;
    p.r = r; p.z = z; p.n = n; p.hn = hn;
    p.hdrop = reinterpret_cast<__nv_bfloat16*>(hdrop_bf16); p.drop_thresh = dropout_threshold(p_drop); p.inv_keep = 1.0f / (1.0f - p_drop); p.seed = seed;
    const int nch = chains_in_flight(B);
    const size_t smem = smem_bytes(2 * nbox * NG * 128, nch, (CS - 1) * 3 * U * NG * 2, 3 * U * NG * 4);
    rc = nch == 4 ? launch_cluster_coop(gru_fwd_ts_kernel<4>, D * nper, CS, smem, tmH, tmH3, p, s)
                  : launch_cluster_coop(gru_fwd_ts_kernel<2>, D * nper, CS, smem, tmH, tmH3, p, s);
    trace_end("gru_fwd_bf16", tr, s, D * nper);
    return rc;
}

int nsd_gru_bwd_bf16(const float* dhseq, int lddh, const float* hseq, int ldh, const float* r, const float* z,
                     const float* n, const float* hn, const void* w_hhT_bf16, int Tp, int B, int H, int D, int reverse0,
                     void* dgi_bf16, void* dgh_bf16, int ldg, float p_drop, uint64_t seed, float* db_ih, float* db_hh,
                     void* workspace, size_t workspace_bytes, void* stream) {
    using namespace nsd;
    using namespace nsd::rts;
    constexpr int CS = 4, U = 32;
    NSD_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "gru_bwd_bf16: p_drop=%f not in [0,1)", (double)p_drop);
    NSD_CHECK_ARG((db_ih == nullptr) == (db_hh == nullptr), "gru_bwd_bf16: db_ih and db_hh must both be set or both be NULL");
    int rc = check_shape("gru_bwd_bf16", Tp, B, H, D, CS, U);
    if (rc) return rc;
    NSD_CHECK_ARG((lddh % 4) == 0 && (ldh % 4) == 0 && (ldg % 8) == 0, "gru_bwd_bf16: leading dimensions must be multiples of 4 (f32) / 8 (bf16)");
    if (workspace_bytes < nsd_gru_tc_workspace(B, H, D)) { set_error("gru_bwd_bf16: workspace too small"); return NSD_ERR_WORKSPACE; }
    cudaStream_t s = (cudaStream_t)stream;
    NSD_CUDA(cudaMemsetAsync(workspace, 0, nsd_gru_tc_workspace(B, H, D), s));
    CUtensorMap tmG;
    rc = make_bf16_map(&tmG, dgh_bf16, (long long)Tp * B, D * 3 * H, ldg, NG);
    if (rc) return rc;
    BwdParams p;
    long long* tr = trace_begin();
    const int nper = cdiv(H, CS * U) * CS;
    const int kper = round_up(cdiv(3 * H, CS), UMMA_K);
    const int nbox = cdiv(kper, BK);      // boxes per ring stage
    const int chunked = (kper % BK == 0) ? 1 : 0;
    CUtensorMap tmG3 = tmG;
    if (chunked) { rc = make_bf16_map_chunked(&tmG3, dgh_bf16, (long long)Tp * B, D * 3 * H, ldg, NG, nbox); if (rc) return rc; }
    p.c = {Tp, B, H, D, reverse0, nper, n_chains(B), 3 * H, kper, 1, 0, nbox, chunked, CS, CS * U, nper / CS, reinterpret_cast<unsigned int*>(workspace), tr};
    p.wT = reinterpret_cast<const __nv_bfloat16*>(w_hhT_bf16);
    p.dhseq = dhseq; p.lddh = lddh; p.hseq = hseq; p.ldh = ldh; p.r = r; p.z = z; p.n = n; p.hn = hn;
    p.dgi = reinterpret_cast<__nv_bfloat16*>(dgi_bf16); p.dgh = reinterpret_cast<__nv_bfloat16*>(dgh_bf16); p.ldg = ldg;
    p.drop_thresh = p_drop > 0.f ? dropout_threshold(p_drop) : 0u; p.inv_keep = 1.0f / (1.0f - p_drop); p.seed = seed;
    p.db_ih = db_ih; p.db_hh = db_hh;
    if (db_ih) {
        NSD_CUDA(cudaMemsetAsync(db_ih, 0, sizeof(float) * (size_t)D * 3 * H, s));
        NSD_CUDA(cudaMemsetAsync(db_hh, 0, sizeof(float) * (size_t)D * 3 * H, s));
    }
    const int nch = chains_in_flight(B);
    const size_t smem = smem_bytes(2 * nbox * NG * 128, nch, (CS - 1) * U * NG * 2, U * NG * 4, db_ih ? sizeof(float) * 2 * 16 * (U / 16) * WG_THREADS : 0);
    rc = nch == 4 ? launch_cluster_coop(gru_bwd_ts_kernel<4>, D * nper, CS, smem, tmG, tmG3, p, s)
                  : launch_cluster_coop(gru_bwd_ts_kernel<2>, D * nper, CS, smem, tmG, tmG3, p, s);
    trace_end("gru_bwd_bf16", tr, s, D * nper);
    return rc;
}

}  // extern "C"
