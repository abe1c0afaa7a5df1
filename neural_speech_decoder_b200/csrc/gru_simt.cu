// K3 (fp32 path): GRU recurrence forward and backward-through-time on CUDA cores.
//
// One layer-direction of nn.GRU (reference model.py:50-57, 104-119).  A CTA owns UT=8 hidden units
// (24 rows of W_hh), keeps them resident in shared memory for the whole sequence and walks the
// timesteps inside ONE cooperative launch with a grid-wide barrier per step; h_{t-1} is re-read from
// L2 each step.  When the grid cannot be co-resident (large H) the same kernel body is launched once
// per step with W_hh streamed from L2 instead.  The tensor-core path is in gru_ts.cu.
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace nsd {

constexpr int GR_UT = 8;          // hidden units per CTA
constexpr int GR_THREADS = 128;   // 16 batch lanes x 8 units
constexpr int GR_BT = 64;         // batch rows per tile (4 per thread, strided by 16)
constexpr int GR_KC = 128;        // reduction chunk staged in shared memory
constexpr int GR_KCP = GR_KC + 4; // padded row (conflict-free LDS.128 per quarter warp)

__device__ __forceinline__ float sigm(float x) { return 1.0f / (1.0f + expf(-x)); }

struct GruFwdParams {
    const float* gi; const float* w_hh; const float* b_hh;
    float* hseq; float* r; float* z; float* n; float* hn;
    const int* n_frames;                               // [B] frames per row (NULL = Tp): rows at t >= n_frames[b] output 0
    int ldgi, ldh, Tp, B, H, reverse, step0, nsteps, w_in_smem;
};

// stage src[b0+row][k0 .. k0+GR_KC) (row stride ld) into s[row][GR_KCP]; rows >= B and k >= klim read as 0
__device__ __forceinline__ void stage_rows(float* s, const float* src, int ld, int b0, int B, int k0, int klim, int tid) {
    for (int i = tid; i < GR_BT * (GR_KC / 4); i += GR_THREADS) {
        const int row = i / (GR_KC / 4), q = i - row * (GR_KC / 4);
        const int b = b0 + row, k = k0 + q * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (b < B) {
            const float* p = src + (size_t)b * ld + k;
            if (k + 4 <= klim && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) v = __ldcg(reinterpret_cast<const float4*>(p));
            else {
                if (k + 0 < klim) v.x = __ldcg(p + 0);
                if (k + 1 < klim) v.y = __ldcg(p + 1);
                if (k + 2 < klim) v.z = __ldcg(p + 2);
                if (k + 3 < klim) v.w = __ldcg(p + 3);
            }
        }
        *reinterpret_cast<float4*>(s + row * GR_KCP + q * 4) = v;
    }
}

__global__ void __launch_bounds__(GR_THREADS) gru_fwd_f32_kernel(GruFwdParams p) {
    extern __shared__ __align__(16) float smem[];
    const int H = p.H, B = p.B;
    const int HP = ((H + 3) / 4) * 4;                 // padded k extent of the resident W slice
    float* hs = smem;                                  // [GR_BT][GR_KCP]
    float* ws = smem + GR_BT * GR_KCP;                 // [3][GR_UT][HP]   (only when w_in_smem)
    const int tid = threadIdx.x;
    const int bq = tid & 15, ul = tid >> 4;
    const int u0 = blockIdx.x * GR_UT;
    const int u = u0 + ul;
    const bool uok = u < H;

    if (p.w_in_smem) {
        for (int i = tid; i < 3 * GR_UT * HP; i += GR_THREADS) {
            const int k = i % HP, gu = i / HP;
            const int g = gu / GR_UT, uu = u0 + (gu % GR_UT);
            ws[i] = (k < H && uu < H) ? __ldg(p.w_hh + ((size_t)g * H + uu) * H + k) : 0.f;
        }
    }
    float bh[3] = {0.f, 0.f, 0.f};
    if (uok) { bh[0] = __ldg(p.b_hh + u); bh[1] = __ldg(p.b_hh + H + u); bh[2] = __ldg(p.b_hh + 2 * H + u); }
    __syncthreads();

    for (int s = 0; s < p.nsteps; ++s) {
        const int step = p.step0 + s;
        const int t = p.reverse ? (p.Tp - 1 - step) : step;
        const int tprev = p.reverse ? t + 1 : t - 1;
        const bool has_prev = step > 0;
        const float* hprev = p.hseq + (size_t)tprev * B * p.ldh;     // only dereferenced when has_prev
        for (int b0 = 0; b0 < B; b0 += GR_BT) {
            float acc[3][4];
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[g][i] = 0.f;
            if (has_prev) {
                for (int k0 = 0; k0 < H; k0 += GR_KC) {
                    __syncthreads();
                    stage_rows(hs, hprev, p.ldh, b0, B, k0, H, tid);
                    __syncthreads();
                    const int kn = min(GR_KC, H - k0);
                    if (uok) {
                        for (int k = 0; k < kn; k += 4) {
                            float4 w[3];
#pragma unroll
                            for (int g = 0; g < 3; ++g) {
                                if (p.w_in_smem) w[g] = *reinterpret_cast<const float4*>(ws + ((size_t)g * GR_UT + ul) * HP + k0 + k);
                                else {
                                    const float* wp = p.w_hh + ((size_t)g * H + u) * H + k0 + k;
                                    w[g].x = __ldg(wp);
                                    w[g].y = (k + 1 < kn) ? __ldg(wp + 1) : 0.f;
                                    w[g].z = (k + 2 < kn) ? __ldg(wp + 2) : 0.f;
                                    w[g].w = (k + 3 < kn) ? __ldg(wp + 3) : 0.f;
                                }
                            }
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float4 h = *reinterpret_cast<const float4*>(hs + (bq + 16 * i) * GR_KCP + k);
#pragma unroll
                                for (int g = 0; g < 3; ++g) {
                                    acc[g][i] = fmaf(h.x, w[g].x, acc[g][i]);
                                    acc[g][i] = fmaf(h.y, w[g].y, acc[g][i]);
                                    acc[g][i] = fmaf(h.z, w[g].z, acc[g][i]);
                                    acc[g][i] = fmaf(h.w, w[g].w, acc[g][i]);
                                }
                            }
                        }
                    }
                }
            }
            if (uok) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int b = b0 + bq + 16 * i;
                    if (b >= B) continue;
                    const size_t row = (size_t)t * B + b;
                    const float* gir = p.gi + row * p.ldgi;
                    const float ghr = acc[0][i] + bh[0], ghz = acc[1][i] + bh[1], ghn = acc[2][i] + bh[2];
                    const float rr = sigm(__ldg(gir + u) + ghr);
                    const float zz = sigm(__ldg(gir + H + u) + ghz);
                    const float nn = tanhf(__ldg(gir + 2 * H + u) + rr * ghn);
                    const float hp = has_prev ? __ldcg(hprev + (size_t)b * p.ldh + u) : 0.f;
                    const float hv = (1.0f - zz) * nn + zz * hp;
                    // past its frames a row outputs 0, which is also the zero initial state the reverse direction then reads
                    p.hseq[row * p.ldh + u] = (p.n_frames == nullptr || t < __ldg(p.n_frames + b)) ? hv : 0.f;
                    if (p.r) {
                        p.r[row * H + u] = rr; p.z[row * H + u] = zz; p.n[row * H + u] = nn; p.hn[row * H + u] = ghn;
                    }
                }
            }
        }
        if (s + 1 < p.nsteps) cg::this_grid().sync();
    }
}

struct GruBwdParams {
    const float* dhseq; const float* hseq; const float* r; const float* z; const float* n; const float* hn;
    const float* w_hh; float* dgi; float* dghn; float* carry;
    const int* n_frames;                               // [B] or NULL: no gradient flows through t >= n_frames[b]
    int lddh, ldh, ldgi, Tp, B, H, reverse, step0, nsteps, w_in_smem;
};

__global__ void __launch_bounds__(GR_THREADS) gru_bwd_f32_kernel(GruBwdParams p) {
    extern __shared__ __align__(16) float smem[];
    const int H = p.H, B = p.B, H3 = 3 * p.H;
    const int JP = ((H3 + 3) / 4) * 4;
    float* ds = smem;                                  // [GR_BT][GR_KCP]
    float* wt = smem + GR_BT * GR_KCP;                 // [GR_UT][JP]: wt[u][j] = W_hh[j][u0+u]
    const int tid = threadIdx.x;
    const int bq = tid & 15, ul = tid >> 4;
    const int u0 = blockIdx.x * GR_UT;
    const int u = u0 + ul;
    const bool uok = u < H;

    if (p.w_in_smem) {
        for (int i = tid; i < GR_UT * JP; i += GR_THREADS) {
            const int uu = i % GR_UT, j = i / GR_UT;       // consecutive threads read consecutive columns of one row
            wt[(size_t)uu * JP + j] = (j < H3 && u0 + uu < H) ? __ldg(p.w_hh + (size_t)j * H + u0 + uu) : 0.f;
        }
    }
    __syncthreads();

    // BPTT visits timesteps in the opposite order of the forward recurrence.
    for (int s = 0; s < p.nsteps; ++s) {
        const int step = p.step0 + s;                       // 0 .. Tp-1 in backward order
        const int t = p.reverse ? step : (p.Tp - 1 - step);
        const int tnext = p.reverse ? t - 1 : t + 1;        // the step handled in the previous iteration
        const int tprev = p.reverse ? t + 1 : t - 1;        // forward-time predecessor (source of h_{t-1})
        const bool has_fwd_prev = p.reverse ? (t + 1 < p.Tp) : (t > 0);
        for (int b0 = 0; b0 < B; b0 += GR_BT) {
            // phase B of the previous iteration: carry = dht*z (already stored) + dgh_{tnext} W_hh[:, u]
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            if (step > 0) {
                for (int j0 = 0; j0 < H3; j0 += GR_KC) {
                    // the chunk [j0, j0+KC) lies in dgi columns (< 2H) and/or in dghn (>= 2H): stage piecewise
                    __syncthreads();
                    if ((2 * H) % GR_KC == 0) {
                        // the chunk lies wholly in the dgi columns (< 2H) or wholly in dghn: vectorised row staging
                        if (j0 < 2 * H) stage_rows(ds, p.dgi + (size_t)tnext * B * p.ldgi, p.ldgi, b0, B, j0, 2 * H, tid);
                        else stage_rows(ds, p.dghn + (size_t)tnext * B * H, H, b0, B, j0 - 2 * H, H, tid);
                    } else
                    for (int i = tid; i < GR_BT * GR_KC; i += GR_THREADS) {
                        const int row = i / GR_KC, jj = i - row * GR_KC;
                        const int b = b0 + row, j = j0 + jj;
                        float v = 0.f;
                        if (b < B && j < H3) {
                            const size_t m = (size_t)tnext * B + b;
                            v = (j < 2 * H) ? __ldcg(p.dgi + m * p.ldgi + j) : __ldcg(p.dghn + m * H + (j - 2 * H));
                        }
                        ds[row * GR_KCP + jj] = v;
                    }
                    __syncthreads();
                    const int jn = min(GR_KC, H3 - j0);
                    if (uok) {
                        for (int j = 0; j < jn; j += 4) {
                            float4 w;
                            if (p.w_in_smem) w = *reinterpret_cast<const float4*>(wt + (size_t)ul * JP + j0 + j);
                            else {
                                const float* wp = p.w_hh + (size_t)(j0 + j) * H + u;
                                w.x = __ldg(wp);
                                w.y = (j + 1 < jn) ? __ldg(wp + H) : 0.f;
                                w.z = (j + 2 < jn) ? __ldg(wp + 2 * (size_t)H) : 0.f;
                                w.w = (j + 3 < jn) ? __ldg(wp + 3 * (size_t)H) : 0.f;
                            }
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float4 d = *reinterpret_cast<const float4*>(ds + (bq + 16 * i) * GR_KCP + j);
                                acc[i] = fmaf(d.x, w.x, acc[i]);
                                acc[i] = fmaf(d.y, w.y, acc[i]);
                                acc[i] = fmaf(d.z, w.z, acc[i]);
                                acc[i] = fmaf(d.w, w.w, acc[i]);
                            }
                        }
                    }
                }
            }
            // phase A: gate gradients of step t for the owned units
            if (uok) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int b = b0 + bq + 16 * i;
                    if (b >= B) continue;
                    const size_t m = (size_t)t * B + b;
                    if (p.n_frames != nullptr && t >= __ldg(p.n_frames + b)) {
                        float* g = p.dgi + m * p.ldgi;
                        g[u] = 0.f; g[H + u] = 0.f; g[2 * H + u] = 0.f;
                        p.dghn[m * H + u] = 0.f;
                        p.carry[(size_t)b * H + u] = 0.f;
                        continue;
                    }
                    float dh = __ldg(p.dhseq + m * p.lddh + u);
                    if (step > 0) dh += p.carry[(size_t)b * H + u] + acc[i];
                    const float rr = __ldg(p.r + m * H + u), zz = __ldg(p.z + m * H + u);
                    const float nn = __ldg(p.n + m * H + u), hn = __ldg(p.hn + m * H + u);
                    const float hp = has_fwd_prev ? __ldg(p.hseq + ((size_t)tprev * B + b) * p.ldh + u) : 0.f;
                    const float dn = dh * (1.0f - zz);
                    const float dz = dh * (hp - nn);
                    const float dnt = dn * (1.0f - nn * nn);
                    const float dzt = dz * zz * (1.0f - zz);
                    const float drt = dnt * hn * rr * (1.0f - rr);
                    float* g = p.dgi + m * p.ldgi;
                    g[u] = drt; g[H + u] = dzt; g[2 * H + u] = dnt;
                    p.dghn[m * H + u] = dnt * rr;
                    p.carry[(size_t)b * H + u] = dh * zz;
                }
            }
        }
        if (s + 1 < p.nsteps) cg::this_grid().sync();
    }
}

static bool fits_cooperative(const void* kernel, int grid, size_t smem) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, GR_THREADS, smem) != cudaSuccess) return false;
    return (long long)per_sm * sm_count() >= grid;
}

}  // namespace nsd

extern "C" {

int nsd_gru_fwd_f32(const float* gi, int ldgi, const float* w_hh, const float* b_hh, int Tp, int B, int H,
                    int reverse, float* hseq, int ldh, float* r, float* z, float* n, float* hn, const int* n_frames, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(Tp > 0 && B > 0 && H > 0, "gru_fwd_f32: bad sizes");
    NSD_CHECK_ARG((r && z && n && hn) || (!r && !z && !n && !hn), "gru_fwd_f32: save pointers must be all set or all NULL");
    GruFwdParams p;
    p.gi = gi; p.w_hh = w_hh; p.b_hh = b_hh; p.hseq = hseq; p.r = r; p.z = z; p.n = n; p.hn = hn; p.n_frames = n_frames;
    p.ldgi = ldgi; p.ldh = ldh; p.Tp = Tp; p.B = B; p.H = H; p.reverse = reverse;
    const int grid = cdiv(H, GR_UT);
    const int HP = ((H + 3) / 4) * 4;
    const size_t smem_small = sizeof(float) * GR_BT * GR_KCP;
    const size_t smem_big = smem_small + sizeof(float) * 3 * GR_UT * HP;
    cudaStream_t s = (cudaStream_t)stream;
    bool coop = false;
    if (smem_big <= 227 * 1024) {
        NSD_CUDA(cudaFuncSetAttribute(gru_fwd_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_big));
        coop = fits_cooperative((const void*)gru_fwd_f32_kernel, grid, smem_big);
    }
    if (coop) {
        p.step0 = 0; p.nsteps = Tp; p.w_in_smem = 1;
        void* args[] = {&p};
        NSD_CUDA(cudaLaunchCooperativeKernel((const void*)gru_fwd_f32_kernel, dim3(grid), dim3(GR_THREADS), args, smem_big, s));
        count_launch(1);
    } else {
        p.nsteps = 1; p.w_in_smem = 0;
        for (int st = 0; st < Tp; ++st) {
            p.step0 = st;
            gru_fwd_f32_kernel<<<grid, GR_THREADS, smem_small, s>>>(p);
        }
        count_launch(Tp - 1);
        NSD_LAUNCH_CHECK();
    }
    return NSD_OK;
}

size_t nsd_gru_bwd_workspace(int B, int H) { return sizeof(float) * (size_t)B * H; }

int nsd_gru_bwd_f32(const float* dhseq, int lddh, const float* hseq, int ldh, const float* r, const float* z,
                    const float* n, const float* hn, const float* w_hh, int Tp, int B, int H, int reverse,
                    float* dgi, int ldgi, float* dghn, const int* n_frames, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace nsd;
    NSD_CHECK_ARG(Tp > 0 && B > 0 && H > 0, "gru_bwd_f32: bad sizes");
    if (workspace_bytes < nsd_gru_bwd_workspace(B, H)) { set_error("gru_bwd_f32: workspace too small"); return NSD_ERR_WORKSPACE; }
    GruBwdParams p;
    p.dhseq = dhseq; p.hseq = hseq; p.r = r; p.z = z; p.n = n; p.hn = hn; p.w_hh = w_hh;
    p.dgi = dgi; p.dghn = dghn; p.carry = reinterpret_cast<float*>(workspace); p.n_frames = n_frames;
    p.lddh = lddh; p.ldh = ldh; p.ldgi = ldgi; p.Tp = Tp; p.B = B; p.H = H; p.reverse = reverse;
    const int grid = cdiv(H, GR_UT);
    const int JP = ((3 * H + 3) / 4) * 4;
    const size_t smem_small = sizeof(float) * GR_BT * GR_KCP;
    const size_t smem_big = smem_small + sizeof(float) * GR_UT * JP;
    cudaStream_t s = (cudaStream_t)stream;
    bool coop = false;
    if (smem_big <= 227 * 1024) {
        NSD_CUDA(cudaFuncSetAttribute(gru_bwd_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_big));
        coop = fits_cooperative((const void*)gru_bwd_f32_kernel, grid, smem_big);
    }
    if (coop) {
        p.step0 = 0; p.nsteps = Tp; p.w_in_smem = 1;
        void* args[] = {&p};
        NSD_CUDA(cudaLaunchCooperativeKernel((const void*)gru_bwd_f32_kernel, dim3(grid), dim3(GR_THREADS), args, smem_big, s));
        count_launch(1);
    } else {
        p.nsteps = 1; p.w_in_smem = 0;
        for (int st = 0; st < Tp; ++st) {
            p.step0 = st;
            gru_bwd_f32_kernel<<<grid, GR_THREADS, smem_small, s>>>(p);
        }
        count_launch(Tp - 1);
        NSD_LAUNCH_CHECK();
    }
    return NSD_OK;
}

}  // extern "C"
