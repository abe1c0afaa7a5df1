/*
 * nsd_b200.h -- C ABI of the B200-native GRUDecoder + CTC hot path.
 *
 * The reference (EdwardoSunny/Neural-Speech-Decoder) is pure Python and has no FFI
 * of its own: the boundary its trainer uses is the torch.nn.Module contract
 *   GRUDecoder.forward(neuralInput[B,T,N], dayIdx[B]) -> logits[B,T',C]   src/neural_decoder/model.py:83-123
 *   torch.nn.CTCLoss(blank=0, reduction="mean", zero_infinity=True)       src/neural_decoder/neural_decoder_trainer.py:139-141, 213-218
 *   argmax / unique_consecutive / drop-blank greedy decode                src/neural_decoder/neural_decoder_trainer.py:313-320
 * Each entry point below replaces the third-party torch operator(s) that one of
 * those lines reaches on a GPU; the citation names the reference line.  The
 * Python mirror of the reference interface (neural_speech_decoder_b200/model.py,
 * ctc.py) is the only caller.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the comment says "host";
 *   - no torch types, no allocation, no host synchronisation inside any call:
 *     the caller supplies outputs and workspaces and a cudaStream_t (as void*);
 *   - return value: 0 on success, a negative NSD_ERR_* code otherwise;
 *     nsd_last_error() gives a thread-local message for the last failure;
 *   - "time-major" activations are [T', B, F] with row m = t*B + b;
 *   - dtype codes: NSD_F32 = 0, NSD_BF16 = 1.
 */
#ifndef NSD_B200_H
#define NSD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NSD_OK 0
#define NSD_ERR_INVALID (-1)     /* bad argument / unsupported shape */
#define NSD_ERR_CUDA (-2)        /* a CUDA runtime call failed */
#define NSD_ERR_WORKSPACE (-3)   /* workspace too small */

#define NSD_F32 0
#define NSD_BF16 1

/* ---- library ---------------------------------------------------------- */
int nsd_version(void);
const char* nsd_last_error(void);
/* number of kernels this library has enqueued in this process (bench.py reports the per-step count). */
unsigned long long nsd_launch_count(void);
/* sm count and compute capability of the current device (host out-pointers). */
int nsd_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- K1: fused front end --------------------------------------------------
 * Replaces F.conv1d(groups=N,"same") + index_select + einsum + Softsign + nn.Unfold
 * (augmentations.py:91; model.py:84-101).
 *   ys[b,t,c]   = sum_k taps[k] * x[b, t-(ntaps-1)/2+k, c]         (zero padded)
 *   pre[b,t,k]  = sum_d ys[b,t,d] * day_w[day[b],d,k] + day_b[day[b],k]
 *   z           = pre / (1+|pre|)
 *   patches[j*B+b, c*K+kk] = z[b, j*S+kk, c]                         (time-major rows)
 * ys and z ([B,T,N] f32) are written for the backward; rows t >= (T'-1)*S+K are
 * left untouched.  err_flag (device-visible int32, may be mapped pinned host
 * memory, may be NULL) is set to 1 if a day index is outside [0,n_days).
 * Fused training augmentation (neural_decoder_trainer.py:194-201; SURVEY 8f rank 2): when
 * white_noise_sd / constant_offset_sd are non-zero, x is read as nsd_input_noise(x, ...) with the
 * same seed would have written it -- no extra pass over X.  Distributional parity with the
 * reference's torch.randn (counter-based Philox + Box-Muller here).
 * Per-utterance lengths (packed sequences): x_len != NULL is [B] int64 on the device; bins t >= x_len[b] of utterance b
 * are read as 0 after the noise (no noise is drawn there), so every frame whose window lies inside the utterance sees what
 * the utterance run alone, zero right-padded, would give.  A length is clamped to [0, T] here; nsd_frame_counts flags one
 * outside [kernel_len, T].  x_len == NULL reads all T bins, as the reference does.                                      */
int nsd_frontend_fwd(const float* x, const int64_t* day_idx, const float* day_w, const float* day_b,
                     const float* taps, int ntaps, int B, int T, int N, int n_days, int kernel_len,
                     int stride_len, float* ys, float* z, void* patches, int patches_dtype,
                     int* err_flag, float white_noise_sd, float constant_offset_sd, uint64_t noise_seed,
                     const int64_t* x_len, void* stream);
/* Frames of each utterance whose whole window lies inside its x_len[b] bins (x_len [B] int64, device):
 * n_frames[b] = floor((x_len[b] - kernel_len) / stride_len) + 1 clamped to [0, T'] ([B] int32, device), with no host
 * synchronisation.  A length outside [kernel_len, T] sets bit 2 (value 2) of *err_flag (may be NULL).                  */
int nsd_frame_counts(const int64_t* x_len, int B, int T, int kernel_len, int stride_len, int* n_frames, int* err_flag,
                     void* stream);
/* The augmentation on its own: out[b,t,c] = x[b,t,c] + white_noise_sd * n0[b,t,c] + constant_offset_sd * n1[b,c],
 * n0, n1 standard normal, functions of (seed, element index) only.  x, out: [B,T,N] f32 contiguous (may alias). */
int nsd_input_noise(const float* x, float* out, int B, int T, int N, float white_noise_sd, float constant_offset_sd,
                    uint64_t seed, void* stream);

/* Backward of K1 w.r.t. dayWeights / dayBias (the gradient w.r.t. X is nsd_frontend_bwd_input): col2im of dpatches,
 * softsign', per-utterance ys^T dpre, then a deterministic segment-reduce over
 * utterances that share a day (autograd of model.py:89-101).
 * workspace: B*N*(N+1) floats.  d_day_w [n_days,N,N], d_day_b [n_days,N] are overwritten. */
int nsd_frontend_bwd(const void* dpatches, int dpatches_dtype, const float* ys, const float* z,
                     const int64_t* day_idx, int B, int T, int N, int n_days, int kernel_len,
                     int stride_len, float* d_day_w, float* d_day_b, void* workspace,
                     size_t workspace_bytes, void* stream);
size_t nsd_frontend_bwd_workspace(int B, int N);
/* Backward of K1 w.r.t. X, one launch: dz = col2im(dpatches) (dpatches [T'*B, N*K] time-major, f32 or bf16),
 * dpre = dz * (1-|z|)^2, dy_b = dpre_b W[day_b]^T, dx[b,s,c] = sum_k taps[k] dy[b,s+L-k,c] over 0 <= s+L-k < T with
 * L = (ntaps-1)/2 (the transpose of the "same"-padded smoother).  The training noise is additive and needs no term.
 * z [B,T,N] f32 as nsd_frontend_fwd wrote it; day_w [n_days,N,N] f32; dx [B,T,N] f32 is overwritten, every row.
 * bf16 dpatches with N in {64,128,256}: the product on tensor cores (bf16 operands, fp32 accumulate); otherwise fp32 FFMA.
 * No atomics: every element is summed in a fixed order.  An out-of-range day id reads day 0 (the forward flags it).
 * x_len != NULL ([B] int64, as given to nsd_frontend_fwd): dx[b, s >= x_len[b]] = 0, the bins the forward read as 0.
 * (nsd_frontend_bwd needs no lengths: with the recurrence's frame counts, dpatches is 0 at every frame that reads such a bin.) */
int nsd_frontend_bwd_input(const void* dpatches, int dpatches_dtype, const float* z, const int64_t* day_idx,
                           const float* day_w, const float* taps, int ntaps, int B, int T, int N, int n_days,
                           int kernel_len, int stride_len, float* dx, const int64_t* x_len, void* stream);

/* ---- K2: GEMMs -----------------------------------------------------------------
 * Row-major C[M,N] = op(A) * op(B) (+ bias[N]) (+ beta*C).  op(A) is [M,K]: stored
 * [M,K] (lda) if !transa, [K,M] (lda) if transa.  op(B) is [K,N]: stored [K,N] (ldb)
 * if !transb, [N,K] (ldb) if transb.  Time-batched W_ih projections, their dgrad /
 * wgrad and the output layer (nn.GRU input GEMMs model.py:50-57,119; nn.Linear
 * model.py:76-81,122).  _f32 is the CUDA-core fp32 path used for fp32 parity;
 * _bf16 is the tcgen05/TMA tensor-core path (bf16 operands, fp32 accumulate in TMEM). */
int nsd_gemm_f32(int transa, int transb, int M, int N, int K, const float* A, int lda, const float* B,
                 int ldb, float* C, int ldc, const float* bias, float beta, void* stream);
int nsd_gemm_bf16(int transa, int transb, int M, int N, int K, const void* A, int lda, const void* B,
                  int ldb, void* C, int ldc, int c_dtype, const float* bias, float beta, void* stream);
/* Two GEMMs of identical shape and layout in ONE launch (operands A0/B0 -> C0 and A1/B1 -> C1, shared leading
 * dimensions; no bias, no beta): the two directions' time-batched W_hh weight gradients each fill only 65 % of the
 * GPU on their own.  Shapes the paired tensor-core form does not take fall back to two nsd_gemm_bf16 calls. */
int nsd_gemm_bf16_x2(int transa, int transb, int M, int N, int K, const void* A0, const void* A1, int lda, const void* B0,
                     const void* B1, int ldb, void* C0, void* C1, int ldc, int c_dtype, void* stream);

/* column sums: out[n] = sum_m a[m*lda + n]  (bias gradients); two fixed-order stages, workspace nsd_colsum_workspace(N). */
int nsd_colsum(const void* a, int a_dtype, int M, int N, int lda, float* out, void* workspace, size_t workspace_bytes,
               void* stream);
size_t nsd_colsum_workspace(int N);
/* dtype conversion of a contiguous buffer, f32 <-> bf16. */
int nsd_cast(const void* src, int src_dtype, void* dst, int dst_dtype, size_t n, void* stream);
/* bf16 copies of a row-major [R,C] matrix (f32 or bf16 source): dst [R,C] (ld_dst) and/or its transpose dstT [C,R]
 * (ld_dstT); either may be NULL.  (nsd_gemm_bf16 takes either operand major natively; the transposed form is what the
 * BPTT kernel's stationary W_hh^T operand is loaded from.) */
int nsd_cast_transpose(const void* src, int src_dtype, int R, int C, int ld_src, void* dst, int ld_dst, void* dstT,
                       int ld_dstT, void* stream);
/* dstT[i] [C,R] (ld_dstT) <- transpose of the bf16 matrix src[i] [R,C] (ld_src), i < n, one launch for all of them (host arrays of device
 * pointers; R, C and the leading dimensions even, bases 4-byte aligned).  The BPTT's W_hh^T operands of every layer and direction per step
 * (model.py:50-57 keeps W_hh as [3H, H]; autograd's matmul backward reads it transposed). */
int nsd_transpose_bf16_multi(int n, const void* const* src, void* const* dstT, int R, int C, int ld_src, int ld_dstT, void* stream);
/* out[B,T,C] <- in[T,B,C] (or the inverse with the roles of T and B swapped by the caller). */
int nsd_swap01_f32(const float* in, float* out, int D0, int D1, int C, void* stream);

/* ---- K3: GRU recurrence ----------------------------------------------------------
 * One layer-direction of nn.GRU with h0 = 0 (model.py:104-119), gate order [r,z,n]:
 *   gh = h_{t-1} W_hh^T + b_hh ; r = s(gi_r+gh_r) ; z = s(gi_z+gh_z)
 *   n = tanh(gi_n + r*gh_n)    ; h_t = (1-z)*n + z*h_{t-1}
 * gi ([T',B,ldgi], already holding x W_ih^T + b_ih) is read at column offset 0 of the
 * pointer given (the caller offsets it for the reverse direction).  hseq is written
 * at the pointer given with row stride ldh.  r,z,n,hn ([T',B,H]) are saved when
 * non-NULL.  reverse != 0 walks t = T'-1..0 over the full padded length.
 * The fp32 path keeps W_hh resident in shared memory across a persistent cooperative
 * launch when it fits, else launches one step at a time.
 * Packed sequences (nn.GRU on pack_padded_sequence): n_frames != NULL is [B] int32 on the device (nsd_frame_counts),
 * each in [0, T'].  Row b then runs its own frames only: the forward direction t = 0 .. n_b-1, the reverse direction from
 * t = n_b-1 with h = 0, and at t >= n_b its output hseq is exactly 0 (pad_packed_sequence), so the next layer's input
 * there is 0.  n_frames == NULL: every row runs all T' steps (the reference's padded batch).                        */
int nsd_gru_fwd_f32(const float* gi, int ldgi, const float* w_hh, const float* b_hh, int Tp, int B, int H,
                    int reverse, float* hseq, int ldh, float* r, float* z, float* n, float* hn,
                    const int* n_frames, void* stream);
/* BPTT: dh_t = dhseq_t + carry ; writes dgi[T',B,ldgi] = [dr~,dz~,dn~] and dghn[T',B,H] = dn~*r.
 * n_frames as in the forward: no gradient flows through t >= n_b (dgi, dghn and the carry are 0 there; dhseq there is
 * not read). */
int nsd_gru_bwd_f32(const float* dhseq, int lddh, const float* hseq, int ldh, const float* r, const float* z,
                    const float* n, const float* hn, const float* w_hh, int Tp, int B, int H, int reverse,
                    float* dgi, int ldgi, float* dghn, const int* n_frames, void* workspace, size_t workspace_bytes,
                    void* stream);
size_t nsd_gru_bwd_workspace(int B, int H);

/* Tensor-core (bf16 operand, fp32 accumulate/state) form of the same recurrence: ONE cooperative launch walks all
 * timesteps of one layer for D directions at once (direction 1, or direction 0 when reverse0 != 0, runs
 * t = T'-1..0).  w_hh_bf16 is the bf16 copy of [weight_hh_l*, weight_hh_l*_reverse] stacked to [D*3H, H];
 * b_hh is [D*3H]; gi is [T'*B, ldgi] with direction d at column d*3H; hseq (f32) and hseq_bf16 are [T'*B, ldh]
 * with direction d at column d*H (the bf16 copy is what the CTAs exchange between steps and the next layer's GEMM
 * operand); r,z,n,hn are [D][T'*B][H] (all NULL to skip).  Requires H % 64 == 0.  workspace: nsd_gru_tc_workspace.
 * Fused inter-layer dropout (model.py:55): if hdrop_bf16 != NULL it receives nsd_dropout(hseq_bf16, p_drop, seed)
 * (same mask, same rounding) as a second [T'*B, ldh] bf16 tensor -- the next layer's input in train mode.
 * Initial state (streaming inference, SURVEY 8f rank 3; D == 1, reverse0 == 0 only): h0 != NULL is [B, ldh] f32 and
 * hseq_bf16 must then hold T'*B + B rows whose FIRST B rows are bf16(h0); the states h_0..h_{T'-1} are written after
 * them.  h0 == NULL is the reference's zero initial state (model.py:104-117).
 * n_frames: per-row frame counts with the semantics of nsd_gru_fwd_f32 (hseq, hseq_bf16 and hdrop_bf16 are 0 at
 * t >= n_b; the saves there are not meaningful and the BPTT does not read them).  Not combinable with h0: NSD_ERR_INVALID. */
int nsd_gru_fwd_bf16(const float* gi, int ldgi, const void* w_hh_bf16, const float* b_hh, int Tp, int B, int H, int D,
                     int reverse0, float* hseq, void* hseq_bf16, int ldh, float* r, float* z, float* n, float* hn,
                     void* hdrop_bf16, float p_drop, uint64_t seed, const float* h0, const int* n_frames, void* workspace,
                     size_t workspace_bytes, void* stream);
/* BPTT of the above.  w_hhT_bf16 is the bf16 TRANSPOSE of each direction's W_hh stacked to [D*H, 3H].  Writes
 * dgi_bf16 = [dr~,dz~,dn~] and dgh_bf16 = [dr~,dz~,dn~*r], both [T'*B, ldg] bf16 with direction d at column d*3H.
 * p_drop > 0: dhseq is the gradient w.r.t. the DROPPED output (mask of nsd_dropout(., p_drop, seed) over the
 * contiguous [T'*B, lddh] tensor) and is masked/scaled on load.  db_ih/db_hh (both or neither; [D*3H] f32, overwritten):
 * the bias gradients = column sums of dgi / dgh over all T'*B rows, accumulated in fp32 before the bf16 rounding.
 * n_frames as in nsd_gru_bwd_f32: dgi and dgh are 0 at t >= n_b and the recurrent gradient into and out of those steps
 * is 0, so the bias sums cover the valid steps only. */
int nsd_gru_bwd_bf16(const float* dhseq, int lddh, const float* hseq, int ldh, const float* r, const float* z,
                     const float* n, const float* hn, const void* w_hhT_bf16, int Tp, int B, int H, int D, int reverse0,
                     void* dgi_bf16, void* dgh_bf16, int ldg, float p_drop, uint64_t seed, const int* n_frames, float* db_ih,
                     float* db_hh, void* workspace, size_t workspace_bytes, void* stream);
size_t nsd_gru_tc_workspace(int B, int H, int D);

/* inter-layer dropout (nn.GRU dropout=p, train mode, model.py:55): out = x * mask / (1-p),
 * mask from a counter-based generator keyed by (seed, element index); the backward is the
 * same call on the gradient.  Distributional, not bit, parity with torch's generator.   */
int nsd_dropout(const void* x, void* out, int dtype, size_t n, float p, uint64_t seed, void* stream);

/* ---- K4: CTC ----------------------------------------------------------------------
 * torch.nn.CTCLoss(blank, zero_infinity=True) forward AND gradient in one launch
 * (trainer:139-141, 213-218, 242).  `act` is addressed as act[t*st + b*sb + c*sc]; if
 * is_logits != 0 a log-softmax over c is applied first (trainer:210) and `grad` is
 * d/d logits, else `act` are log-probs and `grad` is what torch's ctc backward returns
 * w.r.t. log_probs.  grad uses the same strides as act and is fully overwritten
 * (zeros beyond in_len).  nll[b] is 0 for infeasible utterances.  loss_mean =
 * mean_b nll[b]/max(tgt_len[b],1) and grad is pre-scaled by 1/(max(tgt_len,1)*B) when
 * reduction_mean != 0; otherwise grad is unscaled (d nll[b]) and loss_mean = sum nll.
 * workspace: nsd_ctc_workspace bytes.                                              */
int nsd_ctc_loss(const float* act, int64_t st, int64_t sb, int64_t sc, int is_logits, const int32_t* targets,
                 int tgt_stride, const int32_t* in_lens, const int32_t* tgt_lens, int T, int B, int C,
                 int blank, int max_tgt, int reduction_mean, float* nll, float* loss, float* grad,
                 void* workspace, size_t workspace_bytes, void* stream);
size_t nsd_ctc_workspace(int T, int B, int C, int max_tgt);

/* out[r,:] = log_softmax(in[r,:]) for `rows` contiguous rows of C floats (trainer:210, 301). */
int nsd_log_softmax_f32(const float* in, float* out, int64_t rows, int C, void* stream);

/* ---- K5: greedy decode -----------------------------------------------------------
 * argmax over c (ties -> lowest index) for t < lens[b], collapse repeats, drop blank
 * (trainer:313-320).  out [B,T] int64 (first out_len[b] entries valid).             */
int nsd_greedy_decode(const float* act, int64_t st, int64_t sb, int64_t sc, const int32_t* lens, int T, int B,
                      int C, int blank, int64_t* out, int32_t* out_len, void* stream);
/* Levenshtein distance between decoded and true sequences, one warp per utterance
 * (edit_distance.SequenceMatcher.distance, trainer:322-330).  dist [B] int32.       */
int nsd_edit_distance(const int64_t* dec, int dec_stride, const int32_t* dec_len, const int32_t* tgt,
                      int tgt_stride, const int32_t* tgt_len, int B, int32_t* dist, void* workspace,
                      size_t workspace_bytes, void* stream);
size_t nsd_edit_distance_workspace(int B, int max_len);

/* ---- K5b: CTC prefix beam search with an optional phoneme-bigram prior -----------
 * New (the reference decodes greedily, trainer:313-320): N-best lists with scores for a downstream rescorer.  Log space,
 * a (+) b = logaddexp; per frame t < lens[b] (lens == NULL: all T) and beam entry l = (Pb, Pnb, prior):
 *   stay    Pb'(l) (+)= (Pb (+) Pnb) + y[blank];  Pnb'(l) (+)= Pnb + y[last(l)] (l non-empty);
 *   extend  Pnb'(l.c) (+)= (c == last(l) ? Pb : Pb (+) Pnb) + y[c] for c != blank; prior(l.c) = prior(l) + lm_weight *
 *           lm_logp[last(l) or blank][c] + insertion_bonus (lm_logp f32 [C][C] row = previous token, or NULL: bonus only);
 *   an extension whose prefix is already in the beam merges into that entry: Pnb' = (Pnb + y[last]) (+) extension;
 *   rank by total = (Pb' (+) Pnb') + prior, keep the best W (ties -> smaller key: stay of slot i = i*(C+1), extension
 *   by c = i*(C+1)+c+1), never a candidate at -inf; the beam is stored in rank order.
 * is_logits != 0: each row is log-softmaxed first (the arithmetic of nsd_log_softmax_f32).  act: [T][B][C] f32, strides
 * st/sb/sc in elements.  1 <= W <= 128, C <= 128.
 * The state (nsd_ctc_beam_state_bytes, set up by nsd_ctc_beam_init, re-initialisable in place) lives on the device: per
 * utterance the beam, a frame counter and an append-only prefix trie of 1 + W*max_frames nodes.  An advance takes no
 * argument that changes from call to call (graph replay), and any chunking of the same frames gives the same bits.  An
 * utterance whose frames_done + frames of this call would pass max_frames is left untouched and *err_flag (may be NULL)
 * is set to 1.  nsd_ctc_beam_nbest writes the best nbest <= W entries in rank order: hyps int64 [B][nbest][hyp_stride]
 * (hyp_stride >= max_frames; entries past hyp_len are -1), hyp_len i32, score = total and acoustic = Pb (+) Pnb (the CTC
 * prefix probability) f32 [B][nbest]; entries past the beam's size get length 0 and score -inf. */
size_t nsd_ctc_beam_state_bytes(int B, int W, int max_frames);
int nsd_ctc_beam_init(void* state, size_t state_bytes, int B, int W, int max_frames, void* stream);
/* nsd_ctc_beam_init for the utterances with mask[b] != 0 only (mask i32 [B] on the device); the others keep every byte. */
int nsd_ctc_beam_reset(void* state, size_t state_bytes, int B, int W, int max_frames, const int32_t* mask, void* stream);
int nsd_ctc_beam_advance(const float* act, int64_t st, int64_t sb, int64_t sc, int is_logits, const int32_t* lens, int T, int B,
                         int C, int blank, const float* lm_logp, float lm_weight, float insertion_bonus, int W, int max_frames,
                         void* state, size_t state_bytes, int* err_flag, void* stream);
int nsd_ctc_beam_nbest(const void* state, int B, int W, int max_frames, int nbest, int64_t* hyps, int hyp_stride, int32_t* hyp_len,
                       float* score, float* acoustic, void* stream);

/* ---- K5d: lexicon-constrained CTC beam search with a word n-gram LM (order <= 3) -------
 * K5b's beam whose phoneme prefixes spell words of a pronunciation lexicon: a transcript is pron(w1) sep pron(w2) sep ...
 * pron(wn) sep.  Classes [0, C), C <= 128; blank; sep != blank (40 = SIL in the competition's phone set).
 *   lexicon   a prefix tree over pronunciations (non-empty, without blank or sep), node 0 = root; a node is word-final if a
 *             pronunciation ends there; its words (homophones) are listed in ascending word id.
 *   slot      K5b's (Pb, Pnb, prior) plus lexicon node u, LM history (h2, h1) (start (-, bos)), word count and words: all
 *             functions of the phoneme prefix, so K5b's stay, merge and rank rules apply unchanged.
 *   extend    by c not in {blank, sep}: a candidate iff u has a child by c; u' = child, prior unchanged;
 *             by sep: a candidate iff u != root is word-final; w* = argmax over u's homophones of lm(w | h2, h1), ties -> the
 *             smaller word id (no LM: the smallest id); prior += lm_weight * lm(w* | h2, h1) + word_bonus; u' = root,
 *             history (h1, w*), w* appended to the words;
 *             anything else is no candidate (no sep at the root: no leading or doubled separator).
 *   LM        natural log, ARPA backoff: lm(w | a, b) = p3(a,b,w) if present, else bo2(a,b) (0 if the bigram is absent) +
 *             lm(w | b); lm(w | b) = p2(b,w) if present, else bo1(b) + p1(w).  lm_idx == NULL: no LM.
 * Arrays (device, trusted as built by the Python Lexicon / NgramLM):
 *   lex_nodes i32 [n_nodes][8], 16-byte aligned: child mask (4 words, bit c of word c/32), first child (children are
 *             consecutive in class order), first homophone entry, homophone count, 0;
 *   lex_words i32 [n_entries][2], 8-byte aligned: {word id, LM id of the word (its <unk> id if absent; any value without LM)};
 *   lm_idx    i32: b_off[V+1], b_word[n2], t_off[n2+1], t_word[n3] (bigrams of a at b_off[a]..b_off[a+1] sorted by word;
 *             trigrams of bigram j at t_off[j]..t_off[j+1] sorted by word);  lm_val f32: p1[V], bo1[V], p2[n2], bo2[n2], p3[n3].
 * The state block of an utterance is K5b's followed by the word fields and a word trie of 1 + W*max_frames nodes; advance,
 * reset, chunking, batch independence and the max_frames err_flag behave as in K5b.  sep == blank, sep or blank outside
 * [0, C) and bad sizes: NSD_ERR_INVALID.
 * nsd_ctc_word_beam_nbest (the state is not changed): final == 0 reads the beam as it stands; final != 0 adds the end term
 * and re-ranks by total, ties -> beam order: at the root lm_weight * lm(eos | h); at a word-final non-root node the pending
 * word's separator increment (same homophone rule) then lm_weight * lm(eos | h'); at any other node the entry gets score
 * and acoustic -inf and lengths 0.  Outputs as K5b's, plus words int64 [B][nbest][word_stride] (word_stride >=
 * max_frames/2 + 1, -1 past word_len; with final the pending word is included) and word_len i32 [B][nbest]. */
size_t nsd_ctc_word_beam_state_bytes(int B, int W, int max_frames);
int nsd_ctc_word_beam_init(void* state, size_t state_bytes, int B, int W, int max_frames, int lm_bos, void* stream);
int nsd_ctc_word_beam_reset(void* state, size_t state_bytes, int B, int W, int max_frames, int lm_bos, const int32_t* mask, void* stream);
int nsd_ctc_word_beam_advance(const float* act, int64_t st, int64_t sb, int64_t sc, int is_logits, const int32_t* lens, int T, int B,
                              int C, int blank, int sep, const int32_t* lex_nodes, int n_nodes, const int32_t* lex_words, int n_entries,
                              const int32_t* lm_idx, const float* lm_val, int lm_vocab, int lm_n2, int lm_n3, float lm_weight,
                              float word_bonus, int W, int max_frames, void* state, size_t state_bytes, int* err_flag, void* stream);
int nsd_ctc_word_beam_nbest(const void* state, int B, int W, int max_frames, const int32_t* lex_nodes, int n_nodes,
                            const int32_t* lex_words, int n_entries, const int32_t* lm_idx, const float* lm_val, int lm_vocab, int lm_n2,
                            int lm_n3, int lm_eos, float lm_weight, float word_bonus, int final, int nbest, int64_t* hyps, int hyp_stride,
                            int32_t* hyp_len, int64_t* words, int word_stride, int32_t* word_len, float* score, float* acoustic,
                            void* stream);
/* Live read-out of a K5d state for display while the utterance is still streaming; the state is not changed.  Live entries are
 * those with a finite total; their words are the completed ones (final == 0: no pending word).  Every later beam extends a live
 * entry, so the longest common prefix of the live entries' word-id sequences (compared by content, not by word-trie node) is a
 * prefix of every later hypothesis and of the final transcript: those words are committed.  reported i32 [B] (device) counts
 * the committed words already handed out; the caller zeroes it with the state (init, reset).  Per utterance b, out i32
 * [B][4 + cap]: {committed = the prefix length, first = reported[b] on entry, the top entry's word count, overflow}, then the
 * top entry's words first .. first + cap - 1 (-1 past its end).  Its words below `committed` are committed, the rest are
 * tentative.  reported[b] becomes min(committed, first + cap), so every committed word is handed out exactly once, ahead of the
 * tentative ones; overflow = 1 when the top entry's words past first do not fit cap.  No live entry: committed = first, word
 * count first, no words.  The cost grows with the words past first, not with the utterance; graph-capturable. */
int nsd_ctc_word_beam_live(const void* state, int B, int W, int max_frames, int32_t* reported, int cap, int32_t* out, void* stream);

/* ---- K5c: CTC forced alignment ---------------------------------------------------
 * New (no counterpart in the reference): the best path of each utterance through K4's blank-extended lattice, i.e. when each phoneme
 * of the true transcript happens and how well it is supported.  For utterance b:
 *   lattice   L = tgt_lens[b] clamped to [0, max_tgt], S' = 2L+1 states; ext[s] = blank for even s, targets[b*tgt_stride + s/2] for
 *             odd s.  il = in_lens[b] clamped to [0, T]; only frames t < il are used.  y_t[c] = act[t*st + b*sb + c*sc]; if
 *             is_logits != 0 each row is first log-softmaxed with the arithmetic of nsd_log_softmax_f32, so aligning logits is
 *             bit-identical to aligning log_softmax_tbc(logits).
 *   recursion (fp32)  d_0(0) = y_0[blank]; d_0(1) = y_0[ext[1]] if L > 0; every other d_0 is -inf;
 *             d_t(s) = max(d_{t-1}(s), d_{t-1}(s-1), d_{t-1}(s-2)) + y_t[ext[s]], the s-2 term only for odd s with ext[s] != ext[s-2].
 *   ties      among predecessors with equal d prefer s, then s-1, then s-2 (stay as long as possible).  The path ends at
 *             argmax(d_{il-1}(S'-1), d_{il-1}(S'-2)), on a tie at S'-1.  s_t is the path's state at frame t.
 *   outputs   (every element of every output is written)
 *             labels i32 [B][T]              ext[s_t] for t < il, else -1;
 *             frame_logp f32 [B][T]          y_t[labels[b][t]] for t < il, else 0;
 *             score f32 [B]                  the final d, which equals the fp32 left-to-right sum of frame_logp[b][0..il);
 *             spans i32 [B][max_tgt][2]      (first, last) frame of lattice state 2k+1, inclusive, for k < L (each token has at least
 *                                            one frame, its frames are contiguous); (-1, -1) for k >= L;
 *             token_logp f32 [B][max_tgt]    fp32 sum in frame order of frame_logp over span k for k < L; 0 for k >= L.
 *   infeasible  il < L + (number of k with targets[k] == targets[k-1]): score = -inf, labels -1, frame_logp 0, spans -1, token_logp 0.
 *             L = 0 gives the all-blank path; il = 0 with L = 0 gives score 0 (and labels -1).  If the best final d is -inf (act holds
 *             -inf) the outputs are the infeasible ones with score -inf; a NaN that reaches it gives score NaN and those outputs too.
 *   bad targets  a used target (k < L) equal to blank or outside [0, C) sets *err_flag = 1 (err_flag may be NULL); that utterance gets
 *             the infeasible outputs.  The other utterances are unaffected.
 * One CTA per utterance; no allocation and no host synchronisation (graph capture works); an utterance aligns identically alone or
 * inside any batch.  1 <= T <= 8192, 0 <= max_tgt <= 1024, tgt_stride >= max_tgt, C <= 128.  workspace: nsd_ctc_align_workspace bytes
 * (the 2-bit backpointer of every state and frame). */
size_t nsd_ctc_align_workspace(int T, int B, int C, int max_tgt);
int nsd_ctc_align(const float* act, int64_t st, int64_t sb, int64_t sc, int is_logits,
                  const int32_t* targets, int tgt_stride, const int32_t* in_lens, const int32_t* tgt_lens,
                  int T, int B, int C, int blank, int max_tgt,
                  int32_t* labels, float* frame_logp, int32_t* spans, float* token_logp, float* score,
                  int* err_flag, void* workspace, size_t workspace_bytes, void* stream);

/* ---- optimizer step (SURVEY 8f rank 1; inside the timed training step) ------------------
 * torch.optim.Adam semantics (trainer:163-169, 259): g = grad*grad_scale + weight_decay*p;
 * m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr/(1-b1^step) * m / (sqrt(v)/sqrt(1-b2^step) + eps).
 * params/grads/exp_avg/exp_avg_sq are HOST arrays of n_tensors DEVICE pointers (f32, contiguous),
 * numel a HOST array.  One launch per 48 tensors.  shadow_bf16 (NULL, or a HOST array whose entries
 * may be NULL): device pointer of a contiguous bf16 copy of the parameter, rewritten with the
 * updated value in the same pass (the tensor-core operand copy the next forward reads).       */
/* on != 0: the following nsd_adam_step launches are issued directly behind a recurrence kernel (nsd_gru_bwd_bf16) whose output they do not
 * need; they run under it on the SMs it leaves free and complete after it (programmatic dependent launch).  Set it back to 0 afterwards.
 * No counterpart in the reference (trainer:259 steps after the whole backward). */
int nsd_set_adam_late_wait(int on);
int nsd_adam_step(int n_tensors, void* const* params, const void* const* grads, void* const* exp_avg,
                  void* const* exp_avg_sq, const int64_t* numel, void* const* shadow_bf16, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int step, float grad_scale, void* stream);

/* Streaming inference push for B <= 8 (new: the reference's forward has no state API, model.py:104-119 always starts from
 * h0 = 0 and drops h_n).  ONE cooperative launch consumes S new bins and advances the whole unidirectional decoder by one
 * output frame: smoothing of the S bins that became computable (augmentations.py:91; left/right reach (ntaps-1)/2 and
 * ntaps-1-(ntaps-1)/2), day affine + softsign (model.py:89-93; bf16 operands, fp32 accumulate, like nsd_frontend_fwd's bf16
 * form), slide of the k/s patch (model.py:96-101), per layer l: gi = x_l W_ih^T + b_ih, gh = bf16(h_l) W_hh^T + b_hh, gates
 * r,z,n, h_l <- (1-z) n + z h_l (model.py:50-57, 119), logits = h_{L-1} fc_w^T + fc_b (model.py:122) and
 * ids[b] = argmax_c logits[b,c] (ties -> lowest index, trainer:314).  State carried between calls, all on the device:
 *   rawring f32 [B][ring_rows][N]  raw bins by absolute index mod ring_rows (ring_rows >= ntaps-1+2S);
 *   x0buf bf16 [2][B][N*K]         patch row of frame j in half (j & 1), feature order c*K + k;
 *   n_bins i32 [1]                 bins received so far (the launch adds S);   extra = n_bins - (S*j + K + right) in [0, S)
 *                                  for the newest emitted frame j (constant while every push is S bins);
 *   h f32 [L][B][H], h_bf16 [L][B][H]   state of every layer and its bf16 operand copy, updated in place.
 * bins_in f32 [B][S][N]; w_ih/w_hh/b_ih/b_hh: HOST arrays of L device pointers (bf16 [3H,in_l] / bf16 [3H,H] / f32 [3H] / f32
 * [3H], gate rows r|z|n); logits f32 [B,C]; ids i32 [B] or NULL; err_flag: set to 1 on a day index out of range.
 * H and N*K multiples of 512, N a multiple of 32, S <= 8, L <= 8. */
size_t nsd_stream_push_workspace(int B, int F0, int H, int L);
int nsd_stream_push(const float* bins_in, float* rawring, int ring_rows, const int64_t* day_idx, const float* day_w, const float* day_b,
                    int n_days, const float* taps, int ntaps, void* x0buf_bf16, int* n_bins, int extra, int B, int N, int K, int S, int H,
                    int L, int C, const void* const* w_ih_bf16, const void* const* w_hh_bf16, const void* const* b_ih,
                    const void* const* b_hh, float* h, void* h_bf16, const void* fc_w_bf16, const float* fc_b, float* logits, int* ids,
                    int* err_flag, void* workspace, size_t workspace_bytes, void* stream);

/* The same push with an independent stream per batch row (slot), for sessions that start, pause and end at different times.
 * Per-slot device state, read by the launch (so a graph replay takes no per-call argument):
 *   n_bins i32 [B]      bins the slot's current utterance received (the launch adds S to active slots);
 *   active i32 [B]      != 0: bins_in[b] holds the slot's next S bins; == 0: every byte of the slot's state is left as it is;
 *   last_frame i32 [B]  the last frame the utterance may emit (INT_MAX while streaming; the utterance's last frame when it ends);
 *   emitted i32 [B]     out: 1 if the slot emitted a frame in this push, else 0.
 * Every utterance starts at bin 0 (n_bins = 0, fresh h / h_bf16 = 0) and moves S bins per push.  With n = n_bins after the
 * push, a slot emits frame j = (n - K - right) / S once n >= K + right and j <= last_frame: one frame per push after a
 * warm-up of (K + right) / S pushes, during which only the ring and the patch row move.  Patch rows before bin 0 are zeros,
 * and the ring is read only at bins this utterance wrote, so neither needs clearing between utterances.  Only emitting rows
 * update h / h_bf16 and write logits and ids (ids = -1 for the others); a push in which no row emits skips the stack.  A row's
 * results do not depend on B, on the other slots or on when its utterance started. */
int nsd_stream_push_slots(const float* bins_in, float* rawring, int ring_rows, const int64_t* day_idx, const float* day_w, const float* day_b,
                          int n_days, const float* taps, int ntaps, void* x0buf_bf16, int* n_bins, const int* active, const int* last_frame,
                          int* emitted, int B, int N, int K, int S, int H, int L, int C, const void* const* w_ih_bf16,
                          const void* const* w_hh_bf16, const void* const* b_ih, const void* const* b_hh, float* h, void* h_bf16,
                          const void* fc_w_bf16, const float* fc_b, float* logits, int* ids, int* err_flag, void* workspace,
                          size_t workspace_bytes, void* stream);

/* Device-resident seed offset (uint64, or NULL to clear): added to the seed argument of every Conformer kernel that draws a mask and of
 * nsd_input_noise at RUN time, so that a captured CUDA graph of the training step (neural_decoder_trainer.py:181-260 as one replay)
 * sees fresh dropout / DropPath / noise on every replay.  Host-side state, takes effect at the next launch. */
int nsd_set_seed_offset_ptr(const void* dev_u64);

/* ==== Conformer path (BASELINE configs[2]; reference src/neural_decoder/transformer_ctc.py:333-501 and the transformer branch of
 * neural_decoder_trainer.py:137-162, 206-260).  Activations are row-major [rows = B*T', D] f32 (batch-major rows b*T' + t);
 * every kernel that feeds a tensor-core GEMM can also emit the bf16 operand copy.  Stochastic regularisers are counter-based
 * masks keyed by (seed, element index) -- distributional, not bit, parity with torch's generator; the backward regenerates them.
 * act codes: 0 identity, 1 SiLU, 2 GELU (erf form), 3 ReLU. ================================================================== */

/* y = dropout_p(act(LayerNorm(x) * gamma + beta)); nn.LayerNorm(eps) over the last dimension (transformer_ctc.py:97, 156, 167,
 * 202, 212, 219, 231, 411), optionally followed by SiLU (:168) or GELU + Dropout (:412-413).  mean/rstd [M] are saved for the
 * backward.  y_f32 and/or y_bf16.  D % 4 == 0, D <= 2048. */
int nsd_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, int act, float p_drop, uint64_t seed, float* y_f32,
                      void* y_bf16, float* mean, float* rstd, int M, int D, void* stream);
/* dx, dgamma, dbeta of the above (dgamma/dbeta overwritten; two fixed-order stages: deterministic).  dx_addend (NULL or f32 [M,D]) is added to
 * dx: the gradient that reaches x around the LayerNorm in a pre-LN residual block (x + f(LN(x)), transformer_ctc.py:245-257), fused here. */
int nsd_layernorm_bwd(const void* dy, int dy_dtype, const float* x, const float* gamma, const float* beta, const float* mean, const float* rstd, int act,
                      float p_drop, uint64_t seed, const float* dx_addend, float* dx, float* dgamma, float* dbeta, int M, int D, void* workspace,
                      size_t workspace_bytes, void* stream);
size_t nsd_layernorm_bwd_workspace(int M, int D);
/* y = dropout_p(act(x)) over n contiguous elements (n % 4 == 0): SiLU + Dropout of the feed-forward modules (transformer_ctc.py:204-205,
 * 223-224), ReLU of the bottleneck MLP (:140); and its backward dx = dy * mask/(1-p) * act'(x). */
int nsd_act_fwd(const float* x, int act, float p_drop, uint64_t seed, float* y_f32, void* y_bf16, size_t n, void* stream);
int nsd_act_bwd(const void* dy, int dy_dtype, const float* x, int act, float p_drop, uint64_t seed, float* dx, size_t n, void* stream);
/* nn.GLU(dim=-1) (transformer_ctc.py:160, 179): g[M,D] = u[:, :D] * sigmoid(u[:, D:]) for u [M, 2D]; and its backward. */
int nsd_glu_fwd(const float* u, float* g, int M, int D, void* stream);
int nsd_glu_bwd(const float* dg, const float* u, float* du, int M, int D, void* stream);
/* out = x + scale * DropPath_{p_path}(dropout_{p_drop}(y)) (transformer_ctc.py:14-23, 190, 245, 251, 257; DropPath keeps a whole sample,
 * sample = elems_per_sample consecutive elements).  x == NULL gives the gradient w.r.t. y when y holds d(out). */
int nsd_residual(const float* x, const float* y, float scale, float p_drop, uint64_t seed, float p_path, uint64_t path_seed, int64_t elems_per_sample,
                 float* out, size_t n, void* stream);
/* Depthwise convolution over time inside each utterance, zero padding k/2 (nn.Conv1d(groups=D, padding=k//2), transformer_ctc.py:162-166, 183;
 * the Gaussian smoothing F.conv1d(groups=C, padding=k//2) :104-109 with w_shared != 0: one [k] tap vector for all channels):
 * y[b,t,d] = bias[d] + sum_j w[d][j] x[b, t+j-k/2, d]; flip != 0 uses w[d][k-1-j] (the data gradient).  x,y [B,T,D]; odd k <= 32. */
int nsd_dwconv_fwd(const float* x, const float* w, const float* bias, float* y, int B, int T, int D, int k, int flip, int w_shared, void* stream);
/* dw[d][j] = sum_{b,t} dy[b,t,d] x[b,t+j-k/2,d]; db[d] = sum dy (db may be NULL). */
int nsd_dwconv_bwd_w(const float* dy, const float* x, float* dw, float* db, int B, int T, int D, int k, void* workspace, size_t workspace_bytes, void* stream);
size_t nsd_dwconv_bwd_w_workspace(int B, int D, int k);
/* Strided depthwise convolution without padding or bias (NeuralFrontend.temporal_conv, transformer_ctc.py:81-91, 112-114):
 * y[b,j,c] = sum_k w[c][k] x[b, j*S+k, c], j < (T-K)/S+1; x [B,T,N] -> y [B,T',N] (f32 and/or bf16).  Backward: dx [B,T,N] and dw [N,K]. */
int nsd_strided_dwconv_fwd(const float* x, const float* w, float* y_f32, void* y_bf16, int B, int T, int N, int K, int S, void* stream);
int nsd_strided_dwconv_bwd(const float* dy, const float* x, const float* w, float* dx, float* dw, int B, int T, int N, int K, int S, void* workspace,
                           size_t workspace_bytes, void* stream);
size_t nsd_strided_dwconv_bwd_workspace(int B, int N, int K);
/* SpecAugment + positional encoding (transformer_ctc.py:266-308, 311-330, 467-471): out[b,t,d] = (in a masked band ? 0 : z[b,t,d]) + pe[t,d].
 * bands8 (HOST) = {f0,f1, f0,f1, t0,t1, t0,t1}: feature / frame intervals [lo,hi) set to zero for every utterance (empty: lo >= hi).
 * pe == NULL: no addition (the backward: dz = band-masked dout).  bands8_dev != NULL: the eight bounds are read from DEVICE memory
 * instead (a captured CUDA graph of the training step draws new bands for every replay). */
int nsd_posenc_mask(const float* z, const float* pe, const int* bands8, const int* bands8_dev, float* out, int B, int T, int D, void* stream);
/* dst = bf16(src) (row stride ld_dst) and colsum[n] = sum_m src[m,n] from one read of the f32 [M,N] gradient: the operand copy and the
 * bias gradient of an nn.Linear backward.  N % 4 == 0; two fixed-order stages. */
int nsd_cast_colsum(const float* src, int M, int N, void* dst_bf16, int ld_dst, float* colsum, void* workspace, size_t workspace_bytes, void* stream);
size_t nsd_cast_colsum_workspace(int M, int N);
/* Strided batched GEMM  C_z[M,N] = alpha * A_z[M,K] B_z[K,N] (+ bias_z[N]),  z = (z0 < nb0, z1 < nb1):
 *   A_z(m,k) = A[z0*a_b0 + z1*a_b1 + m*a_rs + k*a_cs],  B_z(k,n) = B[zb*b_b0 + z1*b_b1 + k*b_rs + n*b_cs],  zb = b_index ? b_index[z0] : z0,
 *   C_z(m,n) = C[z0*c_b0 + z1*c_b1 + m*c_rs + n],  bias_z = bias + zb*bias_b0  (strides in elements).
 * The attention products of nn.MultiheadAttention (transformer_ctc.py:216, 250: Q K^T, P V and their four gradients, read in place from the
 * packed [B*T', 3D] projection) and the per-day affine x W[day] + b[day] (transformer_ctc.py:41-49; b_index = day ids) and its gradients.
 * tc_mode < 0: any bf16 operand -> mma.sync tensor-core path (operands rounded to bf16 in shared memory, fp32 accumulate), all-f32
 * operands -> FFMA parity path; tc_mode = 1 / 0 forces the tensor-core / FFMA path. */
int nsd_bgemm(const void* A, int a_dtype, int64_t a_rs, int64_t a_cs, int64_t a_b0, int64_t a_b1, const void* B, int b_dtype, int64_t b_rs, int64_t b_cs,
              int64_t b_b0, int64_t b_b1, const int64_t* b_index, void* C, int c_dtype, int64_t c_rs, int64_t c_b0, int64_t c_b1, const float* bias,
              int64_t bias_b0, int M, int N, int K, int nb0, int nb1, float alpha, int tc_mode, void* stream);
/* Attention weights: S [B*H*T rows of T scores, row stride ld >= T (a multiple of 8 keeps the rows 16-byte aligned for nsd_bgemm;
 * the padding columns are written as zeros)] f32, in place -> P = softmax over the keys j < lens[b] (key_padding_mask, transformer_ctc.py:250, 475-477;
 * lens == NULL: no mask); Pd (optional, f32 or bf16) = dropout_p(P) (nn.MultiheadAttention(dropout=p), :216).  Backward: dPd (in place) -> dS. */
int nsd_softmax_mask_fwd(float* S, void* Pd, int pd_dtype, const int32_t* lens, int B, int H, int T, int ld, float p_drop, uint64_t seed, void* stream);
int nsd_softmax_mask_bwd(const float* P, float* dPd, int B, int H, int T, int ld, float p_drop, uint64_t seed, void* stream);
/* out[d, :] = sum of partial[b, :] over the rows b with index[b] == d, in row order (index_select backward for day_weights / day_bias). */
int nsd_index_reduce(const float* partial, const int64_t* index, int B, size_t n, int n_out, float* out, void* stream);
/* y = a*x + b;  *out = (accumulate ? *out : 0) + scale * sum(x) + add (one CTA, fixed order: the KL term of the label-smoothed loss, trainer:235-240);
 * dlogits = dlp - exp(lp) * sum_c dlp (log_softmax backward, rows of C). */
int nsd_axpb(const float* x, float a, float b, float* y, size_t n, void* stream);
int nsd_sum_f32(const float* x, size_t n, float scale, float add, int accumulate, float* out, void* stream);
int nsd_log_softmax_bwd(const float* lp, const float* dlp, float* dlogits, int64_t rows, int C, void* stream);
/* *out = sum over all listed tensors of g^2 (clip_grad_norm_, trainer:255-257); HOST pointer tables; fixed-order two-stage reduction. */
int nsd_sqnorm_multi(int n_tensors, const void* const* grads, const int64_t* numel, float* out, void* workspace, size_t workspace_bytes, void* stream);
size_t nsd_sqnorm_workspace(int n_tensors, const int64_t* numel);
/* torch.optim.AdamW semantics (trainer:144-151): p *= 1 - lr*wd; m,v EMA of g*grad_scale*clip; p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps).
 * grad_sqnorm != NULL (device scalar from nsd_sqnorm_multi): clip = min(1, max_norm / (sqrt(*grad_sqnorm)*grad_scale + 1e-6)) without a host
 * synchronisation.  hyper_dev != NULL (device float[3] = {lr/(1-b1^t), 1/sqrt(1-b2^t), 1-lr*wd}) overrides the values derived from lr / step /
 * weight_decay: the schedule of a replayed CUDA graph.  Same tables and bf16 shadow rewrite as nsd_adam_step. */
int nsd_adamw_step(int n_tensors, void* const* params, const void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
                   const int64_t* numel, void* const* shadow_bf16, float lr, float beta1, float beta2, float eps, float weight_decay, int step,
                   float grad_scale, const float* grad_sqnorm, float max_norm, const float* hyper_dev, void* stream);

/* Keep n_sms SMs free of the persistent tensor-core GEMM grids from now on (0 = use every SM).  New (no reference
 * counterpart): while parallel.GradSync has a gradient bucket in flight, NCCL's CTAs run on the reserved SMs instead of
 * displacing CTAs of a 148-wide persistent GEMM.  Host-side state, takes effect at the next nsd_gemm_bf16* call. */
int nsd_set_gemm_sm_reserve(int n_sms);

/* n small f32 vectors copied src[i] -> dst[i] (numel[i] elements) in one launch: packs the per-direction nn.GRU bias
 * vectors (model.py:50-57: bias_ih_l{k}[_reverse], bias_hh_l{k}[_reverse]) side by side for the two-direction launches. */
int nsd_multi_copy_f32(int n_tensors, const void* const* src, void* const* dst, const int64_t* numel, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NSD_B200_H */
