"""Tensor-level wrappers of the C-ABI entry points (no autograd here).

Each function allocates its outputs with torch (caching allocator, current
stream) and passes raw device pointers to ``libnsd_b200.so``.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import call, ptr, stream, dtype_code, require_cuda


def n_frames(T: int, kernel_len: int, stride_len: int) -> int:
    if T < kernel_len:
        # nn.Unfold raises RuntimeError for an input shorter than the kernel (model.py:96-101)
        raise RuntimeError(f"sequence length {T} is shorter than kernelLen {kernel_len}")
    return (T - kernel_len) // stride_len + 1


# ------------------------------------------------------------------ K1
def frontend_fwd(x, day_idx, day_w, day_b, taps, kernel_len, stride_len, out_dtype, err_flag=None, noise=None, *, x_len=None):
    """-> (patches [T'*B, N*K] time-major, ys [B,T,N], z [B,T,N]).  ``noise`` = (whiteNoiseSD, constantOffsetSD, seed)
    fuses the trainer's in-loop augmentation (trainer:194-201) into the read of x.  ``x_len`` (int64 [B], device): bins
    t >= x_len[b] are read as 0, after the noise."""
    require_cuda(x, "neuralInput")
    B, T, N = x.shape
    Tp = n_frames(T, kernel_len, stride_len)
    x = x.contiguous().float()
    day_idx = day_idx.to(device=x.device, dtype=torch.int64).contiguous()
    ys = torch.empty_like(x)
    z = torch.empty_like(x)
    patches = torch.empty((Tp * B, N * kernel_len), device=x.device, dtype=out_dtype)
    call("nsd_frontend_fwd", ptr(x), ptr(day_idx), ptr(day_w), ptr(day_b), ptr(taps), taps.numel(), B, T, N,
         day_w.shape[0], kernel_len, stride_len, ptr(ys), ptr(z), ptr(patches), dtype_code(out_dtype),
         ptr(err_flag), float(noise[0]) if noise else 0.0, float(noise[1]) if noise else 0.0, int(noise[2]) if noise else 0,
         ptr(_lengths(x_len, B)), stream())
    return patches, ys, z


def _lengths(x_len, B):
    if x_len is not None:
        assert x_len.is_cuda and x_len.dtype == torch.int64 and x_len.is_contiguous() and x_len.shape == (B,)
    return x_len


def frame_counts(x_len, T: int, kernel_len: int, stride_len: int, err_flag=None):
    """-> n_frames int32 [B] on the device: floor((x_len - kernel_len) / stride_len) + 1 clamped to [0, T'], the frames whose
    whole window lies inside each utterance (no host synchronisation).  A length outside [kernel_len, T] sets bit 2 of
    ``err_flag``."""
    B = x_len.shape[0]
    _lengths(x_len, B)
    n = torch.empty(B, device=x_len.device, dtype=torch.int32)
    call("nsd_frame_counts", ptr(x_len), B, T, kernel_len, stride_len, ptr(n), ptr(err_flag), stream())
    return n


def _frames(n_frames, B):
    if n_frames is not None:
        assert n_frames.is_cuda and n_frames.dtype == torch.int32 and n_frames.is_contiguous() and n_frames.shape == (B,)
    return n_frames


def input_noise(x, white_noise_sd: float, constant_offset_sd: float, seed: int, out=None):
    """x + N(0,1)*whiteNoiseSD + N(0,1)[B,1,N]*constantOffsetSD (trainer:194-201) in one pass; the values the fused
    front end uses for the same seed."""
    require_cuda(x, "X")
    assert x.dim() == 3 and x.dtype == torch.float32 and x.is_contiguous()
    out = torch.empty_like(x) if out is None else out
    B, T, N = x.shape
    call("nsd_input_noise", ptr(x), ptr(out), B, T, N, float(white_noise_sd), float(constant_offset_sd), int(seed), stream())
    return out


def frontend_bwd(dpatches, ys, z, day_idx, n_days, kernel_len, stride_len):
    B, T, N = ys.shape
    flat = torch.empty(n_days * N * N + n_days * N, device=ys.device, dtype=torch.float32)   # one gradient bucket
    d_w = flat[:n_days * N * N].view(n_days, N, N)
    d_b = flat[n_days * N * N:].view(n_days, 1, N)
    nbytes = _lib.lib().nsd_frontend_bwd_workspace(B, N)
    ws = torch.empty(nbytes, device=ys.device, dtype=torch.uint8)
    call("nsd_frontend_bwd", ptr(dpatches), dtype_code(dpatches.dtype), ptr(ys), ptr(z), ptr(day_idx), B, T, N,
         n_days, kernel_len, stride_len, ptr(d_w), ptr(d_b), ptr(ws), nbytes, stream())
    return d_w, d_b


def frontend_bwd_input(dpatches, z, day_idx, day_w, taps, kernel_len, stride_len, *, x_len=None):
    """-> dx [B,T,N] f32: the gradient w.r.t. the front end's input X of the patches' gradient ``dpatches`` [T'*B, N*K].
    ``x_len`` (as given to ``frontend_fwd``): dx is 0 at bins t >= x_len[b]."""
    B, T, N = z.shape
    dx = torch.empty((B, T, N), device=z.device, dtype=torch.float32)
    call("nsd_frontend_bwd_input", ptr(dpatches), dtype_code(dpatches.dtype), ptr(z), ptr(day_idx), ptr(day_w), ptr(taps), taps.numel(),
         B, T, N, day_w.shape[0], kernel_len, stride_len, ptr(dx), ptr(_lengths(x_len, B)), stream())
    return dx


# ------------------------------------------------------------------ K2
def gemm(transa: bool, transb: bool, M: int, N: int, K: int, A, lda: int, B, ldb: int, C, ldc: int,
         bias: Optional[torch.Tensor] = None, beta: float = 0.0, a_off: int = 0, b_off: int = 0, c_off: int = 0):
    """C[M,N] = op(A) op(B) (+bias) (+beta*C); element offsets select sub-matrices of the buffers."""
    esz_a, esz_b, esz_c = A.element_size(), B.element_size(), C.element_size()
    pa, pb, pc = A.data_ptr() + a_off * esz_a, B.data_ptr() + b_off * esz_b, C.data_ptr() + c_off * esz_c
    if A.dtype == torch.float32:
        call("nsd_gemm_f32", int(transa), int(transb), M, N, K, pa, lda, pb, ldb, pc, ldc, ptr(bias), beta, stream())
    else:
        call("nsd_gemm_bf16", int(transa), int(transb), M, N, K, pa, lda, pb, ldb, pc, ldc, dtype_code(C.dtype),
             ptr(bias), beta, stream())


def gemm_x2(transa: bool, transb: bool, M: int, N: int, K: int, A, lda: int, B, ldb: int, C, ldc: int, a_offs, b_offs, c_offs):
    """Two bf16 GEMMs of identical shape in ONE launch: problem i reads A / B / writes C at element offsets a_offs[i] /
    b_offs[i] / c_offs[i] of the same three buffers (the two directions' W_hh weight gradients)."""
    ea, eb, ec = A.element_size(), B.element_size(), C.element_size()
    call("nsd_gemm_bf16_x2", int(transa), int(transb), M, N, K, A.data_ptr() + a_offs[0] * ea, A.data_ptr() + a_offs[1] * ea, lda,
         B.data_ptr() + b_offs[0] * eb, B.data_ptr() + b_offs[1] * eb, ldb, C.data_ptr() + c_offs[0] * ec, C.data_ptr() + c_offs[1] * ec, ldc,
         dtype_code(C.dtype), stream())


def colsum(a, M: int, N: int, lda: int, out, a_off: int = 0, out_off: int = 0):
    nbytes = _lib.lib().nsd_colsum_workspace(N)
    ws = torch.empty(nbytes, device=a.device, dtype=torch.uint8)
    call("nsd_colsum", a.data_ptr() + a_off * a.element_size(), dtype_code(a.dtype), M, N, lda,
         out.data_ptr() + out_off * 4, ptr(ws), nbytes, stream())


def cast(src, dst_dtype):
    dst = torch.empty(src.shape, device=src.device, dtype=dst_dtype)
    call("nsd_cast", ptr(src), dtype_code(src.dtype), ptr(dst), dtype_code(dst_dtype), src.numel(), stream())
    return dst


def cast_transpose(src, want_copy: bool, want_t: bool):
    """bf16 copy and/or bf16 transpose of a 2-D row-major tensor (last dim contiguous; row stride free)."""
    R, Cn = src.shape
    assert src.stride(1) == 1
    dst = torch.empty((R, Cn), device=src.device, dtype=torch.bfloat16) if want_copy else None
    dstT = torch.empty((Cn, R), device=src.device, dtype=torch.bfloat16) if want_t else None
    call("nsd_cast_transpose", ptr(src), dtype_code(src.dtype), R, Cn, src.stride(0), ptr(dst), Cn, ptr(dstT), R, stream())
    return dst, dstT


def cast_transpose_into(src, dst, dstT):
    """bf16 copy (dst [R,C] view) and/or bf16 transpose (dstT [C,R] view) of a 2-D view; unit inner strides."""
    R, Cn = src.shape
    assert src.stride(1) == 1 and (dst is None or dst.stride(1) == 1) and (dstT is None or dstT.stride(1) == 1)
    call("nsd_cast_transpose", ptr(src), dtype_code(src.dtype), R, Cn, src.stride(0), ptr(dst),
         dst.stride(0) if dst is not None else 0, ptr(dstT), dstT.stride(0) if dstT is not None else 0, stream())


def transpose_bf16_multi(srcs, dstTs):
    """dstTs[i] [C,R] <- srcs[i]^T for equally shaped bf16 2-D views with unit inner strides and equal row strides, in one launch."""
    import ctypes as C
    n = len(srcs)
    if n == 0:
        return
    R, Cn = srcs[0].shape
    for s_, d_ in zip(srcs, dstTs):
        assert s_.dtype == torch.bfloat16 and d_.dtype == torch.bfloat16 and tuple(s_.shape) == (R, Cn) and tuple(d_.shape) == (Cn, R)
        assert s_.stride(1) == 1 and d_.stride(1) == 1 and s_.stride(0) == srcs[0].stride(0) and d_.stride(0) == dstTs[0].stride(0)
    arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    call("nsd_transpose_bf16_multi", n, arr(srcs), arr(dstTs), R, Cn, srcs[0].stride(0), dstTs[0].stride(0), stream())


def swap01(x):
    """[D0,D1,C] -> contiguous [D1,D0,C]."""
    D0, D1, Cc = x.shape
    out = torch.empty((D1, D0, Cc), device=x.device, dtype=torch.float32)
    call("nsd_swap01_f32", ptr(x), ptr(out), D0, D1, Cc, stream())
    return out


# ------------------------------------------------------------------ K3
def gru_fwd_f32(gi, ldgi, gi_off, w_hh, b_hh, Tp, B, H, reverse, hseq, ldh, h_off, saves, *, n_frames=None):
    """``n_frames`` (int32 [B], device; ``frame_counts``): row b runs its own frames only, as nn.GRU on a packed sequence,
    and its output is 0 at t >= n_frames[b]."""
    r, z, n, hn = saves if saves is not None else (None, None, None, None)
    call("nsd_gru_fwd_f32", gi.data_ptr() + gi_off * 4, ldgi, ptr(w_hh), ptr(b_hh), Tp, B, H, int(reverse),
         hseq.data_ptr() + h_off * 4, ldh, ptr(r), ptr(z), ptr(n), ptr(hn), ptr(_frames(n_frames, B)), stream())


def gru_bwd_f32(dhseq, lddh, dh_off, hseq, ldh, h_off, saves, w_hh, Tp, B, H, reverse, dgi, ldgi, dgi_off, dghn, *, n_frames=None):
    r, z, n, hn = saves
    nbytes = _lib.lib().nsd_gru_bwd_workspace(B, H)
    ws = torch.empty(nbytes, device=dgi.device, dtype=torch.uint8)
    call("nsd_gru_bwd_f32", dhseq.data_ptr() + dh_off * 4, lddh, hseq.data_ptr() + h_off * 4, ldh, ptr(r), ptr(z),
         ptr(n), ptr(hn), ptr(w_hh), Tp, B, H, int(reverse), dgi.data_ptr() + dgi_off * 4, ldgi, ptr(dghn),
         ptr(_frames(n_frames, B)), ptr(ws), nbytes, stream())


def gru_fwd_bf16(gi, w_hh_bf, b_hh, Tp, B, H, D, reverse0, want_saves, p_drop: float = 0.0, seed: int = 0, h0=None, *,
                 n_frames=None):
    """-> (hseq f32 [Tp*B, D*H], hseq bf16, saves (r,z,n,hn) each [D,Tp*B,H] or None[, dropped bf16 copy if p_drop > 0]).
    ``h0`` ([B, H] f32, one forward direction only): initial state instead of the reference's zeros (streaming).
    ``n_frames`` (int32 [B], device; not with ``h0``): packed-sequence rows, as in ``gru_fwd_f32``."""
    dev = gi.device
    M = Tp * B
    hseq = torch.empty((M, D * H), device=dev, dtype=torch.float32)
    if h0 is not None:
        assert D == 1 and not reverse0 and h0.shape == (B, H) and h0.dtype == torch.float32 and h0.is_contiguous()
        full_bf = torch.empty((M + B, H), device=dev, dtype=torch.bfloat16)
        call("nsd_cast", ptr(h0), dtype_code(h0.dtype), ptr(full_bf), dtype_code(torch.bfloat16), h0.numel(), stream())
        hseq_bf = full_bf[B:]
    else:
        full_bf = hseq_bf = torch.empty((M, D * H), device=dev, dtype=torch.bfloat16)
    sv = tuple(torch.empty((D, M, H), device=dev, dtype=torch.float32) for _ in range(4)) if want_saves else (None,) * 4
    nbytes = _lib.lib().nsd_gru_tc_workspace(B, H, D)
    ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    hdrop = torch.empty_like(hseq_bf) if p_drop > 0 else None
    call("nsd_gru_fwd_bf16", ptr(gi), gi.stride(0), ptr(w_hh_bf), ptr(b_hh), Tp, B, H, D, int(reverse0), ptr(hseq),
         ptr(full_bf), D * H, ptr(sv[0]), ptr(sv[1]), ptr(sv[2]), ptr(sv[3]), ptr(hdrop), float(p_drop), int(seed),
         ptr(h0), ptr(_frames(n_frames, B)), ptr(ws), nbytes, stream())
    if p_drop > 0:
        return hseq, hseq_bf, (sv if want_saves else None), hdrop
    return hseq, hseq_bf, (sv if want_saves else None)


def gru_bwd_bf16(dhseq, hseq, saves, w_hhT_bf, Tp, B, H, D, reverse0, p_drop: float = 0.0, seed: int = 0, db_ih=None, db_hh=None, *,
                 n_frames=None):
    """-> (dgi bf16 [Tp*B, D*3H] = [dr~,dz~,dn~], dgh bf16 = [dr~,dz~,dn~*r]).  p_drop > 0 masks dhseq like
    nsd_dropout(dhseq, p_drop, seed); db_ih / db_hh (f32 [D*3H]) receive the bias gradients.  ``n_frames``: no gradient
    flows through t >= n_frames[b] (dgi, dgh are 0 there)."""
    dev = dhseq.device
    M = Tp * B
    dgi = torch.empty((M, D * 3 * H), device=dev, dtype=torch.bfloat16)
    dgh = torch.empty((M, D * 3 * H), device=dev, dtype=torch.bfloat16)
    nbytes = _lib.lib().nsd_gru_tc_workspace(B, H, D)
    ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    r, z, n, hn = saves
    call("nsd_gru_bwd_bf16", ptr(dhseq), dhseq.stride(0), ptr(hseq), hseq.stride(0), ptr(r), ptr(z), ptr(n), ptr(hn),
         ptr(w_hhT_bf), Tp, B, H, D, int(reverse0), ptr(dgi), ptr(dgh), D * 3 * H, float(p_drop), int(seed),
         ptr(_frames(n_frames, B)), ptr(db_ih), ptr(db_hh), ptr(ws), nbytes, stream())
    return dgi, dgh


def dropout(x, p: float, seed: int):
    out = torch.empty_like(x)
    call("nsd_dropout", ptr(x), ptr(out), dtype_code(x.dtype), x.numel(), float(p), int(seed), stream())
    return out


# ------------------------------------------------------------------ K4 / K5
def ctc_loss_raw(act, st, sb, sc, is_logits, targets, in_lens, tgt_lens, T, B, Cc, blank, reduction_mean, want_grad):
    """Returns (loss scalar tensor, nll [B], grad or None).  grad has the memory layout (strides) of ``act``."""
    dev = act.device
    max_tgt = targets.shape[1]
    nll = torch.empty(B, device=dev, dtype=torch.float32)
    loss = torch.empty((), device=dev, dtype=torch.float32)
    grad = torch.empty_like(act) if want_grad else None
    nbytes = _lib.lib().nsd_ctc_workspace(T, B, Cc, max_tgt)
    ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    call("nsd_ctc_loss", ptr(act), st, sb, sc, int(is_logits), ptr(targets), targets.stride(0), ptr(in_lens),
         ptr(tgt_lens), T, B, Cc, blank, max_tgt, int(reduction_mean), ptr(nll), ptr(loss), ptr(grad), ptr(ws),
         nbytes, stream())
    return loss, nll, grad


def ctc_align_raw(act, st, sb, sc, is_logits, targets, in_lens, tgt_lens, T, B, Cc, blank, err_flag):
    """K5c forced alignment -> (labels i32 [B,T], frame_logp f32 [B,T], spans i32 [B,S,2], token_logp f32 [B,S], score f32 [B]) with
    S = targets.shape[1]; ``err_flag`` (i32 [1], zeroed by the caller) is set to 1 on a target equal to blank or outside [0, C)."""
    dev = act.device
    max_tgt = targets.shape[1]
    labels = torch.empty((B, T), device=dev, dtype=torch.int32)
    frame_logp = torch.empty((B, T), device=dev, dtype=torch.float32)
    spans = torch.empty((B, max_tgt, 2), device=dev, dtype=torch.int32)
    token_logp = torch.empty((B, max_tgt), device=dev, dtype=torch.float32)
    score = torch.empty(B, device=dev, dtype=torch.float32)
    nbytes = _lib.lib().nsd_ctc_align_workspace(T, B, Cc, max_tgt)
    ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    call("nsd_ctc_align", ptr(act), st, sb, sc, int(is_logits), ptr(targets), targets.stride(0), ptr(in_lens), ptr(tgt_lens), T, B, Cc,
         blank, max_tgt, ptr(labels), ptr(frame_logp), ptr(spans), ptr(token_logp), ptr(score), ptr(err_flag), ptr(ws), nbytes, stream())
    return labels, frame_logp, spans, token_logp, score


def log_softmax(x):
    """Row-wise log-softmax over the last dim of a contiguous f32 tensor."""
    out = torch.empty_like(x)
    Cc = x.shape[-1]
    call("nsd_log_softmax_f32", ptr(x), ptr(out), x.numel() // Cc, Cc, stream())
    return out


def adam_step(params, grads, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0, shadows=None, under_recurrence=False):
    """torch.optim.Adam (L2-in-gradient, not AdamW) on a list of f32 tensors in as few launches as possible.
    ``shadows``: optional list (entries may be None) of contiguous bf16 tensors rewritten with the updated parameters."""
    import ctypes as C
    n = len(params)
    if n == 0:
        return
    arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    numel = (C.c_int64 * n)(*[t.numel() for t in params])
    sh = None
    if shadows is not None and any(s is not None for s in shadows):
        for s_, p_ in zip(shadows, params):
            assert s_ is None or (s_.is_contiguous() and s_.dtype == torch.bfloat16 and s_.numel() == p_.numel())
        sh = (C.c_void_p * n)(*[None if s_ is None else s_.data_ptr() for s_ in shadows])
    if under_recurrence:       # issued directly behind a K3 launch whose output it does not need: runs under it (nsd_set_adam_late_wait)
        call("nsd_set_adam_late_wait", 1)
    try:
        call("nsd_adam_step", n, arr(params), arr(grads), arr(exp_avg), arr(exp_avg_sq), numel, sh, float(lr), float(beta1),
             float(beta2), float(eps), float(weight_decay), int(step), float(grad_scale), stream())
    finally:
        if under_recurrence:
            call("nsd_set_adam_late_wait", 0)


def stream_push(bins_in, rawring, day, day_w, day_b, taps, x0buf, n_bins, extra, K, S, w_ih_bf, w_hh_bf, b_ih, b_hh, h, hbf, fc_w_bf, fc_b,
                logits, ids, err_flag, ws):
    """One streaming push for B <= 8 in one launch (nsd_stream_push): ``bins_in`` f32 [B,S,N] new bins -> front end of the
    bins that became computable, slide of the patch row in ``x0buf`` bf16 [2,B,N*K], every layer of the unidirectional stack
    (``h`` f32 / ``hbf`` bf16 [L,B,H] updated in place), ``logits`` f32 [B,C] and ``ids`` i32 [B].  ``rawring`` f32 [B,R,N],
    ``n_bins`` i32 [1] and ``extra`` describe the stream position (see include/nsd_b200.h)."""
    import ctypes as C
    L, B, H = h.shape
    N = bins_in.shape[2]
    for t in (bins_in, rawring, day_w, day_b, taps, x0buf, h, hbf, fc_w_bf, fc_b, logits, ids, ws):
        assert t.is_contiguous()
    assert bins_in.shape == (B, S, N) and rawring.shape[0] == B and rawring.shape[2] == N and x0buf.shape == (2, B, N * K)
    assert x0buf.dtype == torch.bfloat16 and hbf.dtype == torch.bfloat16 and h.dtype == torch.float32 and day.dtype == torch.int64
    tab = lambda ts: (C.c_void_p * L)(*[t.data_ptr() for t in ts])
    for l in range(L):
        assert w_ih_bf[l].is_contiguous() and w_hh_bf[l].is_contiguous() and b_ih[l].is_contiguous() and b_hh[l].is_contiguous()
    call("nsd_stream_push", ptr(bins_in), ptr(rawring), rawring.shape[1], ptr(day), ptr(day_w), ptr(day_b), day_w.shape[0], ptr(taps),
         taps.numel(), ptr(x0buf), ptr(n_bins), int(extra), B, N, int(K), int(S), H, L, fc_w_bf.shape[0], tab(w_ih_bf), tab(w_hh_bf),
         tab(b_ih), tab(b_hh), ptr(h), ptr(hbf), ptr(fc_w_bf), ptr(fc_b), ptr(logits), ptr(ids), ptr(err_flag), ptr(ws), ws.numel(), stream())


def stream_push_slots(bins_in, rawring, day, day_w, day_b, taps, x0buf, n_bins, active, last_frame, emitted, K, S, w_ih_bf, w_hh_bf, b_ih,
                      b_hh, h, hbf, fc_w_bf, fc_b, logits, ids, err_flag, ws):
    """``stream_push`` with an independent stream per batch row (nsd_stream_push_slots): ``n_bins``, ``active``,
    ``last_frame`` and ``emitted`` are i32 [B] on the device; inactive rows are left untouched, rows still warming up move
    only their ring and patch row, and only rows with ``emitted`` = 1 update ``h`` / ``hbf`` / ``logits`` (``ids`` = -1 for
    the others)."""
    import ctypes as C
    L, B, H = h.shape
    N = bins_in.shape[2]
    for t in (bins_in, rawring, day, day_w, day_b, taps, x0buf, n_bins, active, last_frame, emitted, h, hbf, fc_w_bf, fc_b, logits, ids, ws):
        assert t.is_contiguous()
    assert bins_in.shape == (B, S, N) and rawring.shape[0] == B and rawring.shape[2] == N and x0buf.shape == (2, B, N * K)
    assert x0buf.dtype == torch.bfloat16 and hbf.dtype == torch.bfloat16 and h.dtype == torch.float32 and day.dtype == torch.int64
    for t in (n_bins, active, last_frame, emitted, ids):
        assert t.dtype == torch.int32 and t.shape == (B,)
    tab = lambda ts: (C.c_void_p * L)(*[t.data_ptr() for t in ts])
    for l in range(L):
        assert w_ih_bf[l].is_contiguous() and w_hh_bf[l].is_contiguous() and b_ih[l].is_contiguous() and b_hh[l].is_contiguous()
    call("nsd_stream_push_slots", ptr(bins_in), ptr(rawring), rawring.shape[1], ptr(day), ptr(day_w), ptr(day_b), day_w.shape[0], ptr(taps),
         taps.numel(), ptr(x0buf), ptr(n_bins), ptr(active), ptr(last_frame), ptr(emitted), B, N, int(K), int(S), H, L, fc_w_bf.shape[0],
         tab(w_ih_bf), tab(w_hh_bf), tab(b_ih), tab(b_hh), ptr(h), ptr(hbf), ptr(fc_w_bf), ptr(fc_b), ptr(logits), ptr(ids), ptr(err_flag),
         ptr(ws), ws.numel(), stream())


def multi_copy(srcs, dsts):
    """Copy the f32 tensors ``srcs[i]`` into the equally sized contiguous views ``dsts[i]`` in one launch."""
    import ctypes as C
    n = len(srcs)
    if n == 0:
        return
    for s_, d_ in zip(srcs, dsts):
        assert s_.dtype == torch.float32 and d_.dtype == torch.float32 and s_.numel() == d_.numel() and s_.is_contiguous() and d_.is_contiguous()
    call("nsd_multi_copy_f32", n, (C.c_void_p * n)(*[t.data_ptr() for t in srcs]), (C.c_void_p * n)(*[t.data_ptr() for t in dsts]),
         (C.c_int64 * n)(*[t.numel() for t in srcs]), stream())


def greedy_decode_raw(act, st, sb, sc, lens, T, B, Cc, blank) -> Tuple[torch.Tensor, torch.Tensor]:
    out = torch.empty((B, T), device=act.device, dtype=torch.int64)
    out_len = torch.empty(B, device=act.device, dtype=torch.int32)
    call("nsd_greedy_decode", ptr(act), st, sb, sc, ptr(lens), T, B, Cc, blank, ptr(out), ptr(out_len), stream())
    return out, out_len


def edit_distance_raw(dec, dec_len, tgt, tgt_len) -> torch.Tensor:
    B = dec.shape[0]
    max_len = max(int(tgt.shape[1]), 1)
    nbytes = _lib.lib().nsd_edit_distance_workspace(B, max_len)
    ws = torch.empty(nbytes, device=dec.device, dtype=torch.uint8)
    dist = torch.empty(B, device=dec.device, dtype=torch.int32)
    call("nsd_edit_distance", ptr(dec), dec.stride(0), ptr(dec_len), ptr(tgt), tgt.stride(0), ptr(tgt_len), B,
         ptr(dist), ptr(ws), nbytes, stream())
    return dist
