"""B200-native drop-in for the reference's Conformer CTC model (BASELINE configs[2]).

``NeuralTransformerCTCModel`` keeps the constructor signature, sub-module / parameter / buffer names and shapes, RNG
consumption order of the initialisation (same seed => same initial weights, strict ``load_state_dict`` both ways) and the
call ``model(x, day_ids, input_lengths) -> (log_probs [T',B,C], out_lengths [B] int32, inter_log_probs | None)`` of
``src/neural_decoder/transformer_ctc.py:333-501``.  The torch.nn sub-modules are parameter containers only: every stage of
the forward AND the backward runs in ``libnsd_b200.so`` --
    day affine, attention products          nsd_bgemm (strided batched mma.sync GEMM, operands read in place)
    all nn.Linear layers                    nsd_gemm_bf16 (tcgen05 / TMA; the dense FLOPs) | nsd_gemm_f32 (parity mode)
    LayerNorm(+SiLU|GELU)(+dropout), SiLU/ReLU(+dropout), GLU, depthwise convs, residual+DropPath, SpecAugment+pos. enc.,
    masked softmax(+dropout), log-softmax   csrc/conformer_ew.cu, csrc/conformer_attn.cu
    CTC / InterCTC / label-smoothing KL     nsd_ctc_loss + nsd_sum_f32 + nsd_axpb (``conformer_loss``)
    AdamW + clip_grad_norm_                 nsd_sqnorm_multi + nsd_adamw_step (``FusedAdamW``)
-- through small ``torch.autograd.Function`` wrappers.  There is no PyTorch/CPU fallback: CPU tensors raise ``NsdError``.

Precision: ``"bf16"`` (default) = bf16 GEMM / attention operands, fp32 accumulation, fp32 residual stream, statistics,
softmax and parameters; ``"fp32"`` = CUDA-core fp32 everywhere (the parity mode).  Dropout / DropPath / SpecAugment are
counter-based (Philox) or host-drawn: distributional, not bit, parity with torch's generators.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch
from torch import nn

from . import _lib, ops
from ._lib import BF16, F32, NsdError, call, ptr, stream
from .model_tc import Bf16Shadows

ACT_NONE, ACT_SILU, ACT_GELU, ACT_RELU = 0, 1, 2, 3
_f32, _bf16 = torch.float32, torch.bfloat16


def _code(dt):
    return F32 if dt == _f32 else BF16


def _ws(nbytes: int, dev) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=dev)


# Weight-gradient GEMMs are off the critical path of the backward (nothing downstream reads dW before the optimizer): while
# ``wgrad_overlap()`` is active they are issued on a side stream and run beside the memory-bound element-wise chain of the main stream
# (a persistent tcgen05 GEMM leaves registers / threads for such kernels on every SM).  ``conformer_train_step`` turns it on around
# ``loss.backward()`` and joins the side stream before the optimizer reads the gradients.
class _Overlap:
    on = False
    side = {}
    pending = None

    @classmethod
    def stream(cls, dev):
        s = cls.side.get(dev)
        if s is None:
            s = cls.side[dev] = torch.cuda.Stream(dev)
        return s


class wgrad_overlap:
    def __init__(self, enabled: bool = True):
        self.enabled = enabled

    def __enter__(self):
        self.prev = _Overlap.on
        _Overlap.on = self.enabled
        _Overlap.pending = None
        return self

    def __exit__(self, *exc):
        _Overlap.on = self.prev
        if _Overlap.pending is not None:                  # join: the current stream waits for the last weight-gradient GEMM
            torch.cuda.current_stream(_Overlap.pending[0]).wait_event(_Overlap.pending[1])
            _Overlap.pending = None
        return False


# ----------------------------------------------------------------------------------------------------------------- autograd pieces
class _Linear(torch.autograd.Function):
    """y = x W^T + b (nn.Linear).  x bf16 [M,K] -> tcgen05 GEMM with the kept bf16 copy of W; x f32 -> CUDA-core fp32 GEMM."""

    @staticmethod
    def forward(ctx, x, w, b, wb, out_dtype):
        M, K = x.shape
        N = w.shape[0]
        y = torch.empty((M, N), device=x.device, dtype=out_dtype)
        ops.gemm(False, True, M, N, K, x, K, wb if x.dtype == _bf16 else w.detach(), K, y, N, bias=b.detach())
        ctx.save_for_backward(x, w)
        ctx.wb = wb
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        M, K = x.shape
        N = w.shape[0]
        dev = x.device
        dy = dy.contiguous()
        dx = None
        dw = torch.empty((N, K), device=dev, dtype=_f32)
        db = torch.empty((N,), device=dev, dtype=_f32)
        if x.dtype == _bf16:
            Np = (N + 7) // 8 * 8
            if dy.dtype == _bf16 and Np == N:
                dyb = dy
                ops.colsum(dy, M, N, N, db)
            elif dy.dtype == _f32 and N % 4 == 0:          # operand copy + bias gradient from one read of dy
                dyb = torch.empty((M, Np), device=dev, dtype=_bf16)
                ws = _ws(_lib.lib().nsd_cast_colsum_workspace(M, N), dev)
                call("nsd_cast_colsum", ptr(dy), M, N, ptr(dyb), Np, ptr(db), ptr(ws), ws.numel(), stream())
            else:
                dyb = torch.empty((M, Np), device=dev, dtype=_bf16)
                ops.cast_transpose_into(dy, dyb[:, :N], None)
                ops.colsum(dy, M, N, N, db)
            if _Overlap.on:
                main, side = torch.cuda.current_stream(dev), _Overlap.stream(dev)
                ready = torch.cuda.Event()
                ready.record(main)                         # dyb (and x) are complete on the main stream at this point
                side.wait_event(ready)
                with torch.cuda.stream(side):
                    ops.gemm(True, False, N, K, M, dyb, Np, x, K, dw, K)
                    done = torch.cuda.Event()
                    done.record(side)
                for t in (dyb, x, dw):                     # the caching allocator must not recycle them under the side stream's GEMM
                    t.record_stream(side)
                _Overlap.pending = (dev, done)
            else:
                ops.gemm(True, False, N, K, M, dyb, Np, x, K, dw, K)
            if ctx.needs_input_grad[0]:
                dx = torch.empty((M, K), device=dev, dtype=_bf16)
                ops.gemm(False, False, M, K, N, dyb, Np, ctx.wb, K, dx, K)
        else:
            dyf = dy if dy.dtype == _f32 else dy.float()
            ops.colsum(dyf, M, N, N, db)
            if ctx.needs_input_grad[0]:
                dx = torch.empty((M, K), device=dev, dtype=_f32)
                ops.gemm(False, False, M, K, N, dyf, N, w.detach(), K, dx, K)
            ops.gemm(True, False, N, K, M, dyf, N, x, K, dw, K)
        return dx, dw, db, None, None


class _LayerNorm(torch.autograd.Function):
    """dropout_p(act(LayerNorm(x))) -> (f32 and/or bf16 copies).  Returns the copy(ies) requested by ``want``.
    ``fork``: additionally returns x itself (an alias) as the LAST output -- the skip path of a pre-LN residual block.  Its gradient then
    arrives here together with the branch's and the backward kernel adds it to dx (no separate accumulation pass over [M, D])."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, act, p, seed, want32, want16, fork=False):
        M, D = x.shape
        dev = x.device
        y32 = torch.empty((M, D), device=dev, dtype=_f32) if want32 else None
        y16 = torch.empty((M, D), device=dev, dtype=_bf16) if want16 else None
        mean, rstd = torch.empty(M, device=dev), torch.empty(M, device=dev)
        call("nsd_layernorm_fwd", ptr(x), ptr(gamma), ptr(beta), float(eps), act, float(p), int(seed), ptr(y32), ptr(y16), ptr(mean), ptr(rstd), M, D, stream())
        ctx.save_for_backward(x, gamma, beta, mean, rstd)
        ctx.set_materialize_grads(False)
        ctx.cfg = (act, p, seed, want32, want16, fork)
        outs = tuple(t for t in (y32, y16) if t is not None)
        if fork:
            outs = outs + (x.view_as(x),)
        return outs if len(outs) > 1 else outs[0]

    @staticmethod
    def backward(ctx, *dys):
        x, gamma, beta, mean, rstd = ctx.saved_tensors
        act, p, seed, want32, want16, fork = ctx.cfg
        M, D = x.shape
        dev = x.device
        skip = None
        if fork:
            skip, dys = dys[-1], dys[:-1]
        dy = None
        for g in dys:                      # the two copies are the same value: their gradients add
            if g is not None:
                dy = g if dy is None else dy.float() + g.float()
        if dy is None:                     # only the skip path carries gradient
            return (skip,) + (None,) * 9
        dy = dy.contiguous()
        if skip is not None:
            skip = skip.contiguous()
        dx = torch.empty((M, D), device=dev, dtype=_f32)
        dg, db = torch.empty(D, device=dev), torch.empty(D, device=dev)
        nb = _lib.lib().nsd_layernorm_bwd_workspace(M, D)
        ws = _ws(nb, dev)
        call("nsd_layernorm_bwd", ptr(dy), _code(dy.dtype), ptr(x), ptr(gamma), ptr(beta), ptr(mean), ptr(rstd), act, float(p), int(seed), ptr(skip),
             ptr(dx), ptr(dg), ptr(db), M, D, ptr(ws), ws.numel(), stream())
        return dx, dg, db, None, None, None, None, None, None, None


class _Act(torch.autograd.Function):
    """dropout_p(act(x)) for f32 x -> out_dtype."""

    @staticmethod
    def forward(ctx, x, act, p, seed, out_dtype):
        y = torch.empty(x.shape, device=x.device, dtype=out_dtype)
        call("nsd_act_fwd", ptr(x), act, float(p), int(seed), ptr(y) if out_dtype == _f32 else None, ptr(y) if out_dtype == _bf16 else None, x.numel(), stream())
        ctx.save_for_backward(x)
        ctx.cfg = (act, p, seed)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        act, p, seed = ctx.cfg
        dy = dy.contiguous()
        dx = torch.empty(x.shape, device=x.device, dtype=_f32)
        call("nsd_act_bwd", ptr(dy), _code(dy.dtype), ptr(x), act, float(p), int(seed), ptr(dx), x.numel(), stream())
        return dx, None, None, None, None


class _GLU(torch.autograd.Function):
    @staticmethod
    def forward(ctx, u):
        M, D2 = u.shape
        g = torch.empty((M, D2 // 2), device=u.device, dtype=_f32)
        call("nsd_glu_fwd", ptr(u), ptr(g), M, D2 // 2, stream())
        ctx.save_for_backward(u)
        return g

    @staticmethod
    def backward(ctx, dg):
        (u,) = ctx.saved_tensors
        du = torch.empty_like(u)
        call("nsd_glu_bwd", ptr(dg.contiguous()), ptr(u), ptr(du), u.shape[0], u.shape[1] // 2, stream())
        return du


class _DwConv(torch.autograd.Function):
    """nn.Conv1d(D, D, k, padding=k//2, groups=D) over time, x [B*T, D] batch-major."""

    @staticmethod
    def forward(ctx, x, w, b, B, T):
        D, k = w.shape[0], w.shape[-1]
        y = torch.empty_like(x)
        call("nsd_dwconv_fwd", ptr(x), ptr(w), ptr(b), ptr(y), B, T, D, k, 0, 0, stream())
        ctx.save_for_backward(x, w)
        ctx.dims = (B, T, D, k)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        B, T, D, k = ctx.dims
        dy = dy.contiguous()
        dx = torch.empty_like(x)
        call("nsd_dwconv_fwd", ptr(dy), ptr(w), None, ptr(dx), B, T, D, k, 1, 0, stream())
        dw, db = torch.empty_like(w), torch.empty(D, device=x.device)
        ws = _ws(_lib.lib().nsd_dwconv_bwd_w_workspace(B, D, k), x.device)
        call("nsd_dwconv_bwd_w", ptr(dy), ptr(x), ptr(dw), ptr(db), B, T, D, k, ptr(ws), ws.numel(), stream())
        return dx, dw, db, None, None


class _Residual(torch.autograd.Function):
    """x + scale * DropPath(dropout(y))."""

    @staticmethod
    def forward(ctx, x, y, scale, p, seed, p_path, path_seed, per_sample):
        out = torch.empty_like(x)
        call("nsd_residual", ptr(x), ptr(y), float(scale), float(p), int(seed), float(p_path), int(path_seed), int(per_sample), ptr(out), x.numel(), stream())
        ctx.cfg = (scale, p, seed, p_path, path_seed, per_sample)
        return out

    @staticmethod
    def backward(ctx, dout):
        scale, p, seed, p_path, path_seed, per_sample = ctx.cfg
        dout = dout.contiguous()
        dy = torch.empty_like(dout)
        call("nsd_residual", None, ptr(dout), float(scale), float(p), int(seed), float(p_path), int(path_seed), int(per_sample), ptr(dy), dout.numel(), stream())
        return dout, dy, None, None, None, None, None, None


class _PosEncMask(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, pe, bands, bands_dev, B, T):
        import ctypes as C
        D = z.shape[1]
        out = torch.empty_like(z)
        arr = (C.c_int * 8)(*bands)
        call("nsd_posenc_mask", ptr(z), ptr(pe), arr, ptr(bands_dev), ptr(out), B, T, D, stream())
        ctx.cfg = (bands, bands_dev, B, T, D)
        return out

    @staticmethod
    def backward(ctx, dout):
        import ctypes as C
        bands, bands_dev, B, T, D = ctx.cfg
        dout = dout.contiguous()
        dz = torch.empty_like(dout)
        call("nsd_posenc_mask", ptr(dout), None, (C.c_int * 8)(*bands), ptr(bands_dev), ptr(dz), B, T, D, stream())
        return dz, None, None, None, None, None


def _bgemm(A, a_str, Bm, b_str, Cm, c_str, M, N, K, nb0, nb1, alpha=1.0, b_index=None, bias=None, bias_b0=0, a_off=0, b_off=0, c_off=0, tc=-1):
    """a_str = (rs, cs, b0, b1), b_str = (rs over k, cs over n, b0, b1), c_str = (rs, b0, b1); offsets in elements.
    tc: -1 = tensor cores iff an operand is bf16, 1 = tensor cores (f32 operands rounded to bf16 on load), 0 = fp32 FFMA."""
    call("nsd_bgemm", A.data_ptr() + a_off * A.element_size(), _code(A.dtype), *a_str, Bm.data_ptr() + b_off * Bm.element_size(), _code(Bm.dtype), *b_str,
         ptr(b_index), Cm.data_ptr() + c_off * Cm.element_size(), _code(Cm.dtype), *c_str, ptr(bias), int(bias_b0), M, N, K, nb0, nb1, float(alpha), int(tc),
         stream())


class _Attention(torch.autograd.Function):
    """softmax(Q K^T / sqrt(dh) + key padding mask) -> dropout -> V, per (utterance, head), on the packed projection qkv [B*T, 3D]
    (nn.MultiheadAttention, transformer_ctc.py:216, 250).  Q, K, V are read in place; the result lands in [B*T, D]."""

    @staticmethod
    def forward(ctx, qkv, lens, B, T, H, p, seed):
        D = qkv.shape[1] // 3
        dh = D // H
        dev = qkv.device
        Tp = (T + 7) // 8 * 8                      # row stride of the score matrices: rows stay 16-byte aligned for the batched GEMM's vector loads
        S = torch.empty((B * H * T, Tp), device=dev, dtype=_f32)
        sc = 1.0 / math.sqrt(dh)
        _bgemm(qkv, (3 * D, 1, T * 3 * D, dh), qkv, (1, 3 * D, T * 3 * D, dh), S, (Tp, H * T * Tp, T * Tp), T, T, dh, B, H, alpha=sc, b_off=D)
        lowp = qkv.dtype == _bf16
        Pd = torch.empty((B * H * T, Tp), device=dev, dtype=qkv.dtype) if (p > 0 or lowp) else None
        call("nsd_softmax_mask_fwd", ptr(S), ptr(Pd), _code(qkv.dtype), ptr(lens), B, H, T, Tp, float(p), int(seed), stream())
        o = torch.empty((B * T, D), device=dev, dtype=qkv.dtype)
        Pv = Pd if Pd is not None else S
        _bgemm(Pv, (Tp, 1, H * T * Tp, T * Tp), qkv, (3 * D, 1, T * 3 * D, dh), o, (D, T * D, dh), T, dh, T, B, H, b_off=2 * D)
        ctx.save_for_backward(qkv, S, Pv)
        ctx.cfg = (B, T, Tp, H, D, dh, p, seed, sc)
        return o

    @staticmethod
    def backward(ctx, do):
        qkv, P, Pv = ctx.saved_tensors
        B, T, Tp, H, D, dh, p, seed, sc = ctx.cfg
        dev = qkv.device
        do = do.contiguous()
        dqkv = torch.empty_like(qkv)
        # dV = Pd^T dO
        _bgemm(Pv, (1, Tp, H * T * Tp, T * Tp), do, (D, 1, T * D, dh), dqkv, (3 * D, T * 3 * D, dh), T, dh, T, B, H, c_off=2 * D)
        # dPd = dO V^T  -> dS (in place)
        dS = torch.empty((B * H * T, Tp), device=dev, dtype=_f32)
        _bgemm(do, (D, 1, T * D, dh), qkv, (1, 3 * D, T * 3 * D, dh), dS, (Tp, H * T * Tp, T * Tp), T, T, dh, B, H, b_off=2 * D)
        call("nsd_softmax_mask_bwd", ptr(P), ptr(dS), B, H, T, Tp, float(p), int(seed), stream())
        dSo = dS
        if qkv.dtype == _bf16:             # bf16 operand for the two products below (tensor-core path)
            dSo = torch.empty((B * H * T, Tp), device=dev, dtype=_bf16)
            call("nsd_cast", ptr(dS), F32, ptr(dSo), BF16, dS.numel(), stream())
        # dQ = sc * dS K ; dK = sc * dS^T Q
        _bgemm(dSo, (Tp, 1, H * T * Tp, T * Tp), qkv, (3 * D, 1, T * 3 * D, dh), dqkv, (3 * D, T * 3 * D, dh), T, dh, T, B, H, alpha=sc, b_off=D)
        _bgemm(dSo, (1, Tp, H * T * Tp, T * Tp), qkv, (3 * D, 1, T * 3 * D, dh), dqkv, (3 * D, T * 3 * D, dh), T, dh, T, B, H, alpha=sc, c_off=D)
        return dqkv, None, None, None, None, None, None


class _Frontend(torch.autograd.Function):
    """day affine -> Gaussian smoothing -> strided depthwise conv (transformer_ctc.py:41-49, 104-114).  X [B,T,N] f32; its gradient
    dxa W[day]^T is made when X requires grad, the day parameters' when they do."""

    @staticmethod
    def forward(ctx, X, day, day_w, day_b, day_w_op, gauss, tconv_w, S, want16):
        B, T, N = X.shape
        dev = X.device
        xa = torch.empty((B, T, N), device=dev, dtype=_f32)
        _bgemm(X, (N, 1, T * N, 0), day_w_op, (N, 1, N * N, 0), xa, (N, T * N, 0), T, N, N, B, 1, b_index=day, bias=day_b, bias_b0=N)
        xs = xa
        if gauss is not None:
            xs = torch.empty_like(xa)
            call("nsd_dwconv_fwd", ptr(xa), ptr(gauss), None, ptr(xs), B, T, N, gauss.numel(), 0, 1, stream())
        if tconv_w is not None:
            K = tconv_w.shape[-1]
            Tp = (T - K) // S + 1
            y32 = torch.empty((B * Tp, N), device=dev, dtype=_f32)
            y16 = torch.empty((B * Tp, N), device=dev, dtype=_bf16) if want16 else None
            call("nsd_strided_dwconv_fwd", ptr(xs), ptr(tconv_w), ptr(y32), ptr(y16), B, T, N, K, S, stream())
        else:
            y32 = xs.view(B * T, N)
            y16 = ops.cast(y32, _bf16) if want16 else None
        ctx.save_for_backward(X, day, day_w, day_w_op, gauss, tconv_w, xs)
        ctx.set_materialize_grads(False)
        ctx.cfg = (S, want16, day_b.shape[0], 1 if day_w_op.dtype == _bf16 else 0)
        return (y32, y16) if want16 else y32

    @staticmethod
    def backward(ctx, *dys):
        X, day, day_w, day_w_op, gauss, tconv_w, xs = ctx.saved_tensors
        S, want16, n_days, tc = ctx.cfg
        B, T, N = X.shape
        dev = X.device
        dy = None
        for g in dys:
            if g is not None:
                dy = g.float() if dy is None else dy + g.float()
        dy = dy.contiguous()
        dtw = None
        if tconv_w is not None:
            K = tconv_w.shape[-1]
            dxs = torch.empty((B, T, N), device=dev, dtype=_f32)
            dtw = torch.empty_like(tconv_w)
            ws = _ws(_lib.lib().nsd_strided_dwconv_bwd_workspace(B, N, K), dev)
            call("nsd_strided_dwconv_bwd", ptr(dy), ptr(xs), ptr(tconv_w), ptr(dxs), ptr(dtw), B, T, N, K, S, ptr(ws), ws.numel(), stream())
        else:
            dxs = dy.view(B, T, N)
        dxa = dxs
        if gauss is not None:
            dxa = torch.empty_like(dxs)
            call("nsd_dwconv_fwd", ptr(dxs), ptr(gauss), None, ptr(dxa), B, T, N, gauss.numel(), 1, 1, stream())
        dX = d_w = d_b = None
        if ctx.needs_input_grad[0]:
            # dX_b = dxa_b W[day_b]^T: the forward's operand (fp32 master or bf16 copy), read transposed
            dX = torch.empty((B, T, N), device=dev, dtype=_f32)
            _bgemm(dxa, (N, 1, T * N, 0), day_w_op, (1, N, N * N, 0), dX, (N, T * N, 0), T, N, N, B, 1, b_index=day)
        if ctx.needs_input_grad[2] or ctx.needs_input_grad[3]:
            # per-utterance X_b^T dxa_b and column sums, then the index_select backward over the day ids (fixed order)
            pw = torch.empty((B, N, N), device=dev, dtype=_f32)
            _bgemm(X, (1, N, T * N, 0), dxa, (N, 1, T * N, 0), pw, (N, N * N, 0), N, N, T, B, 1, tc=tc)
            ones = torch.ones((T,), device=dev, dtype=_f32)
            pb = torch.empty((B, N), device=dev, dtype=_f32)
            _bgemm(ones, (0, 1, 0, 0), dxa, (N, 1, T * N, 0), pb, (N, N, 0), 1, N, T, B, 1, tc=0)
            d_w = torch.empty((n_days, N, N), device=dev, dtype=_f32)
            d_b = torch.empty((n_days, 1, N), device=dev, dtype=_f32)
            call("nsd_index_reduce", ptr(pw), ptr(day), B, N * N, n_days, ptr(d_w), stream())
            call("nsd_index_reduce", ptr(pb), ptr(day), B, N, n_days, ptr(d_b), stream())
        return dX, None, d_w, d_b, None, None, dtw, None, None


class _LogSoftmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits):
        lp = torch.empty_like(logits)
        call("nsd_log_softmax_f32", ptr(logits), ptr(lp), logits.shape[0], logits.shape[1], stream())
        ctx.save_for_backward(lp)
        return lp

    @staticmethod
    def backward(ctx, dlp):
        (lp,) = ctx.saved_tensors
        dl = torch.empty_like(lp)
        call("nsd_log_softmax_bwd", ptr(lp), ptr(dlp.contiguous()), ptr(dl), lp.shape[0], lp.shape[1], stream())
        return dl


# ----------------------------------------------------------------------------------------------------------------- the module
class _DaySpecificLinear(nn.Module):                      # transformer_ctc.py:25-49 (parameter container)
    def __init__(self, n_days, dim):
        super().__init__()
        self.dim = dim
        self.day_weights = nn.Parameter(torch.randn(n_days, dim, dim))
        self.day_bias = nn.Parameter(torch.zeros(n_days, 1, dim))
        with torch.no_grad():
            for d in range(n_days):
                self.day_weights[d].copy_(torch.eye(dim))


class _NeuralFrontend(nn.Module):                         # transformer_ctc.py:52-128 (parameter container)
    def __init__(self, n_channels, frontend_dim, dropout, temporal_kernel, temporal_stride, gaussian_smooth_width):
        super().__init__()
        self.n_channels, self.temporal_kernel, self.temporal_stride = n_channels, temporal_kernel, temporal_stride
        if gaussian_smooth_width > 0:
            ks = int(gaussian_smooth_width * 4) + 1
            x = torch.arange(ks, dtype=torch.float32) - (ks - 1) / 2
            g = torch.exp(-x.pow(2) / (2 * gaussian_smooth_width ** 2))
            self.register_buffer("gaussian_kernel", (g / g.sum()).view(1, 1, -1))
            self.gaussian_padding = ks // 2
        else:
            self.gaussian_kernel = None
        if temporal_kernel > 0:
            self.temporal_conv = nn.Conv1d(n_channels, n_channels, kernel_size=temporal_kernel, stride=temporal_stride, padding=0, groups=n_channels, bias=False)
            nn.init.constant_(self.temporal_conv.weight, 1.0 / temporal_kernel)
        else:
            self.temporal_conv = None
        self.proj = nn.Linear(n_channels, frontend_dim)
        self.ln = nn.LayerNorm(frontend_dim)
        self.dropout = nn.Dropout(dropout)


class _AutoEncoderEncoder(nn.Module):                     # transformer_ctc.py:131-146
    def __init__(self, input_dim, latent_dim, hidden_dim):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.ReLU(inplace=True), nn.Linear(hidden_dim, latent_dim))


class _ConvModule(nn.Module):                             # transformer_ctc.py:148-191
    def __init__(self, d_model, kernel_size, dropout):
        super().__init__()
        self.ln = nn.LayerNorm(d_model)
        self.pw_conv1 = nn.Linear(d_model, d_model * 2)
        self.glu = nn.GLU(dim=-1)
        self.dw_conv = nn.Conv1d(d_model, d_model, kernel_size=kernel_size, padding=kernel_size // 2, groups=d_model)
        self.ln_conv = nn.LayerNorm(d_model)
        self.activation = nn.SiLU()
        self.pw_conv2 = nn.Linear(d_model, d_model)
        self.dropout = nn.Dropout(dropout)


class _DropPath(nn.Module):                               # transformer_ctc.py:9-23
    def __init__(self, drop_prob=0.0):
        super().__init__()
        self.drop_prob = drop_prob


class _ConformerBlock(nn.Module):                         # transformer_ctc.py:194-263
    def __init__(self, d_model, nhead, dim_feedforward, dropout, conv_kernel_size, drop_path_prob):
        super().__init__()
        mk_ff = lambda: nn.Sequential(nn.LayerNorm(d_model), nn.Linear(d_model, dim_feedforward), nn.SiLU(), nn.Dropout(dropout),
                                      nn.Linear(dim_feedforward, d_model), nn.Dropout(dropout))
        self.ff1 = mk_ff()
        self.ln_attn = nn.LayerNorm(d_model)
        self.attn = nn.MultiheadAttention(d_model, nhead, dropout=dropout, batch_first=True)
        self.dropout_attn = nn.Dropout(dropout)
        self.conv_module = _ConvModule(d_model, conv_kernel_size, dropout)
        self.ff2 = mk_ff()
        self.ln_final = nn.LayerNorm(d_model)
        self.drop_path = _DropPath(drop_path_prob)


class _SpecAugment(nn.Module):                            # transformer_ctc.py:266-308
    def __init__(self, freq_mask_param, time_mask_param, num_freq_masks, num_time_masks):
        super().__init__()
        self.freq_mask_param, self.time_mask_param = freq_mask_param, time_mask_param
        self.num_freq_masks, self.num_time_masks = num_freq_masks, num_time_masks

    def draw(self, T: int, F: int):
        """The reference's draws from torch's host generator, in its order (a second draw only when the width is > 0)."""
        bands = []
        for n, limit, size in ((self.num_freq_masks, self.freq_mask_param, F), (self.num_time_masks, self.time_mask_param, T)):
            for _ in range(n):
                w = min(int(torch.rand(1).item() * limit), size)
                lo = int(torch.rand(1).item() * (size - w)) if w > 0 else 0
                bands += [lo, lo + w]
        return bands


class _PositionalEncoding(nn.Module):                     # transformer_ctc.py:311-330
    def __init__(self, d_model, max_len=5000):
        super().__init__()
        pe = torch.zeros(max_len, d_model)
        position = torch.arange(0, max_len, dtype=torch.float).unsqueeze(1)
        div_term = torch.exp(torch.arange(0, d_model, 2).float() * (-math.log(10000.0) / d_model))
        pe[:, 0::2] = torch.sin(position * div_term)
        pe[:, 1::2] = torch.cos(position * div_term)
        self.register_buffer("pe", pe.unsqueeze(0))


class NeuralTransformerCTCModel(nn.Module):
    def __init__(self, n_channels: int, n_classes: int, n_days: int, frontend_dim: int = 1024, latent_dim: int = 1024,
                 autoencoder_hidden_dim: int = 512, transformer_layers: int = 8, transformer_heads: int = 8, transformer_ff_dim: int = 2048,
                 transformer_dropout: float = 0.3, temporal_kernel: int = 32, temporal_stride: int = 4, gaussian_smooth_width: float = 2.0,
                 conformer_conv_kernel: int = 31, use_spec_augment: bool = True, spec_augment_freq_mask: int = 100, spec_augment_time_mask: int = 40,
                 drop_path_prob: float = 0.1, device: str = "cuda", precision: Optional[str] = None):
        super().__init__()
        from .model import default_precision
        self.device_name = device
        self.precision = precision or default_precision()
        self.day_linear = _DaySpecificLinear(n_days, n_channels)
        self.frontend = _NeuralFrontend(n_channels, frontend_dim, transformer_dropout, temporal_kernel, temporal_stride, gaussian_smooth_width)
        self.encoder = _AutoEncoderEncoder(frontend_dim, latent_dim, autoencoder_hidden_dim)
        self.use_spec_augment = use_spec_augment
        if use_spec_augment:
            self.spec_augment = _SpecAugment(spec_augment_freq_mask, spec_augment_time_mask, 2, 2)
        self.pos_enc = _PositionalEncoding(latent_dim)
        self.conformer_layers = nn.ModuleList([_ConformerBlock(latent_dim, transformer_heads, transformer_ff_dim, transformer_dropout,
                                                               conformer_conv_kernel, drop_path_prob) for _ in range(transformer_layers)])
        self.use_interctc = transformer_layers >= 6
        if self.use_interctc:
            self.interctc_layer = transformer_layers // 2
            self.inter_output = nn.Linear(latent_dim, n_classes)
        self.output = nn.Sequential(nn.Linear(latent_dim, latent_dim), nn.LayerNorm(latent_dim), nn.GELU(), nn.Dropout(0.3), nn.Linear(latent_dim, n_classes))
        self.temporal_kernel, self.temporal_stride = temporal_kernel, temporal_stride
        self.n_heads, self.dropout_p, self.conv_kernel = transformer_heads, transformer_dropout, conformer_conv_kernel
        if latent_dim % transformer_heads or latent_dim % 4 or frontend_dim % 8 or n_channels % 8 or autoencoder_hidden_dim % 8 or transformer_ff_dim % 8:
            raise NsdError("NeuralTransformerCTCModel (B200): widths must be multiples of 8 and latent_dim divisible by the head count")
        if conformer_conv_kernel % 2 == 0 or conformer_conv_kernel > 32:
            raise NsdError("NeuralTransformerCTCModel (B200): the depthwise kernel must be odd and <= 32 (reference: 31)")
        self._shadows = Bf16Shadows()
        self._calls = 0
        self._bands_dev = None             # int32[8] device array of SpecAugment bounds (set by GraphedConformerStep)
        self.check_day_ids = True          # validate day_ids like index_select does (costs a device->host sync per call; a trainer that owns its ids can switch it off)

    # ---------------------------------------------------------------------------------------------------------------
    def compute_output_lengths(self, input_lengths: torch.Tensor, actual_seq_len: int) -> torch.Tensor:
        """transformer_ctc.py:422-431."""
        if self.temporal_kernel > 0 and self.temporal_stride > 1:
            output_lengths = ((input_lengths - self.temporal_kernel) / self.temporal_stride).to(torch.int32)
        else:
            output_lengths = input_lengths
        return torch.clamp(output_lengths, max=actual_seq_len)

    def invalidate_weight_copies(self) -> None:
        self._shadows.invalidate()

    def _lin(self, x, mod: nn.Linear, key, out_dtype=_f32):
        wb = self._shadows.stacked(key, [mod.weight]) if x.dtype == _bf16 else None
        return _Linear.apply(x, mod.weight, mod.bias, wb, out_dtype)

    def forward(self, x: torch.Tensor, day_ids: torch.Tensor, input_lengths: Optional[torch.Tensor] = None
                ) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
        if not x.is_cuda:
            raise NsdError("NeuralTransformerCTCModel (B200) runs on CUDA tensors only; there is no CPU fallback")
        if x.dim() != 3 or x.shape[2] != self.day_linear.dim:
            raise RuntimeError(f"x must be [B, T, {self.day_linear.dim}], got {tuple(x.shape)}")
        with torch.cuda.device(x.device):
            return self._forward(x, day_ids, input_lengths)

    def _forward(self, x, day_ids, input_lengths):
        dev = x.device
        B, T, N = x.shape
        lowp = self.precision == "bf16"
        adt = _bf16 if lowp else _f32                     # dtype of GEMM operands
        train = self.training
        pd = self.dropout_p if train else 0.0
        self._calls += 1
        base = (int(torch.initial_seed()) * 0x9E3779B97F4A7C15 + self._calls * 0xD1B54A32D192ED03) & 0x7FFFFFFFFFFFFFFF
        site = [0]

        def seed():
            site[0] += 1
            return (base + site[0] * 0x2545F4914F6CDD1D) & 0x7FFFFFFFFFFFFFFF

        def ln(xx, mod: nn.LayerNorm, act=ACT_NONE, p=0.0, want32=False, want16=None, fork=False):
            want16 = lowp if want16 is None else want16
            if not want32 and not want16:
                want32 = True
            return _LayerNorm.apply(xx, mod.weight, mod.bias, mod.eps, act, p, seed() if p > 0 else 0, want32, want16, fork)

        day = day_ids.to(device=dev, dtype=torch.int64).contiguous()
        if self.check_day_ids and day.numel() and (int(day.min()) < 0 or int(day.max()) >= self.day_linear.day_weights.shape[0]):
            raise IndexError("index out of range in self")                      # index_select (transformer_ctc.py:47); a host synchronisation
        fe = self.frontend
        if fe.temporal_conv is not None and T < fe.temporal_kernel:
            raise RuntimeError(f"Calculated padded input size per channel: ({T}). Kernel size: ({fe.temporal_kernel}). Kernel size can't be greater than actual input size")
        dw = self.day_linear.day_weights
        dw_op = self._shadows.stacked(("day", 0), [dw.view(-1, N)]) if lowp else dw.detach()
        gauss = fe.gaussian_kernel.reshape(-1).contiguous() if fe.gaussian_kernel is not None else None
        tw = fe.temporal_conv.weight if fe.temporal_conv is not None else None
        feats = _Frontend.apply(x.contiguous().float(), day, dw, self.day_linear.day_bias, dw_op, gauss, tw, fe.temporal_stride, lowp)
        f32_feats, op_feats = (feats if lowp else (feats, feats))
        Tn = f32_feats.shape[0] // B
        # proj -> LN -> dropout (transformer_ctc.py:124-127)
        z = self._lin(op_feats, fe.proj, ("fe.proj", 0))
        z = ln(z, fe.ln, p=pd)
        # bottleneck MLP (transformer_ctc.py:131-146)
        z = self._lin(z, self.encoder.net[0], ("enc", 0))
        z = _Act.apply(z, ACT_RELU, 0.0, 0, adt)
        z = self._lin(z, self.encoder.net[2], ("enc", 2))
        # SpecAugment (training) + positional encoding (transformer_ctc.py:466-471)
        D = z.shape[1]
        bands, bands_dev = [0] * 8, None
        if self.use_spec_augment and train:
            if self._bands_dev is not None:
                bands_dev = self._bands_dev                    # graph replay: the host writes this step's draw into the device array
            else:
                bands = self.spec_augment.draw(Tn, D)
        pe = self.pos_enc.pe[0, :Tn].contiguous()
        z = _PosEncMask.apply(z, pe, tuple(bands), bands_dev, B, Tn)
        lens = None
        if input_lengths is not None:
            out_lengths = self.compute_output_lengths(input_lengths.to(dev), Tn)
            lens = out_lengths.to(torch.int32).contiguous()
        else:
            out_lengths = torch.full((B,), Tn, dtype=torch.int32, device=dev)
        per_sample = Tn * D
        inter_log_probs = None
        nl = len(self.conformer_layers)
        for i, blk in enumerate(self.conformer_layers):
            pp = blk.drop_path.drop_prob if train else 0.0
            # half-step feed-forward (transformer_ctc.py:245)
            z = self._ff(z, blk.ff1, (i, "ff1"), ln, seed, pd, pp, per_sample, adt)
            # self-attention (transformer_ctc.py:248-251)
            h, z = ln(z, blk.ln_attn, fork=True)
            wb = self._shadows.stacked((i, "attn.in"), [blk.attn.in_proj_weight]) if lowp else None
            qkv = _Linear.apply(h, blk.attn.in_proj_weight, blk.attn.in_proj_bias, wb, adt)
            o = _Attention.apply(qkv, lens, B, Tn, self.n_heads, pd, seed() if pd > 0 else 0)
            y = self._lin(o, blk.attn.out_proj, (i, "attn.out"))
            z = _Residual.apply(z, y, 1.0, pd, seed(), pp, seed(), per_sample)
            # convolution module (transformer_ctc.py:170-191)
            cm = blk.conv_module
            h, z = ln(z, cm.ln, fork=True)
            u = self._lin(h, cm.pw_conv1, (i, "pw1"))
            g = _GLU.apply(u)
            c = _DwConv.apply(g, cm.dw_conv.weight, cm.dw_conv.bias, B, Tn)
            h = ln(c, cm.ln_conv, act=ACT_SILU)
            y = self._lin(h, cm.pw_conv2, (i, "pw2"))
            z = _Residual.apply(z, y, 1.0, pd, seed(), 0.0, 0, per_sample)
            z = self._ff(z, blk.ff2, (i, "ff2"), ln, seed, pd, pp, per_sample, adt)
            want_op = (self.use_interctc and i == self.interctc_layer - 1 and train) or i == nl - 1
            if want_op and lowp:
                z, z_op = ln(z, blk.ln_final, want32=True, want16=True)
            else:
                z = ln(z, blk.ln_final, want32=True, want16=False)
                z_op = z
            if self.use_interctc and i == self.interctc_layer - 1 and train:
                il = self._lin(z_op, self.inter_output, ("inter", 0))
                inter_log_probs = _LogSoftmax.apply(il).view(B, Tn, -1).transpose(0, 1)
        # deep classification head (transformer_ctc.py:408-415)
        h = self._lin(z_op, self.output[0], ("out", 0))
        h = ln(h, self.output[1], act=ACT_GELU, p=(self.output[3].p if train else 0.0))
        logits = self._lin(h, self.output[4], ("out", 4))
        log_probs = _LogSoftmax.apply(logits).view(B, Tn, -1).transpose(0, 1)
        return log_probs, out_lengths, inter_log_probs

    def _ff(self, z, ff: nn.Sequential, key, ln, seed, pd, pp, per_sample, adt):
        h, z = ln(z, ff[0], fork=True)
        u = self._lin(h, ff[1], (key, 1))
        s = _Act.apply(u, ACT_SILU, pd, seed() if pd > 0 else 0, adt)
        y = self._lin(s, ff[4], (key, 4))
        return _Residual.apply(z, y, 0.5, pd, seed(), pp, seed(), per_sample)


# ----------------------------------------------------------------------------------------------------------------- loss / optimiser
class _ConformerLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lp, inter, y, out_lens, y_len, ls, iw):
        dev = lp.device
        Tn, B, C = lp.shape
        total = torch.zeros(1, device=dev, dtype=_f32)
        w_main = (1.0 - iw) if inter is not None else 1.0
        grads = []
        for t, w in ((lp, w_main), (inter, iw)):
            if t is None:
                grads.append(None)
                continue
            if torch.empty_like(t).stride() != t.stride():     # the kernels address the dense storage with t's own strides
                t = t.contiguous()
            st, sb, sc = t.stride()
            mean = ls <= 0
            loss, nll, grad = ops.ctc_loss_raw(t, st, sb, sc, False, y, out_lens, y_len, Tn, B, C, 0, mean, True)
            if mean:                       # trainer:137-141 reduction="mean", :243/:230 torch.sum of the scalar
                call("nsd_sum_f32", ptr(loss), 1, float(w), 0.0, 1, ptr(total), stream())
                a, b = w, 0.0
            else:                          # reduction="none" + torch.mean (trainer:228, 236)
                is_main = len(grads) == 0
                a = w * ((1.0 - ls) if is_main else 1.0) / B
                call("nsd_sum_f32", ptr(nll), B, float(a), 0.0, 1, ptr(total), stream())
                b = 0.0
                if is_main:                # label smoothing: KL(uniform || p), reduction "batchmean" over dim 0 = T' (trainer:238-240)
                    b = -w * ls / (C * Tn)
                    call("nsd_sum_f32", ptr(t), t.numel(), float(b), float(-w * ls * math.log(C) * B), 1, ptr(total), stream())   # dense view: storage order
            g = torch.empty_like(grad)
            call("nsd_axpb", ptr(grad), float(a), float(b), ptr(g), grad.numel(), stream())
            grads.append(g)
        ctx.save_for_backward(*[g for g in grads if g is not None])
        ctx.has_inter = inter is not None
        return total[0]

    @staticmethod
    def backward(ctx, dloss):
        gs = list(ctx.saved_tensors)
        g_main = gs[0] * dloss
        g_inter = gs[1] * dloss if ctx.has_inter else None
        return g_main, g_inter, None, None, None, None, None


def conformer_loss(log_probs, inter_log_probs, y, out_lens, y_len, label_smoothing: float = 0.1, interctc_weight: float = 0.3):
    """The transformer branch of the trainer's loss (neural_decoder_trainer.py:137-141, 212-249) on the CUDA kernels: CTC on the main
    and the InterCTC log-probs (``reduction="none"`` + mean when label smoothing is on, ``"mean"`` otherwise), the label-smoothing
    KL term, and their weighted sum; the gradient w.r.t. both log-prob tensors comes out of the same launches."""
    dev = log_probs.device
    y = y.to(device=dev, dtype=torch.int32).contiguous()
    if y.shape[1] == 0:
        y = torch.zeros((y.shape[0], 1), device=dev, dtype=torch.int32)
    i32 = lambda t: t.to(device=dev, dtype=torch.int32).contiguous()
    return _ConformerLoss.apply(log_probs, inter_log_probs, y, i32(out_lens), i32(y_len), float(label_smoothing), float(interctc_weight))


def lr_lambda(step: int, warmup_steps: int, total_steps: int) -> float:
    """neural_decoder_trainer.py:154-158."""
    if warmup_steps > 0 and step < warmup_steps:
        return float(step + 1) / float(max(1, warmup_steps))
    progress = (step - warmup_steps) / float(max(1, total_steps - warmup_steps))
    return 0.5 * (1.0 + math.cos(math.pi * progress))


class FusedAdamW(torch.optim.Optimizer):
    """torch.optim.AdamW(betas, eps, weight_decay) + clip_grad_norm_(max_norm) (neural_decoder_trainer.py:144-151, 255-259) as two
    multi-tensor launches: the squared gradient norm stays on the device and the update kernel derives the clip coefficient from it."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0, max_grad_norm: Optional[float] = None, grad_scale=1.0):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self.max_grad_norm, self.grad_scale, self.shadows = max_grad_norm, grad_scale, None
        self.grad_sqnorm: Optional[torch.Tensor] = None        # device scalar of the last step (unscaled gradients)
        self.hyper_dev: Optional[torch.Tensor] = None          # device float[3] schedule (GraphedConformerStep); None = host values

    def attach_shadows(self, shadows) -> None:
        self.shadows = shadows

    @torch.no_grad()
    def step(self, closure=None):
        import ctypes as C
        for group in self.param_groups:
            ps = [p for p in group["params"] if p.grad is not None]
            if not ps:
                continue
            dev = ps[0].device
            gs, ms, vs = [], [], []
            for p in ps:
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                st["step"] += 1
                gs.append(p.grad if p.grad.is_contiguous() else p.grad.contiguous())
                ms.append(st["exp_avg"]); vs.append(st["exp_avg_sq"])
            step = self.state[ps[0]]["step"]
            n = len(ps)
            arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
            numel = (C.c_int64 * n)(*[t.numel() for t in ps])
            with torch.cuda.device(dev):
                sq = None
                if self.max_grad_norm is not None:
                    sq = self.grad_sqnorm if (self.hyper_dev is not None and self.grad_sqnorm is not None) else torch.empty(1, device=dev, dtype=_f32)
                    ws = _ws(_lib.lib().nsd_sqnorm_workspace(n, numel), dev)
                    call("nsd_sqnorm_multi", n, arr(gs), numel, ptr(sq), ptr(ws), ws.numel(), stream())
                    self.grad_sqnorm = sq
                sh_list = [self.shadows.slice_for(p) for p in ps] if self.shadows is not None else None
                sh = None
                if sh_list is not None and any(s is not None for s in sh_list):
                    sh = (C.c_void_p * n)(*[None if s is None else s.data_ptr() for s in sh_list])
                call("nsd_adamw_step", n, arr(ps), arr(gs), arr(ms), arr(vs), numel, sh, float(group["lr"]), float(group["betas"][0]),
                     float(group["betas"][1]), float(group["eps"]), float(group["weight_decay"]), int(step), float(self.grad_scale), ptr(sq),
                     float(self.max_grad_norm or 0.0), ptr(self.hyper_dev), stream())
            torch.autograd.graph.increment_version(ps)
            if sh_list is not None:
                for p, s in zip(ps, sh_list):
                    if s is not None:
                        self.shadows.mark_fresh(p)
        return None


def conformer_train_step(model, optimizer, X, y, X_len, y_len, day_idx, label_smoothing=0.1, interctc_weight=0.3, white_noise_sd=0.0,
                         constant_offset_sd=0.0, noise_seed=0, overlap_wgrad=False):
    """One training step of the transformer branch of the trainer (neural_decoder_trainer.py:181-260): noise augmentation, forward,
    CTC + InterCTC + label smoothing, backward, gradient clipping and AdamW, all on the CUDA kernels.  Returns the loss tensor.
    ``overlap_wgrad``: issue the weight-gradient GEMMs on a side stream beside the element-wise chain (pays off when the step is replayed as a
    graph -- GraphedConformerStep switches it on; issued eagerly from Python the extra events cost more host time than the overlap gains)."""
    model.train()
    if white_noise_sd > 0 or constant_offset_sd > 0:
        X = ops.input_noise(X, white_noise_sd, constant_offset_sd, noise_seed)
    log_probs, out_lens, inter = model(X, day_idx, X_len)
    loss = conformer_loss(log_probs, inter, y, out_lens, y_len, label_smoothing, interctc_weight)
    optimizer.zero_grad(set_to_none=True)
    with wgrad_overlap(overlap_wgrad):
        loss.backward()
    optimizer.step()
    return loss


class GraphedConformerStep:
    """The whole training step of the transformer branch (neural_decoder_trainer.py:181-260: noise, forward, CTC + InterCTC + label
    smoothing, backward, gradient clipping, AdamW with the warm-up / cosine schedule) captured ONCE as a CUDA graph and replayed: one
    launch from the host instead of ~800.  Everything that changes from step to step lives in device memory that the host refreshes
    with one small copy before the replay: the Philox seed offset (fresh dropout / DropPath / noise masks), the SpecAugment bounds
    (drawn on the host in the reference's order), and AdamW's step size / bias corrections / decay for the step's learning rate.
    Shapes are static: batches must be [B, T, N] with targets padded to ``max_tgt``."""

    def __init__(self, model: NeuralTransformerCTCModel, optimizer: FusedAdamW, B: int, T: int, max_tgt: int, *, label_smoothing=0.1,
                 interctc_weight=0.3, white_noise_sd=0.0, constant_offset_sd=0.0, base_lr: Optional[float] = None, warmup_steps: int = 0,
                 total_steps: int = 1 << 30, eager_warmup: int = 2):
        p0 = next(model.parameters())
        dev = p0.device
        if not isinstance(optimizer, FusedAdamW) or len(optimizer.param_groups) != 1:
            raise NsdError("GraphedConformerStep needs a FusedAdamW with a single parameter group (one device-resident schedule)")
        self.model, self.opt, self.dev = model, optimizer, dev
        N = model.day_linear.dim
        self.X = torch.zeros(B, T, N, device=dev)
        self.y = torch.zeros(B, max_tgt, device=dev, dtype=torch.int32)
        self.X_len = torch.full((B,), T, device=dev, dtype=torch.int32)
        self.y_len = torch.ones(B, device=dev, dtype=torch.int32)
        self.day = torch.zeros(B, device=dev, dtype=torch.int64)
        self.cfg = (label_smoothing, interctc_weight, white_noise_sd, constant_offset_sd)
        self.base_lr = optimizer.param_groups[0]["lr"] if base_lr is None else base_lr
        self.warmup_steps, self.total_steps = warmup_steps, total_steps
        # per-step device state: [seed offset u64 | hyper f32 x3 + pad | bands i32 x8] in one 64-byte block, staged through pinned memory
        self._state = torch.zeros(64, device=dev, dtype=torch.uint8)
        self._stages = [torch.zeros(64, dtype=torch.uint8).pin_memory() for _ in range(4)]      # ring: the host may run a few steps ahead
        self._stage_events = [None] * 4
        self._seed = self._state[0:8].view(torch.int64)
        self._hyper = self._state[8:24].view(torch.float32)
        self._bands = self._state[24:56].view(torch.int32)
        self.steps_done = 0
        self.graph = None
        self.loss = None
        self.kernels_per_replay = 0
        self._eager_warmup = eager_warmup
        model.check_day_ids = False
        model.train()

    def _host_state(self):
        import struct
        m, g = self.model, self.opt.param_groups[0]
        t = self.steps_done + 1
        lr = self.base_lr * lr_lambda(self.steps_done, self.warmup_steps, self.total_steps)
        # the same float32 / float64 arithmetic nsd_adamw_step does on the host when it gets lr, betas and step by value
        import numpy as np
        lr32, b1, b2 = np.float32(lr), float(np.float32(g["betas"][0])), float(np.float32(g["betas"][1]))
        hyper = (float(np.float32(float(lr32) / (1.0 - b1 ** t))), float(np.float32(1.0 / math.sqrt(1.0 - b2 ** t))),
                 float(np.float32(1.0) - lr32 * np.float32(g["weight_decay"])))
        Tn = (self.X.shape[1] - m.temporal_kernel) // m.temporal_stride + 1 if m.temporal_kernel > 0 else self.X.shape[1]
        bands = m.spec_augment.draw(Tn, m.pos_enc.pe.shape[-1]) if m.use_spec_augment else [0] * 8
        seed = (self.steps_done * 0x9E3779B97F4A7C15 + 0x632BE59BD9B4E019) & 0x7FFFFFFFFFFFFFFF
        raw = struct.pack("<q3f4x8i8x", seed, *hyper, *bands)
        i = self.steps_done % len(self._stages)
        if self._stage_events[i] is not None:
            self._stage_events[i].synchronize()             # the copy that last read this staging buffer has run
        self._stages[i].copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8))
        self._state.copy_(self._stages[i], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._stage_events[i] = ev
        for grp in self.opt.param_groups:
            grp["lr"] = lr

    def _body(self):
        ls, iw, wsd, csd = self.cfg
        self.loss = conformer_train_step(self.model, self.opt, self.X, self.y, self.X_len, self.y_len, self.day, ls, iw, wsd, csd, noise_seed=12345,
                                         overlap_wgrad=True)

    def _capture(self):
        m, opt = self.model, self.opt
        call("nsd_set_seed_offset_ptr", ptr(self._seed))
        m._bands_dev = self._bands if m.use_spec_augment else None
        opt.hyper_dev = self._hyper
        if opt.max_grad_norm is not None and opt.grad_sqnorm is None:
            opt.grad_sqnorm = torch.zeros(1, device=self.dev, dtype=_f32)
        # torch's capture protocol wants a few eager runs on a side stream first.  They must not count as training steps: parameters
        # and optimizer state are snapshotted before and put back after (the bf16 operand copies are re-made from the restored weights).
        ps = [p for grp in opt.param_groups for p in grp["params"]]
        for p in ps:
            st = opt.state[p]
            if not st:
                st["step"] = 0
                st["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
        snap = [(p.detach().clone(), opt.state[p]["exp_avg"].clone(), opt.state[p]["exp_avg_sq"].clone(), opt.state[p]["step"]) for p in ps]
        done0 = self.steps_done
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            for _ in range(self._eager_warmup):
                self._host_state()
                self._body()
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        n0 = _lib.lib().nsd_launch_count()
        with torch.cuda.graph(g):
            self._body()
        self.kernels_per_replay = int(_lib.lib().nsd_launch_count() - n0)     # this library's kernels inside one replay
        self.graph = g
        with torch.no_grad():
            for p, (w, m1, m2, st) in zip(ps, snap):
                p.copy_(w)
                opt.state[p]["exp_avg"].copy_(m1); opt.state[p]["exp_avg_sq"].copy_(m2); opt.state[p]["step"] = st
                sl = opt.shadows.slice_for(p) if opt.shadows is not None else None
                if sl is not None:
                    ops.cast_transpose_into(p.detach(), sl, None)
                    opt.shadows.mark_fresh(p)
        self.steps_done = done0
        self._host_state()
        g.replay()                                          # the first real step
        self.steps_done += 1

    @torch.no_grad()
    def _load(self, X, y, X_len, y_len, day):
        if y.shape[1] > self.y.shape[1]:
            raise RuntimeError(f"targets are padded to {y.shape[1]} > max_tgt={self.y.shape[1]} of the captured step")
        self.X.copy_(X, non_blocking=True)
        self.y.zero_()
        self.y[:, :y.shape[1]].copy_(y, non_blocking=True)
        self.X_len.copy_(X_len, non_blocking=True)
        self.y_len.copy_(y_len, non_blocking=True)
        self.day.copy_(day, non_blocking=True)

    def step(self, X, y, X_len, y_len, day) -> torch.Tensor:
        """One training step on the given batch (host or device tensors of the captured shapes).  Returns the loss tensor of the captured
        graph (overwritten by the next step)."""
        with torch.cuda.device(self.dev):
            self._load(X, y, X_len, y_len, day)
            if self.graph is None:
                self._capture()
            else:
                self._host_state()
                self.graph.replay()
                self.steps_done += 1
        return self.loss

    def close(self) -> None:
        call("nsd_set_seed_offset_ptr", None)
        self.model._bands_dev = None
        self.opt.hyper_dev = None
