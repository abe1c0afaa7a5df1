"""Drop-in ``GRUDecoder`` backed by the sm_100a kernels in ``libnsd_b200.so``.

Mirrors the reference module (src/neural_decoder/model.py:7-123): same
constructor signature, same parameter / buffer names, shapes and initialisation
(so a reference ``state_dict`` loads with ``strict=True`` and the same torch seed
gives the same weights), same ``forward(neuralInput[B,T,N], dayIdx[B]) ->
logits[B,T',n_classes+1]``.  Everything under ``forward`` runs in the CUDA
library: K1 front end, K2 GEMMs, K3 recurrence; the backward is hand-written
too (``_DecoderFunction.backward``), autograd only sees one node.
"""
from __future__ import annotations

import math
from typing import List, Optional

import torch
from torch import nn
from torch.autograd.function import once_differentiable

from . import ops
from ._lib import NsdError, call
from .model_tc import Bf16Shadows, check_architecture

_DEFAULT_PRECISION = "fp32"


def set_default_precision(p: str) -> None:
    """"fp32": CUDA-core fp32 arithmetic end to end (parity mode).
    "bf16": bf16 tensor-core GEMMs / recurrence with fp32 accumulation and fp32 master weights."""
    global _DEFAULT_PRECISION
    if p not in ("fp32", "bf16"):
        raise ValueError(p)
    _DEFAULT_PRECISION = p


def default_precision() -> str:
    return _DEFAULT_PRECISION


def gaussian_kernel_1d(kernel_size: int, sigma: float) -> torch.Tensor:
    """Normalised Gaussian taps, float32, as GaussianSmoothing builds them (augmentations.py:41-63)."""
    grid = torch.arange(kernel_size, dtype=torch.float32)
    mean = (kernel_size - 1) / 2
    k = 1 / (sigma * math.sqrt(2 * math.pi)) * torch.exp(-(((grid - mean) / sigma) ** 2) / 2)   # sigma=0 -> ZeroDivisionError
    return k / torch.sum(k)


class _GaussianSmootherState(nn.Module):
    """Holds the ``gaussianSmoother.weight`` buffer [N,1,20] of the reference (augmentations.py:66-69)."""

    def __init__(self, channels: int, kernel_size: int, sigma: float):
        super().__init__()
        k = gaussian_kernel_1d(kernel_size, sigma)
        self.register_buffer("weight", k.view(1, 1, -1).repeat(channels, 1, 1))
        self.groups = channels


class _GRUParameters(nn.Module):
    """Parameter container with nn.GRU's names, shapes, registration order and default init
    (uniform(-1/sqrt(H), 1/sqrt(H)) in registration order), so state dicts and seeded inits match
    ``nn.GRU(input, hidden, layers, bidirectional=...)`` (model.py:50-57).  It owns no compute."""

    def __init__(self, input_size: int, hidden_size: int, num_layers: int, bidirectional: bool):
        super().__init__()
        self.input_size, self.hidden_size, self.num_layers, self.bidirectional = input_size, hidden_size, num_layers, bidirectional
        D = 2 if bidirectional else 1
        for layer in range(num_layers):
            in_l = input_size if layer == 0 else hidden_size * D
            for d in range(D):
                sfx = "_reverse" if d == 1 else ""
                self.register_parameter(f"weight_ih_l{layer}{sfx}", nn.Parameter(torch.empty(3 * hidden_size, in_l)))
                self.register_parameter(f"weight_hh_l{layer}{sfx}", nn.Parameter(torch.empty(3 * hidden_size, hidden_size)))
                self.register_parameter(f"bias_ih_l{layer}{sfx}", nn.Parameter(torch.empty(3 * hidden_size)))
                self.register_parameter(f"bias_hh_l{layer}{sfx}", nn.Parameter(torch.empty(3 * hidden_size)))
        stdv = 1.0 / math.sqrt(hidden_size) if hidden_size > 0 else 0
        for w in self.parameters():
            nn.init.uniform_(w, -stdv, stdv)


class GRUDecoder(nn.Module):
    def __init__(self, neural_dim, n_classes, hidden_dim, layer_dim, nDays=24, dropout=0, device="cuda",
                 strideLen=4, kernelLen=14, gaussianSmoothWidth=0, bidirectional=False):
        super().__init__()
        self.layer_dim = layer_dim
        self.hidden_dim = hidden_dim
        self.neural_dim = neural_dim
        self.n_classes = n_classes
        self.nDays = nDays
        self.device = device
        self.dropout = dropout
        self.strideLen = strideLen
        self.kernelLen = kernelLen
        self.gaussianSmoothWidth = gaussianSmoothWidth
        self.bidirectional = bidirectional
        self.precision = _DEFAULT_PRECISION
        self.gaussianSmoother = _GaussianSmootherState(neural_dim, 20, gaussianSmoothWidth)
        self.dayWeights = nn.Parameter(torch.randn(nDays, neural_dim, neural_dim))
        self.dayBias = nn.Parameter(torch.zeros(nDays, 1, neural_dim))
        with torch.no_grad():
            self.dayWeights.copy_(torch.eye(neural_dim).expand(nDays, -1, -1))

        self.gru_decoder = _GRUParameters(neural_dim * kernelLen, hidden_dim, layer_dim, bidirectional)
        for name, param in self.gru_decoder.named_parameters():
            if "weight_hh" in name:
                nn.init.orthogonal_(param)
            if "weight_ih" in name:
                nn.init.xavier_uniform_(param)

        # per-day input layers: present in the reference's state dict but never used by forward (model.py:66-73)
        for d in range(nDays):
            lin = nn.Linear(neural_dim, neural_dim)
            lin.weight = nn.Parameter(lin.weight + torch.eye(neural_dim))
            setattr(self, "inpLayer" + str(d), lin)

        self.fc_decoder_out = nn.Linear(hidden_dim * (2 if bidirectional else 1), n_classes + 1)   # +1: CTC blank
        self._step = 0
        self._err_flag: Optional[torch.Tensor] = None
        self.grad_sync = None       # parallel.GradSync when training data-parallel (set by trainer.train_step)
        self.step_hook = None       # trainer._UpdateSchedule: optimizer updates from inside the backward (set by trainer.train_step)
        # (whiteNoiseSD, constantOffsetSD) of the trainer's in-loop augmentation (trainer:194-201), applied inside K1 while
        # the module is in train mode; None = the caller adds its own noise (or none), as in the reference
        self.input_noise = None
        self._shadows = Bf16Shadows()   # bf16 operand copies of the weights (bf16 precision only), see FusedAdam.attach_shadows

    # ---------------------------------------------------------------- helpers
    def _gru_weights(self) -> List[torch.Tensor]:
        out = []
        D = 2 if self.bidirectional else 1
        for layer in range(self.layer_dim):
            for d in range(D):
                sfx = "_reverse" if d == 1 else ""
                g = self.gru_decoder
                out += [getattr(g, f"weight_ih_l{layer}{sfx}"), getattr(g, f"weight_hh_l{layer}{sfx}"),
                        getattr(g, f"bias_ih_l{layer}{sfx}"), getattr(g, f"bias_hh_l{layer}{sfx}")]
        return out

    def invalidate_weight_copies(self) -> None:
        """Call after writing parameters through ``.data`` / raw pointers (autograd cannot see those writes): the kept
        bf16 operand copies are re-made by the next forward."""
        self._shadows.invalidate()

    def check_errors(self) -> None:
        """Raise the deferred IndexError of an out-of-range dayIdx, or the ValueError of an X_len outside [kernelLen, T] given on
        the device (the kernels flag them asynchronously)."""
        if self._err_flag is not None:
            v = int(self._err_flag.item())
            if v != 0:
                self._err_flag.zero_()
                if v & 1:
                    raise IndexError("index out of range in dayIdx (expected 0 <= dayIdx < nDays)")
                raise ValueError(f"X_len out of range (expected kernelLen={self.kernelLen} <= X_len <= T)")

    def forward(self, neuralInput: torch.Tensor, dayIdx: torch.Tensor, X_len: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``X_len`` (int [B], host or device; None = the reference's padded batch): utterance b is computed as if it ran alone
        on ``neuralInput[b, :X_len[b]]``, as ``nn.GRU`` does on a packed sequence.  Bins at or past X_len[b] are read as 0, the
        recurrence of b runs its own n_b = (X_len[b] - kernelLen) // strideLen + 1 frames in each direction, the logits at
        frames t >= n_b are exactly ``fc_decoder_out.bias``, and no gradient flows through those frames or bins.  A host X_len
        outside [kernelLen, T] raises ValueError; on the device it is flagged for ``check_errors()``."""
        if not neuralInput.is_cuda:
            raise NsdError("GRUDecoder (B200) runs on CUDA tensors only; there is no CPU path")
        if neuralInput.dim() != 3 or neuralInput.shape[2] != self.neural_dim:
            raise RuntimeError(f"neuralInput must be [B,T,{self.neural_dim}], got {tuple(neuralInput.shape)}")
        if self.precision != "fp32":
            check_architecture(self.neural_dim, self.kernelLen, self.hidden_dim)
        if not dayIdx.is_cuda:      # cheap host-side check when the indices are still on the host
            if dayIdx.numel() and (int(dayIdx.min()) < 0 or int(dayIdx.max()) >= self.nDays):
                raise IndexError("index out of range in dayIdx (expected 0 <= dayIdx < nDays)")
        if X_len is not None:
            B, T = neuralInput.shape[0], neuralInput.shape[1]
            if X_len.dim() != 1 or X_len.shape[0] != B or X_len.dtype.is_floating_point or X_len.dtype == torch.bool:
                raise ValueError(f"X_len must be an integer tensor of shape [{B}], got {X_len.dtype} {tuple(X_len.shape)}")
            if not X_len.is_cuda and B and (int(X_len.min()) < self.kernelLen or int(X_len.max()) > T):
                raise ValueError(f"X_len out of range (expected kernelLen={self.kernelLen} <= X_len <= T={T})")
            X_len = X_len.to(device=neuralInput.device, dtype=torch.int64).contiguous()
        if self._err_flag is None or self._err_flag.device != neuralInput.device:
            self._err_flag = torch.zeros(1, dtype=torch.int32, device=neuralInput.device)
        cfg = dict(K=self.kernelLen, S=self.strideLen, H=self.hidden_dim, L=self.layer_dim,
                   D=2 if self.bidirectional else 1, n_days=self.nDays, precision=self.precision,
                   p_drop=float(self.dropout) if self.training else 0.0, seed=0, err_flag=self._err_flag,
                   grad_sync=self.grad_sync, shadows=self._shadows, step_hook=self.step_hook, x_len=X_len)
        noisy = self.training and self.input_noise is not None and any(float(v) != 0.0 for v in self.input_noise)
        if cfg["p_drop"] > 0 or noisy:
            self._step += 1
            cfg["seed"] = (int(torch.initial_seed()) * 1000003 + self._step) & 0x7FFFFFFFFFFFFFFF
        cfg["noise"] = (float(self.input_noise[0]), float(self.input_noise[1]), cfg["seed"] ^ 0x5DEECE66D) if noisy else None
        taps = self.gaussianSmoother.weight[0, 0].contiguous()
        params = (self.dayWeights, self.dayBias, self.fc_decoder_out.weight, self.fc_decoder_out.bias, *self._gru_weights())
        for p in params:
            if p.device != neuralInput.device:
                raise NsdError(f"GRUDecoder parameters live on {p.device} but neuralInput on {neuralInput.device}")
        # grad mode is always off inside autograd.Function.forward: decide here whether the BPTT saves are needed
        cfg["need_grad"] = torch.is_grad_enabled() and (neuralInput.requires_grad or any(p.requires_grad for p in params))
        # raw pointers are handed to the C ABI: the CUDA runtime's current device (kernel launches, TMA maps, cooperative
        # launches) and the stream must be the tensors' device, whatever the caller's current device is
        with torch.cuda.device(neuralInput.device):
            return _DecoderFunction.apply(cfg, neuralInput, dayIdx, taps, *params)


def _flat_views(shapes, dev, zero=False):
    """Views of ONE flat f32 buffer (a gradient bucket).  ``views[0]._base`` is the flat buffer."""
    sizes = [int(torch.Size(s).numel()) for s in shapes]
    flat = (torch.zeros if zero else torch.empty)(sum(sizes), device=dev, dtype=torch.float32)
    out, off = [], 0
    for s, n in zip(shapes, sizes):
        out.append(flat[off:off + n].view(s))
        off += n
    return out


def grad_plan(ctx):
    """-> (dx wanted, [wanted] per parameter in ``ctx.params`` order), from ``ctx.needs_input_grad``.  With ``grad_sync`` or
    ``step_hook`` set (train_step's data-parallel and in-backward update paths) every GRU and output-layer gradient is made, as
    those paths expect one per bucket; the day parameters follow their flags in every case."""
    ni = ctx.needs_input_grad
    need = [bool(v) for v in ni[4:]]
    if ctx.cfg.get("grad_sync") is not None or ctx.cfg.get("step_hook") is not None:
        need[2:] = [True] * (len(need) - 2)
    return bool(ni[1]), need


def _assign_grads(params, grads):
    """Data-parallel mode: the buckets are being all-reduced in place on NCCL's stream, so the parameters must
    end up pointing AT the bucket views (autograd's AccumulateGrad may clone a view, which would capture the
    un-reduced values).  The usual zero_grad(set_to_none=True) -> backward -> step loop is the supported one."""
    for p, g in zip(params, grads):
        if g is None or not isinstance(p, torch.Tensor) or not p.requires_grad:
            continue
        if p.grad is not None:
            raise RuntimeError("data-parallel backward needs optimizer.zero_grad(set_to_none=True) before it")
        p.grad = g
    return (None,) * len(params)


# ---------------------------------------------------------------- layer stacks
# ``gru_w`` holds the GRU parameters in ``GRUDecoder._gru_weights`` order (4 per layer and direction).  The fp32 stack runs one
# direction per launch with a separate dropout pass; the bf16 stack runs both directions in one GEMM / one recurrence launch
# with stacked weights, the dropout fused into the recurrence's epilogue and the bias sums of the BPTT done in-kernel.

def stack_fwd_f32(inp, gru_w, Tp, B, H, D, need_grad, p_drop, seed, nf):
    """fp32 layer stack on the time-major rows ``inp``.  -> (per layer (input, hseq, saves per direction), output-layer input)."""
    dev = inp.device
    M = Tp * B
    L = len(gru_w) // (4 * D)
    layers = []
    gi = torch.empty((M, D * 3 * H), device=dev, dtype=torch.float32)
    for l in range(L):
        in_l = inp.shape[1]
        hseq = torch.empty((M, D * H), device=dev, dtype=torch.float32)
        saves = []
        for d in range(D):
            w_ih, w_hh, b_ih, b_hh = (t.detach() for t in gru_w[(l * D + d) * 4:(l * D + d) * 4 + 4])
            ops.gemm(False, True, M, 3 * H, in_l, inp, in_l, w_ih, in_l, gi, D * 3 * H, bias=b_ih, c_off=d * 3 * H)
            sv = tuple(torch.empty((M, H), device=dev, dtype=torch.float32) for _ in range(4)) if need_grad else None
            ops.gru_fwd_f32(gi, D * 3 * H, d * 3 * H, w_hh, b_hh, Tp, B, H, d == 1, hseq, D * H, d * H, sv, n_frames=nf)
            saves.append(sv)
        nxt = hseq
        if p_drop > 0 and l < L - 1:
            nxt = ops.dropout(hseq, p_drop, seed + l)
        layers.append((inp, hseq, saves))
        inp = nxt
    return layers, inp


def stack_fwd_bf16(inp, gru_w, sh, Tp, B, H, D, need_grad, p_drop=0.0, seed=0, nf=None, h0=None):
    """bf16 tensor-core layer stack on the time-major bf16 rows ``inp``, its weight operands taken from ``sh`` (Bf16Shadows).
    ``h0`` ([L, B, H] f32, one forward direction only, no saves, no dropout): each layer's initial state instead of zeros
    (streaming).  -> (per layer (input, hseq, hseq bf16, saves, W_ih operand, W_hh^T operand), output-layer input)."""
    if h0 is not None and (need_grad or p_drop > 0):
        raise NsdError("stack_fwd_bf16: an initial state h0 is for an inference stack without dropout")
    dev = inp.device
    M = Tp * B
    L = len(gru_w) // (4 * D)
    layers = []
    # both directions run in one GEMM / one recurrence launch: their bias vectors side by side, packed in ONE launch
    if D > 1:
        bias_all = torch.empty((L, 2, D * 3 * H), device=dev, dtype=torch.float32)
        ops.multi_copy([gru_w[(l * D + d) * 4 + 2 + k].detach() for l in range(L) for k in range(2) for d in range(D)],
                       [bias_all[l, k, d * 3 * H:(d + 1) * 3 * H] for l in range(L) for k in range(2) for d in range(D)])
    # gru_w holds the Parameters themselves: their version counters tell whether the kept bf16 copies are current.  Without h0 every
    # layer's W_hh copy is taken up front (the BPTT operands are transposed from all of them in one launch); the streaming form (h0)
    # takes each in its own layer, behind the layer's W_ih copy, so a stale copy is re-made where that form has always re-made it
    w_hh = lambda l: sh.stacked(("hh", l), [gru_w[(l * D + d) * 4 + 1] for d in range(D)])        # [D*3H, H]
    w_hh_all = [w_hh(l) for l in range(L)] if h0 is None else None
    w_hhT_all = None
    if need_grad:                                            # BPTT operands [D*H, 3H] of every layer, all transposed in one launch
        w_hhT_all = torch.empty((L, D * H, 3 * H), device=dev, dtype=torch.bfloat16)
        ops.transpose_bf16_multi([w_hh_all[l][d * 3 * H:(d + 1) * 3 * H] for l in range(L) for d in range(D)],
                                 [w_hhT_all[l, d * H:(d + 1) * H] for l in range(L) for d in range(D)])
    for l in range(L):
        in_l = inp.shape[1]
        ws = [[t.detach() for t in gru_w[(l * D + d) * 4:(l * D + d) * 4 + 4]] for d in range(D)]
        w_ih_bf = sh.stacked(("ih", l), [gru_w[(l * D + d) * 4] for d in range(D)])          # [D*3H, in_l]
        w_hh_bf = w_hh(l) if h0 is not None else w_hh_all[l]
        w_hhT_bf = w_hhT_all[l] if need_grad else None
        b_ih, b_hh = (bias_all[l, 0], bias_all[l, 1]) if D > 1 else (ws[0][2], ws[0][3])
        gi = torch.empty((M, D * 3 * H), device=dev, dtype=torch.float32)
        ops.gemm(False, True, M, D * 3 * H, in_l, inp, in_l, w_ih_bf, in_l, gi, D * 3 * H, bias=b_ih.contiguous())
        if p_drop > 0 and l < L - 1:      # inter-layer dropout fused into the recurrence's epilogue
            hseq, hseq_bf, saves, nxt = ops.gru_fwd_bf16(gi, w_hh_bf, b_hh.contiguous(), Tp, B, H, D, False, need_grad,
                                                         p_drop, seed + l, n_frames=nf)
        else:
            hseq, hseq_bf, saves = ops.gru_fwd_bf16(gi, w_hh_bf, b_hh.contiguous(), Tp, B, H, D, False, need_grad,
                                                    h0=None if h0 is None else h0[l], n_frames=nf)
            nxt = hseq_bf
        del gi
        layers.append((inp, hseq, hseq_bf, saves, w_ih_bf, w_hhT_bf))
        inp = nxt
    return layers, inp


def layer_bwd_f32(ctx, l, dh, need_gru, ggru, want_dinp, gs):
    """Backward of fp32 layer ``l`` from ``dh`` (the gradient of its output): fills ``ggru`` with the layer's weight gradients
    (one flat bucket, handed to ``gs`` once final) and returns the gradient of its input (None unless ``want_dinp``)."""
    cfg = ctx.cfg
    H, L, D = cfg["H"], cfg["L"], cfg["D"]
    B, _, _, Tp = ctx.dims
    M = Tp * B
    gru_w, nf = ctx.weights[2], ctx.lengths[1]
    dev = dh.device
    f32 = dict(device=dev, dtype=torch.float32)
    inp, hseq, saves = ctx.layers[l]
    in_l = inp.shape[1]
    if cfg["p_drop"] > 0 and l < L - 1:
        dh = ops.dropout(dh, cfg["p_drop"], cfg["seed"] + l)
    dgi = torch.empty((M, D * 3 * H), **f32)
    dghn = [torch.empty((M, H), **f32) for _ in range(D)]
    for d in range(D):
        w_hh = gru_w[(l * D + d) * 4 + 1].detach()
        ops.gru_bwd_f32(dh, D * H, d * H, hseq, D * H, d * H, saves[d], w_hh, Tp, B, H, d == 1,
                        dgi, D * 3 * H, d * 3 * H, dghn[d], n_frames=nf)
    dinp = torch.empty((M, in_l), **f32) if want_dinp else None
    wgrad = any(need_gru[l * D * 4:(l + 1) * D * 4])
    # one flat bucket per layer: its all-reduce starts while the layers below are still in BPTT
    views = _flat_views([(3 * H, in_l), (3 * H, H), (3 * H,), (3 * H,)] * D, dev, zero=(Tp == 1)) if wgrad else None
    for d in range(D):
        base = (l * D + d) * 4
        w_ih = gru_w[base].detach()
        if wgrad:
            n_wih, n_whh, n_bih, n_bhh = need_gru[base:base + 4]
            d_w_ih, d_w_hh, d_b_ih, d_b_hh = views[4 * d:4 * d + 4]
            if n_wih:
                ops.gemm(True, False, 3 * H, in_l, M, dgi, D * 3 * H, inp, in_l, d_w_ih, in_l, a_off=d * 3 * H)
            if n_bih or n_bhh:
                ops.colsum(dgi, M, 3 * H, D * 3 * H, d_b_ih, a_off=d * 3 * H)
            if n_bhh:
                d_b_hh[:2 * H].copy_(d_b_ih[:2 * H])
                ops.colsum(dghn[d], M, H, H, d_b_hh, out_off=2 * H)
            if n_whh and Tp > 1:
                Mh = (Tp - 1) * B
                # forward dir: h_{t-1} = hseq[t-1] pairs with dgh[t];  reverse dir: h_{t-1} = hseq[t+1] pairs with dgh[t]
                g_off = (0 if d == 1 else B)
                h_off = (B if d == 1 else 0)
                ops.gemm(True, False, 2 * H, H, Mh, dgi, D * 3 * H, hseq, D * H, d_w_hh, H,
                         a_off=g_off * D * 3 * H + d * 3 * H, b_off=h_off * D * H + d * H)
                ops.gemm(True, False, H, H, Mh, dghn[d], H, hseq, D * H, d_w_hh, H,
                         a_off=g_off * H, b_off=h_off * D * H + d * H, c_off=2 * H * H)
            ggru[base:base + 4] = [g if n else None for g, n in zip((d_w_ih, d_w_hh, d_b_ih, d_b_hh), need_gru[base:base + 4])]
        if dinp is not None:
            ops.gemm(False, False, M, in_l, 3 * H, dgi, D * 3 * H, w_ih, in_l, dinp, in_l,
                     beta=1.0 if d > 0 else 0.0, a_off=d * 3 * H)
    if gs is not None:
        gs.bucket_ready(views[0]._base)
    return dinp


def layer_bwd_bf16(ctx, l, dh, need_gru, ggru, want_dinp, gs, schedule):
    """Backward of bf16 layer ``l``, as ``layer_bwd_f32``; ``schedule`` (trainer._UpdateSchedule or None) issues the BPTT launch and
    is told when the layer's bucket is final."""
    cfg = ctx.cfg
    H, L, D = cfg["H"], cfg["L"], cfg["D"]
    B, _, _, Tp = ctx.dims
    M, Mh = Tp * B, (Tp - 1) * B
    gru_w, nf = ctx.weights[2], ctx.lengths[1]
    dev = dh.device
    inp, hseq, hseq_bf, saves, w_ih_bf, w_hhT_bf = ctx.layers[l]
    in_l = inp.shape[1]
    # what this layer's parameters need, each kind over both directions (one GEMM / one BPTT reduction covers both)
    n_wih, n_whh, n_b = (any(need_gru[(l * D + d) * 4 + k] for d in range(D) for k in ks) for ks in ((0,), (1,), (2, 3)))
    wgrad = n_wih or n_whh or n_b
    # one flat bucket per layer, laid out so that each GEMM writes its whole (both-direction) block at once
    v_wih = v_whh = v_bih = v_bhh = None
    if wgrad:
        v_wih, v_whh, v_bih, v_bhh = _flat_views([(D * 3 * H, in_l), (D * 3 * H, H), (D * 3 * H,), (D * 3 * H,)], dev,
                                                 zero=(Tp == 1))
    drop = cfg["p_drop"] if (cfg["p_drop"] > 0 and l < L - 1) else 0.0
    # BPTT with the output-dropout mask applied on load and the bias gradients (column sums) accumulated in-kernel
    db = (v_bih, v_bhh) if n_b else (None, None)
    bptt = lambda: ops.gru_bwd_bf16(dh, hseq, saves, w_hhT_bf, Tp, B, H, D, False, drop, cfg["seed"] + l, *db, n_frames=nf)
    dgi, dgh = schedule.bptt(bptt) if schedule is not None else bptt()
    # wgrad W_ih: dW[D*3H, in_l] = dgi^T inp -- reduction over the T'*B rows, both operands M/N-major as stored
    if n_wih:
        ops.gemm(True, False, D * 3 * H, in_l, M, dgi, D * 3 * H, inp, in_l, v_wih, in_l)
    if n_whh and Tp > 1:
        # forward dir: dgh[t] pairs with h[t-1];  reverse dir: dgh[t] pairs with h[t+1]  (row-range views, no copies)
        offs = [((B if d == 0 else 0) * D * 3 * H + d * 3 * H, (0 if d == 0 else B) * D * H + d * H, d * 3 * H * H) for d in range(D)]
        if D == 2:                      # both directions in one launch
            ops.gemm_x2(True, False, 3 * H, H, Mh, dgh, D * 3 * H, hseq_bf, D * H, v_whh, H,
                        [o[0] for o in offs], [o[1] for o in offs], [o[2] for o in offs])
        else:
            ops.gemm(True, False, 3 * H, H, Mh, dgh, D * 3 * H, hseq_bf, D * H, v_whh, H,
                     a_off=offs[0][0], b_off=offs[0][1], c_off=offs[0][2])
    # the layer's bucket is final once its wgrads are issued.  With SMs reserved for NCCL (GradSync.reserve_sms) the
    # all-reduce starts now and runs under the dgrad GEMM below; without a reserve NCCL's CTAs would displace CTAs of the
    # 148-wide persistent GEMM, so the bucket is released after it (measured: no gain at 8 GPUs)
    tail = gs is not None and l == 0 and getattr(gs, "tail_sms", 0) > 0 and getattr(gs, "world", 1) > 1
    early = gs is not None and (getattr(gs, "reserve_sms", 0) > 0 or tail)
    handle = gs.bucket_ready(v_wih._base) if early else None
    if tail:           # the last big bucket: its all-reduce runs on the SMs this one GEMM leaves free (measured timeline: profiles/r02_allreduce_timeline_*.json)
        call("nsd_set_gemm_sm_reserve", gs.tail_sms)
    dinp = None
    if want_dinp:
        dinp = torch.empty((M, in_l), device=dev, dtype=torch.float32 if l > 0 else torch.bfloat16)
        ops.gemm(False, False, M, in_l, D * 3 * H, dgi, D * 3 * H, w_ih_bf, in_l, dinp, in_l)       # dgrad: dgi W_ih
    if tail:
        call("nsd_set_gemm_sm_reserve", 0)
    for d in range(D):
        base = (l * D + d) * 4
        if wgrad:
            ggru[base:base + 4] = [v[d * 3 * H:(d + 1) * 3 * H] if n else None
                                   for v, n in zip((v_wih, v_whh, v_bih, v_bhh), need_gru[base:base + 4])]
    if gs is not None and not early:
        handle = gs.bucket_ready(v_wih._base)
    if schedule is not None:
        schedule.released([(gru_w[(l * D + d) * 4 + k], ggru[(l * D + d) * 4 + k]) for d in range(D) for k in range(4)], handle)
    return dinp


class _DecoderFunction(torch.autograd.Function):
    """forward: K1 -> layer stack (per layer: K2 input GEMM, K3 recurrence, dropout) -> K2 output layer.
    backward: the hand-written reverse of that chain (SURVEY.md section 8a, a14).
    The precision picks the front end's output dtype, the layer stack and its backward, and the output layer's weight operand
    (the fp32 weight, or its kept bf16 copy); everything around them is shared.  bf16: the dense contractions on tcgen05 with
    fp32 accumulation; parameters stay fp32 (master weights), and hidden state, gate math, saved activations and all parameter
    gradients are fp32."""

    @staticmethod
    def forward(ctx, cfg, x, day_idx, taps, day_w, day_b, fc_w, fc_b, *gru_w):
        K, S, H, D = cfg["K"], cfg["S"], cfg["H"], cfg["D"]
        bf16 = cfg["precision"] != "fp32"
        dev = x.device
        B, T, N = x.shape
        Tp = ops.n_frames(T, K, S)
        M = Tp * B
        day_idx = day_idx.to(device=dev, dtype=torch.int64).contiguous()
        need_grad = cfg.get("need_grad", True)
        x_len = cfg.get("x_len")
        nf = ops.frame_counts(x_len, T, K, S, cfg["err_flag"]) if x_len is not None else None     # packed rows (GRUDecoder.forward)
        patches, ys, z = ops.frontend_fwd(x, day_idx, day_w.detach().contiguous(), day_b.detach().contiguous(), taps, K, S,
                                          torch.bfloat16 if bf16 else torch.float32, cfg["err_flag"], cfg.get("noise"), x_len=x_len)
        if bf16:
            sh = cfg.get("shadows") or Bf16Shadows()         # the module's cache of bf16 weight copies (a throw-away one otherwise)
            layers, hid = stack_fwd_bf16(patches, gru_w, sh, Tp, B, H, D, need_grad, cfg["p_drop"], cfg["seed"], nf)
            fc_w_op = sh.stacked(("fc", 0), [fc_w])
        else:
            layers, hid = stack_fwd_f32(patches, gru_w, Tp, B, H, D, need_grad, cfg["p_drop"], cfg["seed"], nf)
            fc_w_op = fc_w.detach()
        C = fc_w.shape[0]
        logits_tm = torch.empty((M, C), device=dev, dtype=torch.float32)
        ops.gemm(False, True, M, C, D * H, hid, D * H, fc_w_op, D * H, logits_tm, C, bias=fc_b.detach().contiguous())
        logits = ops.swap01(logits_tm.view(Tp, B, C))
        if need_grad:
            ctx.cfg = cfg
            ctx.dims = (B, T, N, Tp)
            ctx.layers = layers
            ctx.hid = hid
            ctx.front = (ys, z, day_idx, taps)
            ctx.lengths = (x_len, nf)
            ctx.weights = (day_w, fc_w_op, gru_w)
            ctx.params = (day_w, day_b, fc_w, fc_b) + tuple(gru_w)
        return logits

    @staticmethod
    @once_differentiable
    def backward(ctx, dlogits):
        with torch.cuda.device(dlogits.device):
            return _DecoderFunction._backward(ctx, dlogits)

    @staticmethod
    def _backward(ctx, dlogits):
        cfg = ctx.cfg
        K, S, H, L, D = cfg["K"], cfg["S"], cfg["H"], cfg["L"], cfg["D"]
        bf16 = cfg["precision"] != "fp32"
        B, T, N, Tp = ctx.dims
        M = Tp * B
        day_w, fc_w_op, gru_w = ctx.weights
        dev = dlogits.device
        C = fc_w_op.shape[0]
        gs = cfg.get("grad_sync")
        # trainer._UpdateSchedule: updates finished buckets from inside the backward (train_step sets one for bf16 only)
        schedule = cfg.get("step_hook") if bf16 else None
        want_x, need = grad_plan(ctx)
        need_gru = need[4:]
        dl_tm = ops.swap01(dlogits.contiguous().float()).view(M, C)         # [B,T',C] -> time-major rows
        dl, ldl = dl_tm, C
        if bf16:        # the tensor-core GEMMs read a bf16 copy, rows padded to 16 bytes
            ldl = (C + 7) // 8 * 8
            dl = torch.empty((M, ldl), device=dev, dtype=torch.bfloat16)
            ops.cast_transpose_into(dl_tm, dl[:, :C], None)
        d_fc_w = d_fc_b = None
        if need[2] or need[3]:
            d_fc_w, d_fc_b = _flat_views([(C, D * H), (C,)], dev)
            if need[2]:
                ops.gemm(True, False, C, D * H, M, dl, ldl, ctx.hid, D * H, d_fc_w, D * H)          # d_fc_w = dl^T hid
            if need[3]:
                ops.colsum(dl_tm, M, C, C, d_fc_b)
            handle = gs.bucket_ready(d_fc_w._base) if gs is not None else None
            if schedule is not None:
                schedule.released([(ctx.params[2], d_fc_w), (ctx.params[3], d_fc_b)], handle)
        dh = torch.empty((M, D * H), device=dev, dtype=torch.float32)
        ops.gemm(False, False, M, D * H, C, dl, ldl, fc_w_op, D * H, dh, D * H)                     # dh = dl fc_w
        ggru: List[Optional[torch.Tensor]] = [None] * len(gru_w)
        want_front = want_x or need[0] or need[1]
        for l in range(L - 1, -1, -1):
            if bf16:
                dh = layer_bwd_bf16(ctx, l, dh, need_gru, ggru, l > 0 or want_front, gs, schedule)
            else:
                dh = layer_bwd_f32(ctx, l, dh, need_gru, ggru, l > 0 or want_front, gs)
            ctx.layers[l] = None
        ys, z, day_idx, taps = ctx.front
        x_len = ctx.lengths[0]
        d_day_w = d_day_b = dx = None
        if dh is not None:
            if need[0] or need[1]:
                d_day_w, d_day_b = ops.frontend_bwd(dh, ys, z, day_idx, cfg["n_days"], K, S)
                if gs is not None:
                    gs.bucket_ready(d_day_w._base)
            if want_x:
                dx = ops.frontend_bwd_input(dh, z, day_idx, day_w.detach().contiguous(), taps, K, S, x_len=x_len)
        ctx.layers = ctx.hid = ctx.front = ctx.lengths = None
        grads = (d_day_w, d_day_b, d_fc_w, d_fc_b, *ggru)
        if schedule is not None:
            grads = schedule.not_updated(ctx.params, grads)
        if gs is not None:
            grads = _assign_grads(ctx.params, grads)
        return (None, dx, None, None) + grads
