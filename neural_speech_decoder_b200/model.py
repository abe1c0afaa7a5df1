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
from ._lib import NsdError

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
        from .model_tc import Bf16Shadows
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
        """Raise the deferred IndexError of an out-of-range dayIdx (the kernel flags it asynchronously)."""
        if self._err_flag is not None and int(self._err_flag.item()) != 0:
            self._err_flag.zero_()
            raise IndexError("index out of range in dayIdx (expected 0 <= dayIdx < nDays)")

    def forward(self, neuralInput: torch.Tensor, dayIdx: torch.Tensor) -> torch.Tensor:
        if not neuralInput.is_cuda:
            raise NsdError("GRUDecoder (B200) runs on CUDA tensors only; there is no CPU path")
        if neuralInput.dim() != 3 or neuralInput.shape[2] != self.neural_dim:
            raise RuntimeError(f"neuralInput must be [B,T,{self.neural_dim}], got {tuple(neuralInput.shape)}")
        if self.precision != "fp32":
            from .model_tc import check_architecture
            check_architecture(self.neural_dim, self.kernelLen, self.hidden_dim)
        if not dayIdx.is_cuda:      # cheap host-side check when the indices are still on the host
            if dayIdx.numel() and (int(dayIdx.min()) < 0 or int(dayIdx.max()) >= self.nDays):
                raise IndexError("index out of range in dayIdx (expected 0 <= dayIdx < nDays)")
        if self._err_flag is None or self._err_flag.device != neuralInput.device:
            self._err_flag = torch.zeros(1, dtype=torch.int32, device=neuralInput.device)
        cfg = dict(K=self.kernelLen, S=self.strideLen, H=self.hidden_dim, L=self.layer_dim,
                   D=2 if self.bidirectional else 1, n_days=self.nDays, precision=self.precision,
                   p_drop=float(self.dropout) if self.training else 0.0, seed=0, err_flag=self._err_flag,
                   grad_sync=self.grad_sync, shadows=self._shadows, step_hook=self.step_hook)
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


def _flat_views(shapes, dev, grad_sync, zero=False):
    """Views of ONE flat f32 buffer (a gradient bucket); if ``grad_sync`` is given the bucket is all-reduced
    by the caller once filled.  ``views[0]._base`` is the flat buffer."""
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


class _DecoderFunction(torch.autograd.Function):
    """forward: K1 -> per layer (K2 input GEMM, K3 recurrence per direction, dropout) -> K2 output layer.
    backward: the hand-written reverse of that chain (SURVEY.md section 8a, a14)."""

    @staticmethod
    def forward(ctx, cfg, x, day_idx, taps, day_w, day_b, fc_w, fc_b, *gru_w):
        K, S, H, L, D = cfg["K"], cfg["S"], cfg["H"], cfg["L"], cfg["D"]
        if cfg["precision"] != "fp32":
            from .model_tc import decoder_forward_tc
            return decoder_forward_tc(ctx, cfg, x, day_idx, taps, day_w, day_b, fc_w, fc_b, *gru_w)
        dev = x.device
        B, T, N = x.shape
        Tp = ops.n_frames(T, K, S)
        M = Tp * B
        day_idx = day_idx.to(device=dev, dtype=torch.int64).contiguous()
        need_grad = cfg.get("need_grad", True)
        patches, ys, z = ops.frontend_fwd(x, day_idx, day_w.detach().contiguous(), day_b.detach().contiguous(), taps,
                                          K, S, torch.float32, cfg["err_flag"], cfg.get("noise"))
        inp = patches
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
                ops.gru_fwd_f32(gi, D * 3 * H, d * 3 * H, w_hh, b_hh, Tp, B, H, d == 1, hseq, D * H, d * H, sv)
                saves.append(sv)
            nxt = hseq
            if cfg["p_drop"] > 0 and l < L - 1:
                nxt = ops.dropout(hseq, cfg["p_drop"], cfg["seed"] + l)
            layers.append((inp, hseq, saves))
            inp = nxt
        C = fc_w.shape[0]
        logits_tm = torch.empty((M, C), device=dev, dtype=torch.float32)
        ops.gemm(False, True, M, C, D * H, inp, D * H, fc_w.detach(), D * H, logits_tm, C, bias=fc_b.detach())
        logits = ops.swap01(logits_tm.view(Tp, B, C))
        if need_grad:
            ctx.cfg = cfg
            ctx.dims = (B, T, N, Tp)
            ctx.layers = layers
            ctx.hid = inp
            ctx.front = (ys, z, day_idx, taps)
            ctx.weights = (day_w, fc_w, gru_w)
            ctx.params = (day_w, day_b, fc_w, fc_b) + tuple(gru_w)
        return logits

    @staticmethod
    @once_differentiable
    def backward(ctx, dlogits):
        with torch.cuda.device(dlogits.device):
            if ctx.cfg["precision"] != "fp32":
                from .model_tc import decoder_backward_tc
                return decoder_backward_tc(ctx, dlogits)
            return _DecoderFunction._backward_f32(ctx, dlogits)

    @staticmethod
    def _backward_f32(ctx, dlogits):
        cfg = ctx.cfg
        K, S, H, L, D = cfg["K"], cfg["S"], cfg["H"], cfg["L"], cfg["D"]
        B, T, N, Tp = ctx.dims
        M = Tp * B
        day_w, fc_w, gru_w = ctx.weights
        dev = dlogits.device
        C = fc_w.shape[0]
        f32 = dict(device=dev, dtype=torch.float32)
        want_x, need = grad_plan(ctx)
        need_gru = need[4:]
        dl_tm = ops.swap01(dlogits.contiguous().float()).view(M, C)         # [B,T',C] -> time-major rows
        hid = ctx.hid
        gs = cfg.get("grad_sync")
        d_fc_w = d_fc_b = None
        if need[2] or need[3]:
            d_fc_w, d_fc_b = _flat_views([(C, D * H), (C,)], dev, gs)
            if need[2]:
                ops.gemm(True, False, C, D * H, M, dl_tm, C, hid, D * H, d_fc_w, D * H)
            if need[3]:
                ops.colsum(dl_tm, M, C, C, d_fc_b)
            if gs is not None:
                gs.bucket_ready(d_fc_w._base)
        dh = torch.empty((M, D * H), **f32)
        ops.gemm(False, False, M, D * H, C, dl_tm, C, fc_w.detach(), D * H, dh, D * H)
        ggru: List[Optional[torch.Tensor]] = [None] * len(gru_w)
        dgi = torch.empty((M, D * 3 * H), **f32)
        dghn = [torch.empty((M, H), **f32) for _ in range(D)]
        want_front = want_x or need[0] or need[1]
        for l in range(L - 1, -1, -1):
            inp, hseq, saves = ctx.layers[l]
            in_l = inp.shape[1]
            if cfg["p_drop"] > 0 and l < L - 1:
                dh = ops.dropout(dh, cfg["p_drop"], cfg["seed"] + l)
            for d in range(D):
                w_hh = gru_w[(l * D + d) * 4 + 1].detach()
                ops.gru_bwd_f32(dh, D * H, d * H, hseq, D * H, d * H, saves[d], w_hh, Tp, B, H, d == 1,
                                dgi, D * 3 * H, d * 3 * H, dghn[d])
            dinp = torch.empty((M, in_l), **f32) if l > 0 or want_front else None
            wgrad = any(need_gru[l * D * 4:(l + 1) * D * 4])
            # one flat bucket per layer: its all-reduce starts while the layers below are still in BPTT
            views = _flat_views([(3 * H, in_l), (3 * H, H), (3 * H,), (3 * H,)] * D, dev, None, zero=(Tp == 1)) if wgrad else None
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
            dh = dinp
        ys, z, day_idx, taps = ctx.front
        d_day_w = d_day_b = dx = None
        if dh is not None:
            if need[0] or need[1]:
                d_day_w, d_day_b = ops.frontend_bwd(dh, ys, z, day_idx, cfg["n_days"], K, S)
                if gs is not None:
                    gs.bucket_ready(d_day_w._base)
            if want_x:
                dx = ops.frontend_bwd_input(dh, z, day_idx, day_w.detach().contiguous(), taps, K, S)
        ctx.layers = ctx.hid = ctx.front = None
        grads = (d_day_w, d_day_b, d_fc_w, d_fc_b, *ggru)
        if gs is not None:
            return (None, dx, None, None) + _assign_grads(ctx.params, grads)
        return (None, dx, None, None) + grads
