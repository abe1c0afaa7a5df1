"""bf16 tensor-core execution of GRUDecoder.forward / backward (precision="bf16").

Same chain as model._DecoderFunction, with the dense contractions on tcgen05:
  K1 (bf16 patches) -> per layer [K2 tcgen05 GEMM for both directions' W_ih at once -> K3 tcgen05 persistent
  recurrence for both directions at once -> dropout] -> output layer (tcgen05 GEMM, N = 41 classes).
Parameters stay fp32 (master weights); bf16 operand copies are made per step.  Accumulation, hidden state, gate
math, saved activations and all parameter gradients are fp32.  Reference: model.py:83-123, autograd of it.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import ops
from ._lib import NsdError

MAX_HIDDEN = 1024       # largest hidden size of the tensor-core recurrence (csrc/gru_ts.cu, MAX_H)


def check_architecture(neural_dim: int, kernel_len: int, hidden_dim: int) -> None:
    """Refuse an architecture the bf16 kernels cannot run before anything is launched (the recurrence and the GEMMs would
    otherwise reject it part-way through the step, after the front end has run)."""
    if hidden_dim % 64 != 0 or hidden_dim > MAX_HIDDEN:
        raise NsdError(f"precision 'bf16': hidden_dim={hidden_dim} must be a multiple of 64 and at most {MAX_HIDDEN} (tensor-core "
                       "recurrence); precision 'fp32' runs any hidden size")
    if (neural_dim * kernel_len) % 8 != 0:
        raise NsdError(f"precision 'bf16': neural_dim*kernelLen={neural_dim * kernel_len} must be a multiple of 8 (16-byte rows of "
                       "the bf16 input GEMM); precision 'fp32' runs any input width")


class Bf16Shadows:
    """bf16 operand copies of the fp32 master weights, kept across steps.  A copy is valid while the parameter's
    (data_ptr, autograd version) is the one it was made from; anything that modifies a parameter in place THROUGH
    AUTOGRAD-VISIBLE OPS (optimizers, load_state_dict, ``p.copy_``/``dist.broadcast(p)`` under no_grad) bumps the version and
    the copy is re-made by the next forward.  FusedAdam, when attached, rewrites the copies inside its update kernel and
    marks them fresh, so a training step does no weight casts at all.
    Writes through ``p.data`` (``p.data.copy_()``, ``p.data[...] =``, NCCL broadcast of ``p.data``, raw pointers) do NOT bump
    the version: call ``invalidate()`` (or ``GRUDecoder.invalidate_weight_copies()``) after them."""

    def __init__(self):
        self.bufs = {}        # key -> stacked bf16 buffer [D*R, C]
        self.tags = {}        # (key, d) -> (data_ptr, version) of the fp32 source
        self.where = {}       # data_ptr of the fp32 source -> (key, d)

    def invalidate(self) -> None:
        """Forget every copy's validity (the buffers are kept and re-filled by the next forward)."""
        self.tags.clear()
        self.where.clear()

    def stacked(self, key, ws):
        """Up-to-date bf16 copy of the D fp32 matrices ``ws`` ([R, C] each) stacked by rows."""
        D = len(ws)
        R, Cn = ws[0].shape
        buf = self.bufs.get(key)
        if buf is None or tuple(buf.shape) != (D * R, Cn) or buf.device != ws[0].device:
            buf = torch.empty((D * R, Cn), device=ws[0].device, dtype=torch.bfloat16)
            self.bufs[key] = buf
            for d in range(D):
                self.tags.pop((key, d), None)
        for d, w in enumerate(ws):
            tag = (w.data_ptr(), w._version)
            old = self.tags.get((key, d))
            if old != tag:
                ops.cast_transpose_into(w.detach(), buf[d * R:(d + 1) * R], None)
                if old is not None and old[0] != tag[0] and self.where.get(old[0]) == (key, d):
                    del self.where[old[0]]               # the parameter was reallocated: its old address may be reused
                self.tags[(key, d)] = tag
                self.where[w.data_ptr()] = (key, d)
        return buf

    def slice_for(self, p):
        loc = self.where.get(p.data_ptr())
        if loc is None:
            return None
        key, d = loc
        buf = self.bufs[key]
        if p.dim() != 2 or self.tags.get(loc, (None,))[0] != p.data_ptr():
            return None
        R = p.shape[0]
        if buf.shape[1] != p.shape[1] or (d + 1) * R > buf.shape[0]:
            return None
        return buf[d * R:(d + 1) * R]

    def mark_fresh(self, p) -> None:
        loc = self.where.get(p.data_ptr())
        if loc is not None:
            self.tags[loc] = (p.data_ptr(), p._version)


def decoder_forward_tc(ctx, cfg, x, day_idx, taps, day_w, day_b, fc_w, fc_b, *gru_w):
    K, S, H, L, D = cfg["K"], cfg["S"], cfg["H"], cfg["L"], cfg["D"]
    dev = x.device
    B, T, N = x.shape
    Tp = ops.n_frames(T, K, S)
    M = Tp * B
    day_idx = day_idx.to(device=dev, dtype=torch.int64).contiguous()
    need_grad = cfg.get("need_grad", True)
    patches, ys, z = ops.frontend_fwd(x, day_idx, day_w.detach().contiguous(), day_b.detach().contiguous(), taps,
                                      K, S, torch.bfloat16, cfg["err_flag"], cfg.get("noise"))
    inp = patches                                            # bf16 [M, in_l]
    sh = cfg.get("shadows") or Bf16Shadows()                 # the module's cache of bf16 weight copies (a throw-away one otherwise)
    layers = []
    hseq = None
    # both directions run in one GEMM / one recurrence launch: their bias vectors side by side, packed in ONE launch
    if D > 1:
        bias_all = torch.empty((L, 2, D * 3 * H), device=dev, dtype=torch.float32)
        ops.multi_copy([gru_w[(l * D + d) * 4 + 2 + k].detach() for l in range(L) for k in range(2) for d in range(D)],
                       [bias_all[l, k, d * 3 * H:(d + 1) * 3 * H] for l in range(L) for k in range(2) for d in range(D)])
    # gru_w holds the Parameters themselves: their version counters tell whether the kept bf16 copies are current
    w_hh_all = [sh.stacked(("hh", l), [gru_w[(l * D + d) * 4 + 1] for d in range(D)]) for l in range(L)]      # [D*3H, H] each
    w_hhT_all = None
    if need_grad:                                            # BPTT operands [D*H, 3H] of every layer, all transposed in one launch
        w_hhT_all = torch.empty((L, D * H, 3 * H), device=dev, dtype=torch.bfloat16)
        ops.transpose_bf16_multi([w_hh_all[l][d * 3 * H:(d + 1) * 3 * H] for l in range(L) for d in range(D)],
                                 [w_hhT_all[l, d * H:(d + 1) * H] for l in range(L) for d in range(D)])
    for l in range(L):
        in_l = inp.shape[1]
        ws = [[t.detach() for t in gru_w[(l * D + d) * 4:(l * D + d) * 4 + 4]] for d in range(D)]
        w_ih_bf = sh.stacked(("ih", l), [gru_w[(l * D + d) * 4] for d in range(D)])          # [D*3H, in_l]
        w_hh_bf = w_hh_all[l]
        w_hhT_bf = w_hhT_all[l] if need_grad else None
        b_ih, b_hh = (bias_all[l, 0], bias_all[l, 1]) if D > 1 else (ws[0][2], ws[0][3])
        gi = torch.empty((M, D * 3 * H), device=dev, dtype=torch.float32)
        ops.gemm(False, True, M, D * 3 * H, in_l, inp, in_l, w_ih_bf, in_l, gi, D * 3 * H, bias=b_ih.contiguous())
        if cfg["p_drop"] > 0 and l < L - 1:      # inter-layer dropout fused into the recurrence's epilogue
            hseq, hseq_bf, saves, nxt = ops.gru_fwd_bf16(gi, w_hh_bf, b_hh.contiguous(), Tp, B, H, D, False, need_grad,
                                                         cfg["p_drop"], cfg["seed"] + l)
        else:
            hseq, hseq_bf, saves = ops.gru_fwd_bf16(gi, w_hh_bf, b_hh.contiguous(), Tp, B, H, D, False, need_grad)
            nxt = hseq_bf
        del gi
        layers.append((inp, hseq, hseq_bf, saves, w_ih_bf, w_hhT_bf))
        inp = nxt
    C = fc_w.shape[0]
    logits_tm = torch.empty((M, C), device=dev, dtype=torch.float32)
    fc_w_bf = sh.stacked(("fc", 0), [fc_w])
    ops.gemm(False, True, M, C, D * H, hseq_bf, D * H, fc_w_bf, D * H, logits_tm, C, bias=fc_b.detach().contiguous())
    logits = ops.swap01(logits_tm.view(Tp, B, C))
    if need_grad:
        ctx.cfg = cfg
        ctx.dims = (B, T, N, Tp)
        ctx.layers = layers
        ctx.hid = hseq_bf
        ctx.front = (ys, z, day_idx, taps)
        ctx.weights = (day_w, fc_w, gru_w)
        ctx.fc_w_bf = fc_w_bf
        ctx.params = (day_w, day_b, fc_w, fc_b) + tuple(gru_w)
    return logits


def decoder_backward_tc(ctx, dlogits):
    from .model import _assign_grads, _flat_views, grad_plan
    cfg = ctx.cfg
    K, S, H, L, D = cfg["K"], cfg["S"], cfg["H"], cfg["L"], cfg["D"]
    B, T, N, Tp = ctx.dims
    M = Tp * B
    day_w, fc_w, gru_w = ctx.weights
    dev = dlogits.device
    C = fc_w.shape[0]
    f32 = dict(device=dev, dtype=torch.float32)
    gs = cfg.get("grad_sync")
    schedule = cfg.get("step_hook")    # trainer._UpdateSchedule: updates finished buckets from inside the backward
    want_x, need = grad_plan(ctx)
    need_gru = need[4:]
    dl_tm = ops.swap01(dlogits.contiguous().float()).view(M, C)
    hid = ctx.hid
    # output layer on tensor cores.  Reductions over the T'*B rows take their operands in the natural (MN-major) layout.
    Cp = (C + 7) // 8 * 8
    dl_bf = torch.empty((M, Cp), device=dev, dtype=torch.bfloat16)
    ops.cast_transpose_into(dl_tm, dl_bf[:, :C], None)
    d_fc_w = d_fc_b = None
    if need[2] or need[3]:
        d_fc_w, d_fc_b = _flat_views([(C, D * H), (C,)], dev, gs)
        if need[2]:
            ops.gemm(True, False, C, D * H, M, dl_bf, Cp, hid, D * H, d_fc_w, D * H)        # d_fc_w = dl^T hid
        if need[3]:
            ops.colsum(dl_tm, M, C, C, d_fc_b)
        handle = gs.bucket_ready(d_fc_w._base) if gs is not None else None
        if schedule is not None:
            schedule.released([(ctx.params[2], d_fc_w), (ctx.params[3], d_fc_b)], handle)
    dh = torch.empty((M, D * H), **f32)
    ops.gemm(False, False, M, D * H, C, dl_bf, Cp, ctx.fc_w_bf, D * H, dh, D * H)       # dh = dl fc_w
    ggru: List[Optional[torch.Tensor]] = [None] * len(gru_w)
    Mh = (Tp - 1) * B
    for l in range(L - 1, -1, -1):
        inp, hseq, hseq_bf, saves, w_ih_bf, w_hhT_bf = ctx.layers[l]
        in_l = inp.shape[1]
        # what this layer's parameters need, each kind over both directions (one GEMM / one BPTT reduction covers both)
        n_wih, n_whh, n_b = (any(need_gru[(l * D + d) * 4 + k] for d in range(D) for k in ks) for ks in ((0,), (1,), (2, 3)))
        wgrad = n_wih or n_whh or n_b
        # one flat bucket per layer, laid out so that each GEMM writes its whole (both-direction) block at once
        v_wih = v_whh = v_bih = v_bhh = None
        if wgrad:
            v_wih, v_whh, v_bih, v_bhh = _flat_views([(D * 3 * H, in_l), (D * 3 * H, H), (D * 3 * H,), (D * 3 * H,)], dev, None,
                                                     zero=(Tp == 1))
        drop = cfg["p_drop"] if (cfg["p_drop"] > 0 and l < L - 1) else 0.0
        # BPTT with the output-dropout mask applied on load and the bias gradients (column sums) accumulated in-kernel
        db = (v_bih, v_bhh) if n_b else (None, None)
        bptt = lambda: ops.gru_bwd_bf16(dh, hseq, saves, w_hhT_bf, Tp, B, H, D, False, drop, cfg["seed"] + l, *db)
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
            from ._lib import call
            call("nsd_set_gemm_sm_reserve", gs.tail_sms)
        dinp = None
        if l > 0 or want_x or need[0] or need[1]:
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
        ctx.layers[l] = None
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
    if schedule is not None:
        grads = schedule.not_updated(ctx.params, grads)
    if gs is not None:
        return (None, dx, None, None) + _assign_grads(ctx.params, grads)
    return (None, dx, None, None) + grads
