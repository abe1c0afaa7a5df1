"""bf16 operand copies of fp32 master weights for the tensor-core kernels (precision="bf16"), and the architecture limits of
those kernels.  GRUDecoder's bf16 chain (model._DecoderFunction), the Conformer, FusedAdam / FusedAdamW and streaming use them.
"""
from __future__ import annotations

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

