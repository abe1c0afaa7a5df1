"""fp64 torch restatement of GRUDecoder.forward(X, dayIdx, X_len): packed-sequence semantics.

Built from ``oracle/torch_port.PortGRUDecoder``'s own operators (which are the reference's): X is zeroed past X_len, the front end
runs as in the port (smoother, day affine, softsign, unfold), and the GRU is called through
``pack_padded_sequence(lengths=n_b, enforce_sorted=False)`` / ``pad_packed_sequence(total_length=T')`` with
n_b = (X_len - kernelLen) // strideLen + 1, so every utterance runs alone on its own frames and the outputs past them are 0.
Test infrastructure only.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence


def frame_counts(X_len: torch.Tensor, kernel_len: int, stride_len: int, T: int) -> torch.Tensor:
    Tp = (T - kernel_len) // stride_len + 1
    return ((X_len.long() - kernel_len) // stride_len + 1).clamp(0, Tp)


def packed_forward(port, x: torch.Tensor, dayIdx: torch.Tensor, X_len: torch.Tensor) -> torch.Tensor:
    """logits [B, T', C] of ``port`` (a PortGRUDecoder, any dtype) on ``x`` [B, T, N] with per-utterance lengths ``X_len``."""
    B, T, N = x.shape
    X_len = X_len.long().cpu()
    keep = torch.arange(T).view(1, T, 1) < X_len.view(B, 1, 1)
    x = torch.where(keep, x, torch.zeros((), dtype=x.dtype))        # a select: padding may hold anything, NaN included
    x = x.permute(0, 2, 1)
    x = F.conv1d(x, port.smooth_w, groups=port.neural_dim, padding="same")
    x = x.permute(0, 2, 1)
    w = torch.index_select(port.dayWeights, 0, dayIdx)
    x = torch.einsum("btd,bdk->btk", x, w) + torch.index_select(port.dayBias, 0, dayIdx)
    x = F.softsign(x)
    x = F.unfold(x.permute(0, 2, 1).unsqueeze(3), (port.kernelLen, 1), stride=port.strideLen).permute(0, 2, 1)
    Tp = x.shape[1]
    n = frame_counts(X_len, port.kernelLen, port.strideLen, T)
    D = 2 if port.bidirectional else 1
    h0 = torch.zeros(port.layer_dim * D, B, port.hidden_dim, dtype=x.dtype, device=x.device)
    packed = pack_padded_sequence(x, n, batch_first=True, enforce_sorted=False)
    hid, _ = port.gru(packed, h0)
    hid, _ = pad_packed_sequence(hid, batch_first=True, total_length=Tp)
    return port.fc(hid)
