"""fp64 restatement of oracle/conformer_port.forward with the stochastic regularisers applied as CHOSEN masks.

TEST INFRASTRUCTURE ONLY.  oracle/conformer_port.py is the deterministic part of the reference's Conformer (dropout, DropPath and
SpecAugment are the identity there).  This restatement multiplies given masks in at the sites where the reference's modules apply
them, so a training step's own draws (rebuilt from its seeds with the same kernels) can be fed to an fp64 model.  The reference
source is not in this tree: the placement of each site is taken from the module containers of
neural_speech_decoder_b200/conformer.py and the reference line numbers they cite:
    front end      Linear -> LayerNorm -> Dropout                                   transformer_ctc.py:124-127 (_NeuralFrontend.dropout)
    SpecAugment    two frequency bands over D, two time bands over T', zeroed BEFORE the positional encoding is added
                                                                                    transformer_ctc.py:266-308, 466-471
    feed-forward   LN -> Linear -> SiLU -> Dropout -> Linear -> Dropout             transformer_ctc.py:194-263 (ff1 / ff2: nn.Sequential
                   z + 0.5 * DropPath(ff(z))                                        indices 3 and 5), :245, :257
    attention      softmax weights -> Dropout (nn.MultiheadAttention(dropout=p)) -> out_proj -> dropout_attn
                   z + DropPath(...)                                                transformer_ctc.py:216, 248-251
    conv module    x + Dropout(pw_conv2(...)), no DropPath                          transformer_ctc.py:170-191
    head           Linear -> LayerNorm -> GELU -> Dropout(0.3) -> Linear            transformer_ctc.py:408-415
    DropPath       per utterance: kept with probability 1-p and scaled by 1/(1-p)   transformer_ctc.py:9-23
A mask here is the multiplier itself (0 or 1/(1-p)), as the kernels apply it.  With every mask None (or all ones) and no bands this
is conformer_port.forward (tests/test_gpu_conformer_training.py::test_masked_port_with_unit_masks_is_the_port).

``masks`` keys (all optional; shapes batch-major like the activations):
    "fe" [B,T',Dfe], "bands" 8 ints (f0,f1, f0,f1, t0,t1, t0,t1), "head" [B,T',D], and "blocks": one dict per layer with
    "ff1_act" / "ff2_act" [B,T',FF], "ff1_drop" / "attn_drop" / "conv_drop" / "ff2_drop" [B,T',D], "ff1_path" / "attn_path" /
    "ff2_path" [B], "attn_p" [B,H,T',T'].
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle.conformer_port import _lin, _ln, out_lengths


def _mul(t, k):
    return t if k is None else t * k


def _path(t, f):
    return t if f is None else t * f.reshape(-1, *([1] * (t.dim() - 1)))


def band_keep(bands, T, D, dtype=torch.float64):
    """[T, D] multiplier of SpecAugment: 0 inside any frequency band (over D) or time band (over T), 1 elsewhere."""
    t = torch.arange(T)[:, None]
    f = torch.arange(D)[None, :]
    hit = ((f >= bands[0]) & (f < bands[1])) | ((f >= bands[2]) & (f < bands[3])) | ((t >= bands[4]) & (t < bands[5])) | ((t >= bands[6]) & (t < bands[7]))
    return (~hit).to(dtype)


def _ff(x, sd, name, act_mask, drop_mask):
    h = _ln(x, sd, name + ".0")
    h = _mul(F.silu(_lin(h, sd, name + ".1")), act_mask)
    return _mul(_lin(h, sd, name + ".4"), drop_mask)


def _mhsa(x, sd, name, n_heads, key_pad, p_mask):
    """conformer_port._mhsa with the attention-weight dropout multiplied into the softmax output."""
    B, T, D = x.shape
    dh = D // n_heads
    qkv = F.linear(x, sd[name + ".in_proj_weight"], sd[name + ".in_proj_bias"])
    q, k, v = qkv.split(D, dim=-1)
    sh = lambda t: t.reshape(B, T, n_heads, dh).transpose(1, 2)
    q, k, v = sh(q) * (1.0 / math.sqrt(dh)), sh(k), sh(v)
    s = q @ k.transpose(-1, -2)
    if key_pad is not None:
        s = s.masked_fill(key_pad[:, None, None, :], float("-inf"))
    p = _mul(torch.softmax(s, dim=-1), p_mask)
    o = (p @ v).transpose(1, 2).reshape(B, T, D)
    return F.linear(o, sd[name + ".out_proj.weight"], sd[name + ".out_proj.bias"])


def _conv(x, sd, name, ksize, drop_mask):
    """conformer_port._conv_module with the module's dropout on the branch: x + dropout(pw_conv2(...))."""
    h = _ln(x, sd, name + ".ln")
    h = F.glu(_lin(h, sd, name + ".pw_conv1"), dim=-1)
    h = F.conv1d(h.transpose(1, 2), sd[name + ".dw_conv.weight"], sd[name + ".dw_conv.bias"], padding=ksize // 2,
                 groups=h.shape[-1]).transpose(1, 2)
    h = F.silu(_ln(h, sd, name + ".ln_conv"))
    return x + _mul(_lin(h, sd, name + ".pw_conv2"), drop_mask)


def forward(sd, x, day_ids, input_lengths, *, n_layers, n_heads, temporal_kernel, temporal_stride, conv_kernel, masks=None):
    """Train-mode conformer_port.forward (InterCTC head on) with the masks above -> (log_probs [T',B,C], out_lengths, inter)."""
    m = masks or {}
    blocks = m.get("blocks") or [{}] * n_layers
    C = x.shape[-1]
    x = torch.einsum("btd,bdk->btk", x, sd["day_linear.day_weights"][day_ids]) + sd["day_linear.day_bias"][day_ids]
    if "frontend.gaussian_kernel" in sd:
        g = sd["frontend.gaussian_kernel"]
        x = F.conv1d(x.transpose(1, 2), g.repeat(C, 1, 1), padding=g.shape[-1] // 2, groups=C).transpose(1, 2)
    if temporal_kernel > 0:
        x = F.conv1d(x.transpose(1, 2), sd["frontend.temporal_conv.weight"], None, stride=temporal_stride, groups=C).transpose(1, 2)
    z = _mul(_ln(_lin(x, sd, "frontend.proj"), sd, "frontend.ln"), m.get("fe"))
    z = _lin(F.relu(_lin(z, sd, "encoder.net.0")), sd, "encoder.net.2")
    Tn, D = z.shape[1], z.shape[2]
    if m.get("bands") is not None:
        z = z * band_keep(m["bands"], Tn, D, z.dtype)
    z = z + sd["pos_enc.pe"][:, :Tn]
    key_pad = None
    if input_lengths is not None:
        olen = out_lengths(input_lengths, temporal_kernel, temporal_stride, Tn)
        key_pad = torch.arange(Tn)[None, :] >= olen[:, None]
    else:
        olen = torch.full((x.shape[0],), Tn, dtype=torch.int32)
    inter = None
    for i in range(n_layers):
        p, k = f"conformer_layers.{i}", blocks[i]
        z = z + 0.5 * _path(_ff(z, sd, p + ".ff1", k.get("ff1_act"), k.get("ff1_drop")), k.get("ff1_path"))
        a = _mul(_mhsa(_ln(z, sd, p + ".ln_attn"), sd, p + ".attn", n_heads, key_pad, k.get("attn_p")), k.get("attn_drop"))
        z = z + _path(a, k.get("attn_path"))
        z = _conv(z, sd, p + ".conv_module", conv_kernel, k.get("conv_drop"))
        z = z + 0.5 * _path(_ff(z, sd, p + ".ff2", k.get("ff2_act"), k.get("ff2_drop")), k.get("ff2_path"))
        z = _ln(z, sd, p + ".ln_final")
        if n_layers >= 6 and i == n_layers // 2 - 1:
            inter = _lin(z, sd, "inter_output").log_softmax(-1).transpose(0, 1)
    h = _mul(F.gelu(_ln(_lin(z, sd, "output.0"), sd, "output.1")), m.get("head"))
    logits = _lin(h, sd, "output.4")
    return logits.log_softmax(-1).transpose(0, 1), olen, inter
