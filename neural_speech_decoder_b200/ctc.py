"""CTC loss, greedy decode, prefix beam search, forced alignment, phoneme error rate, and lexicon-constrained word beam search
with a word n-gram LM and word error rate, on the sm_100a kernels (K4 / K5 / K5b / K5c / K5d).

``CTCLoss`` mirrors ``torch.nn.CTCLoss`` as the reference trainer uses it
(neural_decoder_trainer.py:139-141, 213-218): call signature
``(log_probs[T',B,C], targets i32[B,S], input_lengths[B], target_lengths[B])``,
``blank``, ``reduction`` in {"mean","sum","none"} and ``zero_infinity``.  The
log-probs may be any strided view (the trainer passes ``.permute(1,0,2)`` of a
``[B,T',C]`` tensor); lengths and targets stay on the device, there is no host
synchronisation.

``ctc_loss_from_logits`` is the fused form used by ``train_step``: log-softmax,
alpha/beta, loss and d loss / d logits in one launch (trainer:210-218, 242, 252).
"""
from __future__ import annotations

import math
import re
from collections import namedtuple
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch import nn

from . import _lib, ops
from ._lib import NsdError, call, ptr, require_cuda, stream


def _as_i32(t: torch.Tensor, dev) -> torch.Tensor:
    return t.to(device=dev, dtype=torch.int32).contiguous()


def _prep_targets(targets: torch.Tensor, dev) -> torch.Tensor:
    if targets.dim() != 2:
        raise NsdError("CTCLoss (B200): targets must be 2-D padded [B,S] as the trainer's collate produces them")
    t = _as_i32(targets, dev)
    if t.shape[1] == 0:
        t = torch.zeros((t.shape[0], 1), device=dev, dtype=torch.int32)
    return t


class _CtcFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, act, targets, in_lens, tgt_lens, blank, reduction, zero_infinity, is_logits, tbc):
        """act: log-probs [T,B,C] (any strides) when tbc else logits [B,T,C]."""
        require_cuda(act, "log_probs")
        if not zero_infinity:
            raise NsdError("CTCLoss (B200): only zero_infinity=True (the reference's setting) is implemented")
        if act.dtype != torch.float32:
            act = act.float()
        if torch.empty_like(act).stride() != act.stride():      # the gradient is written with act's own strides
            act = act.contiguous()
        if tbc:
            T, B, C = act.shape
            st, sb, sc = act.stride()
        else:
            B, T, C = act.shape
            sb, st, sc = act.stride()
        want_grad = bool(ctx.needs_input_grad[0])
        mean = reduction == "mean"
        loss, nll, grad = ops.ctc_loss_raw(act, st, sb, sc, is_logits, targets, in_lens, tgt_lens, T, B, C, blank,
                                           mean, want_grad)
        ctx.reduction, ctx.tbc = reduction, tbc
        ctx.save_for_backward(grad)
        if reduction == "none":
            return nll
        return loss

    @staticmethod
    def backward(ctx, gout):
        (grad,) = ctx.saved_tensors
        if grad is None:
            return (None,) * 9
        if ctx.reduction == "none":
            # grad holds d nll[b] / d act; scale each utterance by its upstream gradient
            g = grad * (gout.view(1, -1, 1) if ctx.tbc else gout.view(-1, 1, 1))
        else:
            g = grad * gout
        return (g,) + (None,) * 8


def _ctc_apply(act, targets, in_lens, tgt_lens, blank, reduction, zero_infinity, is_logits, tbc):
    require_cuda(act, "log_probs")
    dev = act.device
    targets = _prep_targets(targets, dev)
    in_lens = _as_i32(in_lens, dev)
    tgt_lens = _as_i32(tgt_lens, dev)
    if reduction not in ("mean", "sum", "none"):
        raise ValueError(reduction)
    with torch.cuda.device(dev):            # raw-pointer launches must target the tensors' device, not the caller's current one
        return _CtcFunction.apply(act, targets, in_lens, tgt_lens, blank, reduction, zero_infinity, is_logits, tbc)


class CTCLoss(nn.Module):
    """Drop-in for ``torch.nn.CTCLoss`` on CUDA tensors (trainer:139-141)."""

    def __init__(self, blank: int = 0, reduction: str = "mean", zero_infinity: bool = False):
        super().__init__()
        self.blank, self.reduction, self.zero_infinity = blank, reduction, zero_infinity

    def forward(self, log_probs, targets, input_lengths, target_lengths):
        return _ctc_apply(log_probs, targets, input_lengths, target_lengths, self.blank, self.reduction,
                          self.zero_infinity, False, True)


def ctc_loss_from_logits(logits, targets, input_lengths, target_lengths, blank=0, reduction="mean"):
    """log_softmax(2) + CTCLoss(blank, reduction, zero_infinity=True) on logits [B,T',C]; one launch, and the
    backward is the already-computed d loss / d logits (trainer:210, 213-218, 252)."""
    return _ctc_apply(logits, targets, input_lengths, target_lengths, blank, reduction, True, True, False)


def log_softmax_tbc(logits: torch.Tensor) -> torch.Tensor:
    """``logits.log_softmax(2).permute(1, 0, 2)`` (trainer:210, 301): logits [B,T',C] -> log-probs as a
    [T',B,C] view of a contiguous [B,T',C] buffer, exactly the layout the reference hands to CTCLoss."""
    require_cuda(logits, "logits")
    with torch.cuda.device(logits.device):
        return ops.log_softmax(logits.float().contiguous()).permute(1, 0, 2)


def out_lens(X_len: torch.Tensor, kernel_len: int, stride_len: int) -> torch.Tensor:
    """((X_len - kernelLen) / strideLen).to(int32)  -- trainer:209, 300 (true division, truncation)."""
    return ((X_len - kernel_len) / stride_len).to(torch.int32)


def greedy_decode(log_probs: torch.Tensor, lens: torch.Tensor, blank: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """argmax -> unique_consecutive -> drop blank for every utterance of ``log_probs`` [T',B,C] (any strides)
    in ONE launch (trainer:313-320 does it per utterance with a device->host sync each).
    Returns (decoded int64 [B,T'], decoded_len int32 [B]) on the device."""
    require_cuda(log_probs, "log_probs")
    if log_probs.dtype != torch.float32:
        log_probs = log_probs.float()
    T, B, C = log_probs.shape
    st, sb, sc = log_probs.stride()
    with torch.cuda.device(log_probs.device):
        return ops.greedy_decode_raw(log_probs, st, sb, sc, _as_i32(lens, log_probs.device), T, B, C, blank)


def decoded_to_lists(dec: torch.Tensor, dec_len: torch.Tensor) -> List[List[int]]:
    d, l = dec.cpu().numpy(), dec_len.cpu().numpy()
    return [d[i, :l[i]].tolist() for i in range(d.shape[0])]


def edit_distances(dec, dec_len, targets, target_lengths) -> torch.Tensor:
    """Levenshtein distance per utterance on the device (SequenceMatcher.distance(), trainer:322-330)."""
    dev = dec.device
    with torch.cuda.device(dev):
        return ops.edit_distance_raw(dec.contiguous(), _as_i32(dec_len, dev), _prep_targets(targets, dev),
                                     _as_i32(target_lengths, dev))


class CtcBeamSearch:
    """CTC prefix beam search over [T,B,C] log-probs or logits with an optional phoneme-bigram prior (K5b,
    ``nsd_ctc_beam_*``; no counterpart in the reference, which decodes greedily).

    The beam of every utterance lives on the device and resumes where the last ``advance`` stopped: one call over all
    frames and any chunking of the same frames give the same bits.  ``lm`` (``[C, C]`` log-probs, row = previous emitted
    token, row ``blank`` = start of the utterance) adds ``lm_weight * lm[prev, c] + insertion_bonus`` to every emitted
    token; hypotheses are ranked by ``acoustic + prior``.  At most ``max_frames`` frames per utterance fit the state."""

    def __init__(self, batch: int, num_classes: int, beam_width: int = 16, max_frames: int = 4096, blank: int = 0,
                 lm: Optional[torch.Tensor] = None, lm_weight: float = 0.0, insertion_bonus: float = 0.0, device=None):
        self.B, self.C, self.W, self.max_frames, self.blank = int(batch), int(num_classes), int(beam_width), int(max_frames), int(blank)
        if not 1 <= self.W <= 128:
            raise NsdError(f"ctc beam search: beam_width={self.W} outside [1, 128]")
        if not 1 <= self.C <= 128:
            raise NsdError(f"ctc beam search: num_classes={self.C} outside [1, 128]")
        if not 0 <= self.blank < self.C:
            raise NsdError(f"ctc beam search: blank={self.blank} outside [0, {self.C})")
        if self.B < 1 or self.max_frames < 1:
            raise NsdError(f"ctc beam search: batch={self.B} and max_frames={self.max_frames} must be positive")
        self.dev = torch.device("cuda") if device is None else torch.device(device)
        if self.dev.type != "cuda":
            raise NsdError(f"ctc beam search: the beam state lives on a CUDA device (got {self.dev}); this package has no CPU path")
        if self.dev.index is None:         # "cuda" means the current device; inputs carry an index, so compare with one
            self.dev = torch.device("cuda", torch.cuda.current_device())
        self.lm_weight, self.insertion_bonus = float(lm_weight), float(insertion_bonus)
        self.lm = None
        if lm is not None:
            if tuple(lm.shape) != (self.C, self.C):
                raise NsdError(f"ctc beam search: lm must be [{self.C}, {self.C}], got {tuple(lm.shape)}")
            self.lm = lm.detach().to(device=self.dev, dtype=torch.float32).contiguous()
        self._lm_arg = self.lm if self.lm_weight != 0.0 else None     # weight 0: the table is not read (exactly lm=None)
        self.state_bytes = self._state_bytes()
        self.state = torch.empty(self.state_bytes, device=self.dev, dtype=torch.uint8)
        self.err_flag = torch.zeros(1, device=self.dev, dtype=torch.int32)
        self.reset()

    def _state_bytes(self) -> int:
        return _lib.lib().nsd_ctc_beam_state_bytes(self.B, self.W, self.max_frames)

    def reset(self) -> None:
        """Back to the empty hypothesis, in place (a captured graph keeps valid addresses)."""
        with torch.cuda.device(self.dev):
            call("nsd_ctc_beam_init", ptr(self.state), self.state_bytes, self.B, self.W, self.max_frames, stream())
            self.err_flag.zero_()
        self.frames = 0            # frames advanced so far, counted on the host (an upper bound per utterance)

    def reset_utterances(self, mask: torch.Tensor) -> None:
        """Back to the empty hypothesis for the utterances with ``mask[b] != 0`` (i32 [B] on the beam's device), in place; the
        others keep every byte.  The host frame count of ``reserve`` is left as it is: a caller that recycles utterances
        counts frames per utterance itself."""
        if mask.device != self.dev or mask.dtype != torch.int32 or tuple(mask.shape) != (self.B,) or not mask.is_contiguous():
            raise NsdError(f"ctc beam search: mask must be a contiguous int32 [{self.B}] tensor on {self.dev}")
        with torch.cuda.device(self.dev):
            call("nsd_ctc_beam_reset", ptr(self.state), self.state_bytes, self.B, self.W, self.max_frames, ptr(mask), stream())

    def reserve(self, T: int) -> None:
        """Count ``T`` more frames; raise before anything is launched if they would pass ``max_frames``."""
        if self.frames + T > self.max_frames:
            raise NsdError(f"ctc beam search: {self.frames} + {T} frames exceed max_frames={self.max_frames}")
        self.frames += T

    def _check(self, act: torch.Tensor) -> torch.Tensor:
        require_cuda(act, "log_probs")
        if act.dim() != 3 or act.shape[1] != self.B or act.shape[2] != self.C:
            raise NsdError(f"ctc beam search: expected [T, {self.B}, {self.C}], got {tuple(act.shape)}")
        if act.device != self.dev:
            raise NsdError(f"ctc beam search: input on {act.device}, beam state on {self.dev}")
        return act if act.dtype == torch.float32 else act.float()

    def enqueue(self, act: torch.Tensor, lens: Optional[torch.Tensor] = None, is_logits: bool = False) -> None:
        """Launch the advance without counting frames (the caller has reserved them): the unit a CUDA graph captures."""
        T = act.shape[0]
        st, sb, sc = act.stride()
        call("nsd_ctc_beam_advance", ptr(act), st, sb, sc, int(bool(is_logits)), ptr(lens), T, self.B, self.C, self.blank,
             ptr(self._lm_arg), self.lm_weight, self.insertion_bonus, self.W, self.max_frames, ptr(self.state), self.state_bytes,
             ptr(self.err_flag), stream())

    def advance(self, act_tbc: torch.Tensor, lens: Optional[torch.Tensor] = None, is_logits: bool = False) -> None:
        """Consume frames ``act_tbc`` [T,B,C] (any strides); ``lens[b]``: how many of them belong to utterance b (None: all)."""
        act = self._check(act_tbc)
        self.reserve(act.shape[0])
        with torch.cuda.device(self.dev):
            self.enqueue(act, None if lens is None else _as_i32(lens, self.dev), is_logits)

    def nbest(self, k: int = 1):
        """-> (hyps i64 [B,k,max_frames] (-1 past the length), hyp_len i32 [B,k], score f32 [B,k] = acoustic + prior,
        acoustic f32 [B,k] = CTC prefix log-probability), best first, on the device.  Slots past the beam's size: length 0,
        score -inf."""
        k = int(k)
        if not 1 <= k <= self.W:
            raise NsdError(f"ctc beam search: nbest={k} outside [1, beam_width={self.W}]")
        hyps = torch.empty((self.B, k, self.max_frames), device=self.dev, dtype=torch.int64)
        hyp_len = torch.empty((self.B, k), device=self.dev, dtype=torch.int32)
        score = torch.empty((self.B, k), device=self.dev, dtype=torch.float32)
        acoustic = torch.empty((self.B, k), device=self.dev, dtype=torch.float32)
        with torch.cuda.device(self.dev):
            call("nsd_ctc_beam_nbest", ptr(self.state), self.B, self.W, self.max_frames, k, ptr(hyps), self.max_frames, ptr(hyp_len),
                 ptr(score), ptr(acoustic), stream())
        return hyps, hyp_len, score, acoustic


def ctc_beam_search(act: torch.Tensor, lens: Optional[torch.Tensor], beam_width: int = 16, nbest: int = 1, blank: int = 0,
                    lm: Optional[torch.Tensor] = None, lm_weight: float = 0.0, insertion_bonus: float = 0.0, is_logits: bool = False):
    """One-shot prefix beam search over ``act`` [T',B,C] (any strides; GRU logits go in as ``logits.permute(1, 0, 2)`` with
    ``is_logits=True``) -> the ``CtcBeamSearch.nbest`` tuple with ``max_frames = T'``."""
    require_cuda(act, "log_probs")
    if act.dim() != 3:
        raise NsdError(f"ctc beam search: expected [T', B, C], got {tuple(act.shape)}")
    T, B, C = act.shape
    if not 1 <= int(nbest) <= int(beam_width):
        raise NsdError(f"ctc beam search: nbest={nbest} outside [1, beam_width={beam_width}]")
    bs = CtcBeamSearch(B, C, beam_width, max(T, 1), blank, lm, lm_weight, insertion_bonus, device=act.device)
    bs.advance(act, lens, is_logits)
    return bs.nbest(nbest)


CtcAlignment = namedtuple("CtcAlignment", ["labels", "frame_logp", "spans", "token_logp", "score"])
CtcAlignment.__doc__ = """Result of ``ctc_forced_align``, all on the device: labels i32 [B,T'] (the path's label per frame, -1 past the
input length), frame_logp f32 [B,T'] (its log-probability, 0 past the length), spans i32 [B,S,2] (first and last frame of target k,
inclusive; -1 past the target length), token_logp f32 [B,S] (sum of frame_logp over the span, 0 past the target length) and score
f32 [B] (the path's log-probability; -inf for an utterance no path fits)."""


def ctc_forced_align(log_probs: torch.Tensor, targets: torch.Tensor, input_lengths: torch.Tensor, target_lengths: torch.Tensor,
                     blank: int = 0, is_logits: bool = False, check: bool = True) -> CtcAlignment:
    """CTC forced alignment (K5c, ``nsd_ctc_align``; no counterpart in the reference): the most probable path of every utterance
    through the blank-extended lattice of its true transcript, for a whole batch in one launch.  It says when each phoneme happens
    (``spans``) and how well each is supported (``token_logp``); ties go to the path that stays longest in each state.

    ``log_probs`` [T',B,C] may be any strided view, as for ``CTCLoss``: the trainer's ``.permute(1, 0, 2)``, or GRU logits with
    ``is_logits=True`` (log-softmaxed in the kernel, bit-identical to aligning ``log_softmax_tbc(logits)``).  The Conformer's
    ``log_probs`` go in as they are.  ``targets`` is 2-D padded [B,S] (S <= 1024); T' <= 8192, C <= 128.  An utterance with fewer
    frames than its target length plus its adjacent repeats gets score -inf and labels / spans -1.

    ``check=True`` reads the error flag once (a host synchronisation) and raises ``NsdError`` if a target equals ``blank`` or lies
    outside [0, C); those utterances get the infeasible outputs, the others are aligned normally.  ``check=False`` skips the read,
    so the call can be captured in a CUDA graph."""
    require_cuda(log_probs, "log_probs")
    if log_probs.dim() != 3:
        raise NsdError(f"ctc_forced_align: expected log_probs [T', B, C], got {tuple(log_probs.shape)}")
    if targets.dim() != 2:
        raise NsdError("ctc_forced_align: targets must be 2-D padded [B,S]")
    if log_probs.dtype != torch.float32:
        log_probs = log_probs.float()
    T, B, C = log_probs.shape
    if targets.shape[0] != B or input_lengths.numel() != B or target_lengths.numel() != B:
        raise NsdError(f"ctc_forced_align: batch {B} of log_probs does not match targets {tuple(targets.shape)} and the lengths")
    if not 1 <= C <= 128:
        raise NsdError(f"ctc_forced_align: C={C} outside [1, 128]")
    if not 0 <= blank < C:
        raise NsdError(f"ctc_forced_align: blank={blank} outside [0, {C})")
    dev = log_probs.device
    st, sb, sc = log_probs.stride()
    with torch.cuda.device(dev):          # raw-pointer launches must target the tensors' device, not the caller's current one
        err = torch.zeros(1, device=dev, dtype=torch.int32)
        out = CtcAlignment(*ops.ctc_align_raw(log_probs, st, sb, sc, is_logits, _as_i32(targets, dev), _as_i32(input_lengths, dev),
                                              _as_i32(target_lengths, dev), T, B, C, int(blank), err))
    if check and int(err.item()) != 0:
        raise NsdError(f"ctc_forced_align: a target equals blank={blank} or lies outside [0, {C})")
    return out


def frames_to_bins(spans: torch.Tensor, kernel_len: int, stride_len: int) -> torch.Tensor:
    """Frame spans of ``GRUDecoder`` output -> input-bin spans.  Frame t is the unfold window over bins
    [t*strideLen, t*strideLen + kernelLen) (model.py:96-101), so a span (f0, f1) of inclusive frames covers the half-open bin range
    [f0*strideLen, f1*strideLen + kernelLen); -1 stays -1.  The range does not include the reach of the Gaussian smoother in front
    of the unfold (its "same" padding reaches (n-1)//2 bins before and n-1-(n-1)//2 after for n taps: 9 and 10 for the 20 taps of
augmentations.py:91).  For the GRU only: mapping Conformer
    frames to bins is not provided."""
    f0, f1 = spans[..., 0], spans[..., 1]
    lo = torch.where(f0 >= 0, f0 * stride_len, f0)
    hi = torch.where(f1 >= 0, f1 * stride_len + kernel_len, f1)
    return torch.stack([lo, hi], dim=-1)


def phoneme_error_rate(log_probs, lens, targets, target_lengths, blank: int = 0, beam_width: Optional[int] = None,
                       lm: Optional[torch.Tensor] = None, lm_weight: float = 0.0, insertion_bonus: float = 0.0) -> Tuple[int, int]:
    """(sum of edit distances, sum of true lengths) for a batch -- `cer` numerator/denominator (trainer:332-333).
    ``beam_width=None`` decodes greedily as the reference does; otherwise the top hypothesis of the prefix beam search
    (with the optional prior) is scored.  One device->host read for the whole batch."""
    if beam_width is None:
        dec, dec_len = greedy_decode(log_probs, lens, blank)
    else:
        hyps, hyp_len, _, _ = ctc_beam_search(log_probs, lens, beam_width, 1, blank, lm, lm_weight, insertion_bonus)
        dec, dec_len = hyps[:, 0], hyp_len[:, 0]
    dist = edit_distances(dec, dec_len, targets, target_lengths)
    both = torch.stack([dist.sum(), _as_i32(target_lengths, dist.device).sum()]).cpu()
    return int(both[0]), int(both[1])


# ------------------------------------------------------------------------------------------------ K5d: words
# The competition's phone set in id order: PHONEMES[i] has class id i + 1 (0 = blank), SIL = 40 separates words.
PHONEMES = ("AA", "AE", "AH", "AO", "AW", "AY", "B", "CH", "D", "DH", "EH", "ER", "EY", "F", "G", "HH", "IH", "IY", "JH", "K", "L",
            "M", "N", "NG", "OW", "OY", "P", "R", "S", "SH", "T", "TH", "UH", "UW", "V", "W", "Y", "Z", "ZH")
SIL = len(PHONEMES) + 1
_PHONE_ID = {p: i + 1 for i, p in enumerate(PHONEMES)}


class Lexicon:
    """A pronunciation lexicon for ``WordBeamSearch``: a prefix tree over pronunciations (sequences of classes other than
    ``blank`` and ``sep``), node 0 = the root.  A word may have several pronunciations; several words may share one
    (homophones).  ``words[i]`` is the word with id i, in order of first appearance; ``prons[i]`` its pronunciations.

    ``nodes`` (int32 [n, 8]: child mask in four 32-bit words, first child, first homophone entry, homophone count, 0) and
    ``entries`` (int32 [m]: word ids, ascending within a node) are the arrays the kernel reads (include/nsd_b200.h, K5d)."""

    def __init__(self, pairs, num_classes: int, blank: int = 0, sep: int = SIL):
        self.num_classes, self.blank, self.sep = int(num_classes), int(blank), int(sep)
        C = self.num_classes
        if not 1 <= C <= 128:
            raise ValueError(f"lexicon: num_classes={C} outside [1, 128]")
        if not (0 <= self.blank < C and 0 <= self.sep < C) or self.blank == self.sep:
            raise ValueError(f"lexicon: blank={self.blank} and sep={self.sep} must be distinct classes of [0, {C})")
        self.words: List[str] = []
        self.word_index = {}
        self.prons: List[List[List[int]]] = []     # per word id: its pronunciations as class ids
        children = [{}]                          # build order; renumbered breadth first below
        homophones = [set()]
        for word, pron in pairs:
            ids = []
            for ph in pron:
                c = _PHONE_ID.get(_strip_stress(ph)) if isinstance(ph, str) else int(ph)
                if c is None:
                    raise ValueError(f"lexicon: unknown phone {ph!r} in the pronunciation of {word!r}")
                if not 0 <= c < C or c in (self.blank, self.sep):
                    raise ValueError(f"lexicon: class {c} in the pronunciation of {word!r} is outside [0, {C}) or is blank / sep")
                ids.append(c)
            if not ids:
                raise ValueError(f"lexicon: empty pronunciation of {word!r}")
            if word not in self.word_index:
                self.word_index[word] = len(self.words)
                self.words.append(word)
                self.prons.append([])
            self.prons[self.word_index[word]].append(ids)
            u = 0
            for c in ids:
                if c not in children[u]:
                    children[u][c] = len(children)
                    children.append({})
                    homophones.append(set())
                u = children[u][c]
            homophones[u].add(self.word_index[word])
        if not self.words:
            raise ValueError("lexicon: no words")
        # breadth-first numbering: the children of a node are consecutive, in class order
        order, new_id = [0], {0: 0}
        for u in order:
            for c in sorted(children[u]):
                new_id[children[u][c]] = len(order)
                order.append(children[u][c])
        nodes = np.zeros((len(order), 8), dtype=np.int64)
        entries = []
        self.children = []                       # per new node: {class: child}, host mirror of the mask
        self.node_words = []                     # per new node: sorted word ids
        for v, u in enumerate(order):
            kids = {c: new_id[x] for c, x in children[u].items()}
            self.children.append(kids)
            for c in kids:
                nodes[v, c >> 5] |= 1 << (c & 31)
            nodes[v, 4] = min(kids.values()) if kids else 0
            ws = sorted(homophones[u])
            self.node_words.append(ws)
            nodes[v, 5], nodes[v, 6] = len(entries), len(ws)
            entries.extend(ws)
        self.nodes = nodes.astype(np.uint32).view(np.int32)
        self.entries = np.asarray(entries, dtype=np.int32)

    @classmethod
    def from_pronunciations(cls, pairs, num_classes: int, blank: int = 0, sep: int = SIL) -> "Lexicon":
        """``pairs``: (word, pronunciation) with the pronunciation a sequence of class ids (or phone names of ``PHONEMES``)."""
        return cls(pairs, num_classes, blank, sep)

    @classmethod
    def from_file(cls, path: str) -> "Lexicon":
        """CMUdict-style lines ``WORD PH1 PH2 ...`` over the competition's phones (``PHONEMES``, stress digits stripped,
        variants ``WORD(2)`` folded into WORD; lines starting with ``;;;`` are comments): 41 classes, blank 0, sep SIL = 40."""
        pairs = []
        with open(path, encoding="utf-8") as f:
            for line in f:
                parts = line.split()
                if not parts or parts[0].startswith(";;;"):
                    continue
                word = re.sub(r"\(\d+\)$", "", parts[0])
                pairs.append((word, [_strip_stress(p) for p in parts[1:]]))
        return cls(pairs, len(PHONEMES) + 2, 0, SIL)


def _strip_stress(ph: str) -> str:
    return ph.rstrip("0123456789")


class NgramLM:
    """A word n-gram LM (order <= 3) loaded from an ARPA file, in natural log (ARPA's log10 x ln 10), stored as the sorted
    trie ``WordBeamSearch``'s kernel reads: unigrams (p1, bo1), the bigrams of each history word at ``b_off[a]..b_off[a+1]``
    sorted by word (p2, bo2), the trigrams of each bigram j at ``t_off[j]..t_off[j+1]`` sorted by word (p3).  Words have
    ids in the order of the 1-gram section.  Absent backoffs are 0."""

    def __init__(self, vocab, p1, bo1, bigrams, trigrams):
        self.vocab = list(vocab)
        self.index = {w: i for i, w in enumerate(self.vocab)}
        V = len(self.vocab)
        self.p1, self.bo1 = np.asarray(p1, np.float32), np.asarray(bo1, np.float32)
        big = sorted(bigrams.items())                # ((a, w), (p, bo))
        self.b_word = np.array([w for (a, w), _ in big], dtype=np.int32)
        self.p2 = np.array([v[0] for _, v in big], dtype=np.float32)
        self.bo2 = np.array([v[1] for _, v in big], dtype=np.float32)
        self.b_off = np.searchsorted(np.array([a for (a, _), _ in big], dtype=np.int64), np.arange(V + 1)).astype(np.int32)
        bindex = {k: j for j, (k, _) in enumerate(big)}
        tri = sorted(((bindex[(a, b)], w), p) for (a, b, w), p in trigrams.items())
        self.t_word = np.array([w for (_, w), _ in tri], dtype=np.int32)
        self.p3 = np.array([p for _, p in tri], dtype=np.float32)
        self.t_off = np.searchsorted(np.array([j for (j, _), _ in tri], dtype=np.int64), np.arange(len(big) + 1)).astype(np.int32)
        self.order = 3 if tri else (2 if big else 1)

    @classmethod
    def from_arpa(cls, path: str) -> "NgramLM":
        """Parse an ARPA file of order 1..3.  Raises ``ValueError`` if a section's count differs from its ``\\data\\`` line,
        an n-gram appears twice, an n-gram's (n-1)-prefix is absent, or a word of a longer n-gram is not a unigram."""
        ln10 = math.log(10.0)
        counts, grams, section = {}, {1: {}, 2: {}, 3: {}}, None
        with open(path, encoding="utf-8") as f:
            for raw in f:
                line = raw.strip()
                if not line:
                    continue
                if line == "\\data\\":
                    section = 0
                    continue
                if line == "\\end\\":
                    break
                m = re.fullmatch(r"\\(\d+)-grams:", line)
                if m:
                    section = int(m.group(1))
                    if not 1 <= section <= 3:
                        raise ValueError(f"ARPA {path}: order {section} > 3 is not supported")
                    continue
                if section == 0:
                    m = re.fullmatch(r"ngram\s+(\d+)\s*=\s*(\d+)", line)
                    if not m:
                        raise ValueError(f"ARPA {path}: bad \\data\\ line {line!r}")
                    counts[int(m.group(1))] = int(m.group(2))
                    continue
                if section is None:
                    continue
                parts = line.split()
                n = section
                if len(parts) not in (n + 1, n + 2):
                    raise ValueError(f"ARPA {path}: bad {n}-gram line {line!r}")
                key = tuple(parts[1:n + 1])
                if key in grams[n]:
                    raise ValueError(f"ARPA {path}: duplicate {n}-gram {' '.join(key)}")
                grams[n][key] = (float(parts[0]) * ln10, float(parts[n + 1]) * ln10 if len(parts) == n + 2 else 0.0)
        if max(counts, default=0) > 3:
            raise ValueError(f"ARPA {path}: order {max(counts)} > 3 is not supported")
        for n in (1, 2, 3):
            if counts.get(n, 0) != len(grams[n]):
                raise ValueError(f"ARPA {path}: \\data\\ says {counts.get(n, 0)} {n}-grams, the file has {len(grams[n])}")
        if not grams[1]:
            raise ValueError(f"ARPA {path}: no unigrams")
        vocab = [k[0] for k in grams[1]]
        idx = {w: i for i, w in enumerate(vocab)}
        for n in (2, 3):
            for key in grams[n]:
                if key[:-1] not in grams[n - 1] or key[-1] not in idx:
                    raise ValueError(f"ARPA {path}: {n}-gram {' '.join(key)} has no {n - 1}-gram prefix or an unknown word")
        p1 = [grams[1][(w,)][0] for w in vocab]
        bo1 = [grams[1][(w,)][1] for w in vocab]
        big = {(idx[a], idx[w]): v for (a, w), v in grams[2].items()}
        tri = {(idx[a], idx[b], idx[w]): v[0] for (a, b, w), v in grams[3].items()}
        return cls(vocab, p1, bo1, big, tri)

    def _find2(self, a: int, b: int) -> int:
        lo, hi = int(self.b_off[a]), int(self.b_off[a + 1])
        j = lo + int(np.searchsorted(self.b_word[lo:hi], b))
        return j if j < hi and self.b_word[j] == b else -1

    def logp_ids(self, w: int, a: int, b: int) -> float:
        """lm(w | a, b) over word ids; a < 0: history of one word."""
        bo = 0.0
        if a >= 0:
            j = self._find2(a, b)
            if j >= 0:
                lo, hi = int(self.t_off[j]), int(self.t_off[j + 1])
                k = lo + int(np.searchsorted(self.t_word[lo:hi], w))
                if k < hi and self.t_word[k] == w:
                    return float(self.p3[k])
                bo = float(self.bo2[j])
        j = self._find2(b, w)
        return bo + (float(self.p2[j]) if j >= 0 else float(self.bo1[b]) + float(self.p1[w]))

    def word_id(self, word: str) -> int:
        if word in self.index:
            return self.index[word]
        if "<unk>" in self.index:
            return self.index["<unk>"]
        raise KeyError(f"word LM: {word!r} is not in the vocabulary and the LM has no <unk>")

    def logp(self, word: str, history: Sequence[str] = ("<s>",)) -> float:
        """Natural-log lm(word | the last two words of ``history``), with ARPA backoff; unknown words map to ``<unk>``."""
        h = [self.word_id(x) for x in history][-2:]
        if not h:
            raise ValueError("word LM: the history needs at least one word (the start is '<s>')")
        return self.logp_ids(self.word_id(word), h[0] if len(h) == 2 else -1, h[-1])

    def arrays(self):
        """-> (idx int32, val float32): b_off | b_word | t_off | t_word and p1 | bo1 | p2 | bo2 | p3, as the kernel reads them."""
        idx = np.concatenate([self.b_off, self.b_word, self.t_off, self.t_word]).astype(np.int32)
        val = np.concatenate([self.p1, self.bo1, self.p2, self.bo2, self.p3]).astype(np.float32)
        return idx, val


WordHypotheses = namedtuple("WordHypotheses", ["hyps", "hyp_len", "words", "word_len", "score", "acoustic"])
WordHypotheses.__doc__ = """``WordBeamSearch.nbest``, best first, on the device: hyps i64 [B,k,max_frames] (phonemes, -1 past hyp_len), hyp_len i32
[B,k], words i64 [B,k,max_frames//2+1] (lexicon word ids, -1 past word_len), word_len i32 [B,k], score f32 [B,k] (acoustic + prior,
plus the end term when final) and acoustic f32 [B,k] (the CTC prefix log-probability).  Entries past the beam, and with
``final`` entries inside an unfinished word, have lengths 0 and score / acoustic -inf."""


LIVE_HEADER = 4      # a live read-out row: committed, first, top word count, overflow; then the words


def read_live(buf):
    """A live read-out on the host (``WordBeamSearch.enqueue_live``'s buffer, int32 [B, LIVE_HEADER + cap], or one row of it) -> per
    row (the committed word ids this read-out hands out, the tentative word ids after all committed ones, more): ``more`` when
    committed words did not fit the row; they come with the next read-out, and the tentative list is then empty."""
    a = np.asarray(buf)
    out = []
    for r in (a[None] if a.ndim == 1 else a).tolist():
        committed, first, top, cap = r[0], r[1], r[2], len(r) - LIVE_HEADER
        n = min(committed, first + cap) - first
        out.append((r[LIVE_HEADER:LIVE_HEADER + n], r[LIVE_HEADER + n:LIVE_HEADER + min(top - first, cap)], committed - first > cap))
    return out[0] if a.ndim == 1 else out


class WordBeamSearch(CtcBeamSearch):
    """Lexicon-constrained CTC prefix beam search with an optional word n-gram LM (K5d, ``nsd_ctc_word_beam_*``).

    K5b's beam (``CtcBeamSearch``: resumable on the device, any chunking gives the same bits) whose hypotheses spell
    ``pron(w1) sep pron(w2) sep ...``: a phoneme extends a hypothesis only along the lexicon, and ``sep`` ends a word,
    adding ``lm_weight * lm(word | two previous words) + word_bonus`` to its prior (the best-scoring homophone, ties to the
    smaller word id).  The classes, ``blank`` and ``sep`` are the lexicon's.  K5b's phoneme-bigram ``lm`` tensor does not
    combine with a lexicon (raises)."""

    def __init__(self, batch: int, lexicon: Lexicon, lm: Optional[NgramLM] = None, beam_width: int = 16, max_frames: int = 4096,
                 lm_weight: float = 0.0, word_bonus: float = 0.0, blank: Optional[int] = None, sep: Optional[int] = None, device=None):
        if isinstance(lm, torch.Tensor):
            raise NsdError("word beam search: a phoneme-bigram lm tensor (K5b) cannot be combined with a lexicon; pass an NgramLM")
        if lm is not None and not isinstance(lm, NgramLM):
            raise NsdError(f"word beam search: lm must be an NgramLM, got {type(lm).__name__}")
        if not isinstance(lexicon, Lexicon):
            raise NsdError(f"word beam search: lexicon must be a Lexicon, got {type(lexicon).__name__}")
        if (blank is not None and int(blank) != lexicon.blank) or (sep is not None and int(sep) != lexicon.sep):
            raise NsdError(f"word beam search: blank={blank} / sep={sep} differ from the lexicon's {lexicon.blank} / {lexicon.sep}")
        self.lexicon, self.word_lm, self.sep = lexicon, lm, lexicon.sep
        lm_ids = np.zeros(len(lexicon.words), dtype=np.int32)
        self._bos = self._eos = -1
        if lm is not None:
            try:
                lm_ids = np.array([lm.word_id(w) for w in lexicon.words], dtype=np.int32)
                self._bos, self._eos = lm.index["<s>"], lm.index["</s>"]
            except KeyError as e:
                raise NsdError(f"word beam search: {e}") from None
        super().__init__(batch, lexicon.num_classes, beam_width, max_frames, lexicon.blank, None, 0.0, 0.0, device)
        self.lm_weight, self.word_bonus = float(lm_weight), float(word_bonus)
        self.max_words = self.max_frames // 2 + 1
        self._nodes = torch.from_numpy(lexicon.nodes).to(self.dev).contiguous()
        self._entries = torch.from_numpy(np.stack([lexicon.entries, lm_ids[lexicon.entries]], axis=1)).to(self.dev).contiguous()
        self._lm_idx = self._lm_val = None
        self._lm_sizes = (0, 0, 0)
        if lm is not None:
            idx, val = lm.arrays()
            self._lm_idx, self._lm_val = torch.from_numpy(idx).to(self.dev), torch.from_numpy(val).to(self.dev)
            self._lm_sizes = (len(lm.vocab), len(lm.b_word), len(lm.t_word))

    def _state_bytes(self) -> int:
        return _lib.lib().nsd_ctc_word_beam_state_bytes(self.B, self.W, self.max_frames)

    def reset(self) -> None:
        """Back to the empty hypothesis at the lexicon root, in place; the live read-out's counters back to 0."""
        with torch.cuda.device(self.dev):
            call("nsd_ctc_word_beam_init", ptr(self.state), self.state_bytes, self.B, self.W, self.max_frames, self._bos, stream())
            self.err_flag.zero_()
            self.reset_reported()
        self.frames = 0

    def _check_mask(self, mask: torch.Tensor) -> None:
        if mask.device != self.dev or mask.dtype != torch.int32 or tuple(mask.shape) != (self.B,) or not mask.is_contiguous():
            raise NsdError(f"word beam search: mask must be a contiguous int32 [{self.B}] tensor on {self.dev}")

    def reset_utterances(self, mask: torch.Tensor) -> None:
        """As ``CtcBeamSearch.reset_utterances``: only the utterances with ``mask[b] != 0`` start again; the others keep every byte.
        The live read-out's counters are not touched (``reset_reported(mask)``)."""
        self._check_mask(mask)
        with torch.cuda.device(self.dev):
            call("nsd_ctc_word_beam_reset", ptr(self.state), self.state_bytes, self.B, self.W, self.max_frames, self._bos, ptr(mask),
                 stream())

    # ---- live read-out
    def reset_reported(self, mask: Optional[torch.Tensor] = None) -> None:
        """Zero the live read-out's counters of committed words handed out (``reported``, i32 [B] on the device), in place: all of
        them, or those with ``mask[b] != 0``.  Goes with ``reset`` / ``reset_utterances`` of the same utterances."""
        if getattr(self, "reported", None) is None:
            self.reported = torch.zeros(self.B, device=self.dev, dtype=torch.int32)
        elif mask is None:
            self.reported.zero_()
        else:
            self._check_mask(mask)
            self.reported.masked_fill_(mask != 0, 0)

    def live_buffer(self, cap: int = 64) -> torch.Tensor:
        """A device buffer for ``enqueue_live``: int32 [B, LIVE_HEADER + cap]."""
        if int(cap) < 1:
            raise NsdError(f"word beam search: live read-out cap={cap} must be positive")
        return torch.empty((self.B, LIVE_HEADER + int(cap)), device=self.dev, dtype=torch.int32)

    def enqueue_live(self, out: torch.Tensor) -> None:
        """Launch the live read-out into ``out`` (``live_buffer``): per utterance {committed, first, top word count, overflow} and the
        top hypothesis's words from ``first`` on; ``read_live`` decodes a row.  Committed = the longest common word-id prefix of the
        hypotheses alive now, final whatever frames follow.  Each committed word is handed out once: the device counter
        ``reported`` moves past the words written here.  No host synchronisation: the unit a CUDA graph captures."""
        if out.device != self.dev or out.dtype != torch.int32 or out.dim() != 2 or out.shape[0] != self.B or out.shape[1] <= LIVE_HEADER \
                or not out.is_contiguous():
            raise NsdError(f"word beam search: live buffer must be a contiguous int32 [{self.B}, {LIVE_HEADER} + cap] tensor on {self.dev}")
        call("nsd_ctc_word_beam_live", ptr(self.state), self.B, self.W, self.max_frames, ptr(self.reported), out.shape[1] - LIVE_HEADER,
             ptr(out), stream())

    def _model_args(self):
        V, n2, n3 = self._lm_sizes
        return (ptr(self._nodes), self._nodes.shape[0], ptr(self._entries), self._entries.shape[0], ptr(self._lm_idx), ptr(self._lm_val),
                V, n2, n3)

    def enqueue(self, act: torch.Tensor, lens: Optional[torch.Tensor] = None, is_logits: bool = False) -> None:
        """Launch the advance without counting frames (the caller has reserved them): the unit a CUDA graph captures."""
        T = act.shape[0]
        st, sb, sc = act.stride()
        call("nsd_ctc_word_beam_advance", ptr(act), st, sb, sc, int(bool(is_logits)), ptr(lens), T, self.B, self.C, self.blank, self.sep,
             *self._model_args(), self.lm_weight, self.word_bonus, self.W, self.max_frames, ptr(self.state), self.state_bytes,
             ptr(self.err_flag), stream())

    def nbest(self, k: int = 1, final: bool = True) -> WordHypotheses:
        """The best ``k`` hypotheses (``WordHypotheses``); the state is not changed.  ``final=False``: the beam as it stands.
        ``final=True``: the utterance ends here: a hypothesis at the lexicon root gets ``lm_weight * lm(</s> | history)``,
        one at the end of a word gets that word (its separator increment) and then ``</s>``, any other is dropped; re-ranked."""
        k = int(k)
        if not 1 <= k <= self.W:
            raise NsdError(f"word beam search: nbest={k} outside [1, beam_width={self.W}]")
        hyps = torch.empty((self.B, k, self.max_frames), device=self.dev, dtype=torch.int64)
        hyp_len = torch.empty((self.B, k), device=self.dev, dtype=torch.int32)
        words = torch.empty((self.B, k, self.max_words), device=self.dev, dtype=torch.int64)
        word_len = torch.empty((self.B, k), device=self.dev, dtype=torch.int32)
        score = torch.empty((self.B, k), device=self.dev, dtype=torch.float32)
        acoustic = torch.empty((self.B, k), device=self.dev, dtype=torch.float32)
        with torch.cuda.device(self.dev):
            call("nsd_ctc_word_beam_nbest", ptr(self.state), self.B, self.W, self.max_frames, *self._model_args(), self._eos,
                 self.lm_weight, self.word_bonus, int(bool(final)), k, ptr(hyps), self.max_frames, ptr(hyp_len), ptr(words),
                 self.max_words, ptr(word_len), ptr(score), ptr(acoustic), stream())
        return WordHypotheses(hyps, hyp_len, words, word_len, score, acoustic)


def word_beam_search(act: torch.Tensor, lens: Optional[torch.Tensor], lexicon: Lexicon, lm: Optional[NgramLM] = None,
                     beam_width: int = 16, nbest: int = 1, lm_weight: float = 0.0, word_bonus: float = 0.0, is_logits: bool = False,
                     final: bool = True) -> WordHypotheses:
    """One-shot lexicon-constrained beam search over ``act`` [T',B,C] (any strides; GRU logits as ``logits.permute(1, 0, 2)`` with
    ``is_logits=True``) -> ``WordBeamSearch.nbest`` with ``max_frames = T'``."""
    require_cuda(act, "log_probs")
    if act.dim() != 3:
        raise NsdError(f"word beam search: expected [T', B, C], got {tuple(act.shape)}")
    T, B, _ = act.shape
    if not 1 <= int(nbest) <= int(beam_width):
        raise NsdError(f"word beam search: nbest={nbest} outside [1, beam_width={beam_width}]")
    bs = WordBeamSearch(B, lexicon, lm, beam_width, max(T, 1), lm_weight, word_bonus, device=act.device)
    bs.advance(act, lens, is_logits)
    return bs.nbest(nbest, final)


def words_to_ids(transcripts, lexicon: Lexicon) -> Tuple[torch.Tensor, torch.Tensor]:
    """Transcripts (strings split on whitespace, or sequences of words) -> (ids int32 [B,S], lengths int32 [B]) on the host,
    exact-match lexicon word ids; a word outside the lexicon gets -1, which no hypothesis contains (always an error)."""
    rows = [t.split() if isinstance(t, str) else list(t) for t in transcripts]
    S = max([1] + [len(r) for r in rows])
    ids = torch.full((len(rows), S), -1, dtype=torch.int32)
    for b, r in enumerate(rows):
        ids[b, :len(r)] = torch.tensor([lexicon.word_index.get(w, -1) for w in r], dtype=torch.int32)
    return ids, torch.tensor([len(r) for r in rows], dtype=torch.int32)


def ids_to_words(ids, lexicon: Lexicon) -> List[str]:
    """Word ids (a 1-D sequence or tensor) -> words; negative entries (padding) are skipped."""
    vals = ids.tolist() if isinstance(ids, torch.Tensor) else list(ids)
    return [lexicon.words[i] for i in vals if i >= 0]


def word_error_rate(act: torch.Tensor, lens: torch.Tensor, word_targets: torch.Tensor, word_target_lengths: torch.Tensor,
                    decoder: WordBeamSearch, is_logits: bool = False) -> Tuple[int, int]:
    """(sum of word edit distances, sum of target words) for a batch: ``decoder`` (a ``WordBeamSearch`` of the batch's size,
    reset here) decodes ``act`` [T',B,C] and its final top hypothesis is compared with ``word_targets`` (2-D padded lexicon
    word ids, ``words_to_ids``; -1 never matches) by the Levenshtein kernel.  One device->host read for the whole batch.  The
    Conformer's ``log_probs`` go in as they are; GRU logits with ``is_logits=True`` (``trainer.eval_batch_words``)."""
    if not isinstance(decoder, WordBeamSearch):
        raise NsdError("word_error_rate: decoder must be a WordBeamSearch")
    decoder.reset()
    decoder.advance(act, lens, is_logits)
    r = decoder.nbest(1, final=True)
    dist = edit_distances(r.words[:, 0], r.word_len[:, 0], word_targets, word_target_lengths)
    both = torch.stack([dist.sum(), _as_i32(word_target_lengths, dist.device).sum()]).cpu()
    return int(both[0]), int(both[1])
