"""CTC loss, greedy decode, prefix beam search, forced alignment and phoneme error rate on the sm_100a kernels (K4 / K5 / K5b / K5c).

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

from collections import namedtuple
from typing import List, Optional, Sequence, Tuple

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
        self.state_bytes = _lib.lib().nsd_ctc_beam_state_bytes(self.B, self.W, self.max_frames)
        self.state = torch.empty(self.state_bytes, device=self.dev, dtype=torch.uint8)
        self.err_flag = torch.zeros(1, device=self.dev, dtype=torch.int32)
        self.reset()

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
