"""Hot-loop lines of the reference trainer, on the B200 kernels.

Only what sits on the north-star path is mirrored here (neural_decoder_trainer.py):
  make_optimizer  :163-175   Adam(lr, betas .9/.999, eps=0.1, weight_decay=l2) + LinearLR
  train_step      :208-218, 242, 251-260   forward -> out_lens -> log-softmax + CTC -> backward -> step
  eval_batch      :299-333   forward -> CTC loss -> greedy decode -> edit distance
  align_batch     (new)      forward -> forced alignment of the true transcript -> per-phoneme frame and bin spans
  input_attribution (new)    forward + backward to the input: saliency / integrated gradients of each utterance's CTC NLL
Data loading, wandb, checkpointing stay the reference's business; its ``trainModel`` runs unchanged with
``GRUDecoder`` / ``CTCLoss`` swapped in (INTEGRATION.md).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import ctc as _ctc
from .adam import FusedAdam


def _step_in_backward() -> bool:
    import os
    return os.environ.get("NSD_STEP_IN_BACKWARD", "1") != "0"


def make_optimizer(model: torch.nn.Module, args: dict):
    """trainer:163-175 (the non-AdamW branch, which the GRU configs use)."""
    opt = FusedAdam(model.parameters(), lr=args["lrStart"], betas=(0.9, 0.999), eps=0.1,
                    weight_decay=args.get("l2_decay", 0.0))
    if getattr(model, "_shadows", None) is not None:
        opt.attach_shadows(model._shadows)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=args["lrEnd"] / args["lrStart"],
                                              total_iters=args["nBatch"])
    return opt, sched


class _UpdateSchedule:
    """Which parameters the bf16 train step updates when, relative to the BPTT launches and the all-reduces.

    K3 leaves SMs and most of the HBM bandwidth idle, so the update of a gradient bucket that is final is issued from inside the
    backward as the launch directly behind a BPTT launch, and runs under it (``FusedAdam.step(under_recurrence=True)``).  A bucket
    released in front of BPTT(l) is updated directly behind
      - BPTT(l) on one GPU;
      - BPTT(l-1) when data parallel: its all-reduce runs under BPTT(l), and the compute stream waits for it in front of BPTT(l-1).
    At most one bucket waits at a time.  What is released after the last BPTT launch, or is still waiting then, is updated by
    ``train_step`` after the backward.  ``decoder_backward_tc`` reports to it through ``released`` and ``bptt``."""

    def __init__(self, optimizer: FusedAdam, data_parallel: bool):
        self.optimizer = optimizer
        self.data_parallel = data_parallel
        self.updated = set()            # id() of every parameter updated so far
        self._released = None           # (pairs, collective handle): released since the last BPTT launch
        self._waiting = None            # data parallel: released in front of the last BPTT launch, its all-reduce running under it

    def released(self, pairs, handle) -> None:
        """The gradients of ``pairs`` [(parameter, gradient)] are final; ``handle`` is their all-reduce's work handle (or None)."""
        self._released = (pairs, handle)

    def bptt(self, launch):
        """Issue a BPTT launch (``launch()``, whose result is returned) with the update that is due directly behind it."""
        if self.data_parallel:
            due, self._waiting = self._waiting, self._released
            if due is not None:
                due[1].wait()
        else:
            due = self._released
        self._released = None
        out = launch()
        if due is not None:
            ps = []
            for p, g in due[0]:
                if p.requires_grad and p.grad is None and g is not None:
                    p.grad = g
                    ps.append(p)
            if ps:
                self.updated.update(id(p) for p in ps)
                self.optimizer.step(only=ps, under_recurrence=True)
        return out

    def not_updated(self, params, grads) -> tuple:
        """``grads`` with None for every parameter this schedule has updated (its ``.grad`` is set already)."""
        return tuple(None if id(p) in self.updated else g for p, g in zip(params, grads))


class LossReader:
    """Host read-back of a step's loss that does not drain the backward behind it.  ``loss.item()`` on the compute stream waits for the
    whole step (the stream is in order) and the GPU then idles until the host has enqueued the next step's first kernels; the loss itself
    is final after the forward + CTC kernel, ~40 % into the step.  ``train_step(..., loss_reader=r)`` copies it to a pinned float on a side
    stream as soon as it exists; ``r.item()`` waits for that copy only, so the host enqueues step i+1 while step i's backward still runs."""

    def __init__(self, device):
        self.device = torch.device(device)
        self.buf = torch.zeros(1, dtype=torch.float32).pin_memory()
        self.stream = torch.cuda.Stream(self.device)
        self.done = torch.cuda.Event()
        self._ready = torch.cuda.Event()

    def capture(self, loss: torch.Tensor) -> None:
        self._ready.record(torch.cuda.current_stream(self.device))
        self.stream.wait_event(self._ready)
        with torch.cuda.stream(self.stream):
            self.buf.copy_(loss.detach().reshape(1), non_blocking=True)
            self.done.record(self.stream)
        loss.record_stream(self.stream)

    def item(self) -> float:
        self.done.synchronize()
        return float(self.buf[0])


def train_step(model, optimizer, X, y, X_len, y_len, dayIdx, scheduler=None, grad_sync=None,
               white_noise_sd: float = 0.0, constant_offset_sd: float = 0.0, loss_reader: Optional[LossReader] = None) -> torch.Tensor:
    """One optimisation step; returns the (device) loss scalar.  ``grad_sync`` is the data-parallel hook
    (parallel.GradSync): it all-reduces gradients bucket by bucket while the backward is still running.
    ``white_noise_sd`` / ``constant_offset_sd`` (args["whiteNoiseSD"], args["constantOffsetSD"]): the in-loop
    augmentation of trainer:194-201, generated inside the front-end kernel instead of in extra passes over X.
    ``loss_reader`` (LossReader): host read-back of the loss that does not wait for the backward."""
    model.grad_sync = grad_sync
    # the buckets are all-reduced with SUM: the 1/world average is folded into the Adam kernel.  Adam with eps=0.1 and
    # L2-in-gradient is NOT scale-invariant, so the scale must follow the sync object on every step.
    want_scale = grad_sync.grad_scale if grad_sync is not None else 1.0
    if isinstance(optimizer, FusedAdam):
        optimizer.grad_scale = want_scale
    elif grad_sync is not None and grad_sync.world > 1:
        raise RuntimeError("train_step(grad_sync=...) sums gradients over ranks; use FusedAdam (make_optimizer), which folds the "
                           "1/world_size average into its update, or divide the gradients yourself")
    model.input_noise = (white_noise_sd, constant_offset_sd) if (white_noise_sd or constant_offset_sd) else None
    schedule = None
    if (isinstance(optimizer, FusedAdam) and getattr(model, "precision", None) == "bf16" and _step_in_backward()
            and len(optimizer.param_groups) == 1 and (grad_sync is None or grad_sync.world > 1)):
        schedule = _UpdateSchedule(optimizer, data_parallel=grad_sync is not None)
    model.step_hook = schedule
    pred = model.forward(X, dayIdx)                                         # trainer:208
    lens = _ctc.out_lens(X_len, model.kernelLen, model.strideLen)           # trainer:209
    loss = _ctc.ctc_loss_from_logits(pred, y, lens, y_len, blank=0, reduction="mean")   # trainer:210-218, 242
    if loss_reader is not None:
        loss_reader.capture(loss)
    optimizer.zero_grad(set_to_none=True)                                   # trainer:251
    if grad_sync is not None:
        grad_sync.begin()
    try:
        loss.backward()                                                     # trainer:252
    finally:
        model.step_hook = None
    if not isinstance(optimizer, FusedAdam):
        if grad_sync is not None:
            grad_sync.finish()
        optimizer.step()                                                    # trainer:259
    else:
        done = schedule.updated if schedule is not None else set()
        left = [p for g in optimizer.param_groups for p in g["params"] if p.grad is not None and id(p) not in done]
        if grad_sync is not None and grad_sync.world > 1:
            # the last big bucket (layer 0) is still being all-reduced when the backward's kernels are done: update the parameters of
            # every finished bucket under it, then the rest (same arithmetic per parameter; the step is just issued in two launches)
            in_flight = grad_sync.finish_early()
            if in_flight:
                optimizer.step(only=[p for p in left if p.grad.untyped_storage().data_ptr() not in in_flight])
                left = [p for p in left if p.grad.untyped_storage().data_ptr() in in_flight]
        if grad_sync is not None:
            grad_sync.finish()
        optimizer.step(only=left)                                           # trainer:259
    if scheduler is not None:
        scheduler.step()                                                    # trainer:260
    return loss.detach()


@torch.no_grad()
def eval_batch(model, X, y, X_len, y_len, dayIdx, beam_width=None, lm=None, lm_weight=0.0,
               insertion_bonus=0.0) -> Tuple[torch.Tensor, int, int]:
    """trainer:299-333 for one batch: (ctc loss, sum edit distance, sum true length).  ``beam_width`` (None: greedy, as the
    reference) scores the top hypothesis of the prefix beam search instead, optionally with a phoneme-bigram prior."""
    logits = model.forward(X, dayIdx)                                       # trainer:299
    lens = _ctc.out_lens(X_len, model.kernelLen, model.strideLen)           # trainer:300
    pred = _ctc.log_softmax_tbc(logits)                                     # trainer:301  [T',B,C] view
    loss = _ctc.CTCLoss(blank=0, reduction="mean", zero_infinity=True)(pred, y, lens, y_len)   # trainer:303-309
    # decode from the log-probs, as the reference does: log-softmax can create ties the raw logits lack
    dist, tot = _ctc.phoneme_error_rate(pred, lens, y, y_len, beam_width=beam_width, lm=lm, lm_weight=lm_weight,
                                        insertion_bonus=insertion_bonus)    # trainer:313-333
    return loss, dist, tot


@torch.no_grad()
def align_batch(model, X, y, X_len, y_len, dayIdx):
    """The alignment twin of ``eval_batch`` (no counterpart in the reference): forward, ``out_lens``, then ``ctc_forced_align`` of
    the true transcripts on the logits (log-softmaxed in the kernel).  Returns ``(alignment, bins)``: the ``CtcAlignment`` and the
    input-bin span [start, end) of every target phoneme (``frames_to_bins``; -1 past the target length or for infeasible
    utterances).  For ``GRUDecoder``; a Conformer's ``log_probs`` can go to ``ctc_forced_align`` directly."""
    logits = model.forward(X, dayIdx)                                       # trainer:299
    lens = _ctc.out_lens(X_len, model.kernelLen, model.strideLen)           # trainer:300
    ali = _ctc.ctc_forced_align(logits.permute(1, 0, 2), y, lens, y_len, blank=0, is_logits=True)
    return ali, _ctc.frames_to_bins(ali.spans, model.kernelLen, model.strideLen)


def _utterance_nll(model, X, y, X_len, y_len, dayIdx) -> torch.Tensor:
    """CTC NLL of every utterance's true transcript (zero_infinity=True) on the trainer's output lengths, differentiable in X."""
    from .conformer import NeuralTransformerCTCModel
    if isinstance(model, NeuralTransformerCTCModel):
        log_probs, lens, _ = model(X, dayIdx, X_len)
        return _ctc.CTCLoss(blank=0, reduction="none", zero_infinity=True)(log_probs, y, lens, y_len)
    logits = model.forward(X, dayIdx)
    lens = _ctc.out_lens(X_len, model.kernelLen, model.strideLen)
    return _ctc.ctc_loss_from_logits(logits, y, lens, y_len, blank=0, reduction="none")


def input_attribution(model, X, y, X_len, y_len, dayIdx, method: str = "saliency", steps: int = 32,
                      baseline: Optional[torch.Tensor] = None, max_batch: int = 256) -> Tuple[torch.Tensor, torch.Tensor]:
    """Which input bins and channels drive each utterance's transcript (no counterpart in the reference; the analysis twin of
    ``eval_batch`` / ``align_batch``), for ``GRUDecoder`` and ``NeuralTransformerCTCModel``.

    The target is nll_b, the CTC NLL of utterance b's true transcript on the trainer's output lengths (``zero_infinity=True``),
    summed over the batch; utterances do not interact, so the gradient at X[b] is d nll_b / d X[b].
      method="saliency":             that gradient.
      method="integrated_gradients": (X - baseline) times the mean gradient at baseline + a_k (X - baseline), a_k = (k + 1/2) / steps,
                                     k < steps (midpoint rule).  baseline None = zeros; any tensor that broadcasts to X.
    The inputs (B of them, or steps*B for integrated gradients) run in batches of at most ``max_batch`` utterances.
    Returns ``(attribution f32 [B,T,N], nll f32 [B] at X)`` on the device.

    The model runs in eval mode with every parameter frozen, so the backward makes no parameter gradient; the ``training`` flag of
    every submodule and every ``requires_grad`` flag are restored afterwards, also when the call raises.  Bins at or past ``X_len``
    are not masked: the reverse GRU direction runs over the padding, as in the reference, so they can receive gradient."""
    if method not in ("saliency", "integrated_gradients"):
        raise ValueError(f"method must be 'saliency' or 'integrated_gradients', got {method!r}")
    if int(steps) < 1 or int(max_batch) < 1:
        raise ValueError(f"steps={steps} and max_batch={max_batch} must be at least 1")
    if X.dim() != 3:
        raise RuntimeError(f"X must be [B,T,N], got {tuple(X.shape)}")
    X = X.detach().float()
    B = X.shape[0]
    dev = X.device
    y, X_len, y_len, dayIdx = (t.to(dev) for t in (y, X_len, y_len, dayIdx))
    params = list(model.parameters())
    flags = [p.requires_grad for p in params]
    modes = {mod: mod.training for mod in model.modules()}
    grad_sync = getattr(model, "grad_sync", None)
    try:
        model.eval()
        if grad_sync is not None:
            model.grad_sync = None
        for p in params:
            p.requires_grad_(False)

        def grad_at(xs, idx):
            """(nll, d nll / d xs) of the utterances ``idx`` at inputs ``xs``."""
            with torch.enable_grad():
                xs = xs.detach().requires_grad_(True)
                nll = _utterance_nll(model, xs, y[idx], X_len[idx], y_len[idx], dayIdx[idx])
                (g,) = torch.autograd.grad(nll.sum(), xs)
            return nll.detach(), g

        if method == "saliency":
            parts = [grad_at(X[i:i + max_batch], torch.arange(i, min(B, i + max_batch), device=dev)) for i in range(0, B, max_batch)]
            return torch.cat([g for _, g in parts]), torch.cat([n for n, _ in parts])
        base = torch.zeros_like(X) if baseline is None else baseline.to(device=dev, dtype=torch.float32).expand_as(X)
        diff = X - base
        total = torch.zeros_like(X)
        # the steps*B inputs in (k, b) order; each chunk's gradients are added per step k, in ascending k: a fixed order
        for i in range(0, steps * B, max_batch):
            flat = torch.arange(i, min(steps * B, i + max_batch), device=dev)
            k, b = flat // B, flat % B
            alpha = ((k.float() + 0.5) / steps).view(-1, 1, 1)
            _, g = grad_at(base[b] + alpha * diff[b], b)
            for kk in range(i // B, (i + len(flat) - 1) // B + 1):
                f0, f1 = max(kk * B, i), min((kk + 1) * B, i + len(flat))       # flat indices of step kk in this chunk
                total[f0 - kk * B:f1 - kk * B] += g[f0 - i:f1 - i]
        with torch.no_grad():
            nll = torch.cat([_utterance_nll(model, X[j:j + max_batch], y[j:j + max_batch], X_len[j:j + max_batch],
                                            y_len[j:j + max_batch], dayIdx[j:j + max_batch]) for j in range(0, B, max_batch)])
        return total / steps * diff, nll
    finally:
        for p, f in zip(params, flags):
            p.requires_grad_(f)
        if grad_sync is not None:
            model.grad_sync = grad_sync
        for mod, mode in modes.items():
            mod.training = mode
