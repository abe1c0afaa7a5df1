"""Stateful streaming inference for the unidirectional GRUDecoder (BASELINE configs[3]; SURVEY.md section 8f rank 3).

The reference has no streaming API: ``forward`` always starts from h0 = 0 and drops the final state
(model.py:104-119).  ``StreamingDecoder`` carries the fp32 hidden state of every layer between calls and keeps the raw
bins a future frame still needs.  Two execution forms:
  * exact (any batch, any chunking): the SAME time-batched kernels fed incrementally; logits bit-identical to the offline
    forward;
  * fast (batch <= 8, steady pushes of one stride = one new frame): ONE launch of ``nsd_stream_push`` per push -- front end
    of the bins that became computable, slide of the patch row, the whole 5-layer stack, logits and greedy id -- replayed as
    a captured CUDA graph together with the read-back of the ids into pinned memory; all stream state (a ring of the last 64
    raw bins, the patch row, fp32 + bf16 hidden states, the bin counter) lives on the device, the 107 MB of bf16 weights are
    streamed once per push and stay resident in the 126 MB L2 between pushes.  Same arithmetic up to fp32 summation order
    (checked against the reference operators with carried state, tests/test_gpu_streaming.py).  Frame j covers bins [4j, 4j+32) (kernel 32 / stride 4, model.py:37-39) of the smoothed signal, and the 20-tap
Gaussian is padded 9 left / 10 right (augmentations.py:91), so frame j can be emitted once bin 4j+41 has arrived: a
fixed look-ahead of 10 bins (200 ms).  ``finish()`` flushes the frames the offline model would still produce by zero
padding past the end of the utterance, exactly as the offline smoothing does.

With ``beam_width`` set, a CTC prefix beam search (``ctc.CtcBeamSearch``, optionally with a phoneme-bigram prior) follows
the stream on the device: the exact form advances it on the logits each call returns, the fast form launches the advance
inside the captured push.  ``hypotheses()`` gives the N-best of the frames emitted so far, bit-identical to
``ctc_beam_search(is_logits=True)`` over the concatenated logits.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import _lib, ops
from ._lib import NsdError
from .ctc import CtcBeamSearch


def complete_frames(n_bins: int, kernel_len: int, stride_len: int, lookahead: int) -> int:
    """Number of output frames that can be emitted once ``n_bins`` bins have arrived: frame j reads smoothed bins
    [S*j, S*j+K) and the smoothing reads ``lookahead`` raw bins past each of them."""
    if n_bins < kernel_len + lookahead:
        return 0
    return (n_bins - kernel_len - lookahead) // stride_len + 1


def window_for(j0: int, stride_len: int, halo: int):
    """(first raw bin, number of leading frames to discard) of the window that recomputes frames from j0 on with
    ``halo`` bins (a multiple of the stride, >= the smoothing's left reach) of true history in front."""
    r0 = max(0, stride_len * j0 - halo)
    return r0, (stride_len * j0 - r0) // stride_len


class StreamingDecoder:
    def __init__(self, model, batch_size: int, dayIdx: torch.Tensor, fast: Optional[bool] = None, use_graph: bool = True,
                 beam_width: Optional[int] = None, nbest: int = 1, lm: Optional[torch.Tensor] = None, lm_weight: float = 0.0,
                 insertion_bonus: float = 0.0, max_frames: int = 4096):
        if model.bidirectional:
            raise NsdError("streaming needs the unidirectional GRUDecoder (the reverse direction reads the future)")
        if model.precision != "bf16":
            raise NsdError("StreamingDecoder runs the bf16 tensor-core path (set_default_precision('bf16'))")
        self.m = model
        self.B = int(batch_size)
        p = next(model.parameters())
        self.dev = p.device
        self.day = dayIdx.to(device=self.dev, dtype=torch.int64).contiguous()
        if self.day.shape != (self.B,):
            raise RuntimeError(f"dayIdx must be [{self.B}]")
        self.K, self.S, self.N = model.kernelLen, model.strideLen, model.neural_dim
        taps = model.gaussianSmoother.weight[0, 0]
        self.left = (taps.numel() - 1) // 2                     # 9
        self.right = taps.numel() - 1 - self.left               # 10
        self.halo = -(-self.left // self.S) * self.S            # left context re-read per call, a multiple of the stride (12)
        fast_ok = (self.B <= 8 and model.hidden_dim % 512 == 0 and (self.N * self.K) % 512 == 0 and self.N % 32 == 0 and model.layer_dim <= 8
                   and self.S <= 8 and self.K > self.S and taps.numel() - 1 + 2 * self.S <= self.RING
                   and self.halo + self.K + self.right + 2 * self.S <= self.RING)
        if fast and not fast_ok:
            raise NsdError("the fast streaming form needs batch <= 8, hidden size and neural_dim*kernelLen multiples of 512, neural_dim a "
                           "multiple of 32, stride <= 8, <= 8 layers")
        self.fast = fast_ok if fast is None else bool(fast)
        self.use_graph = use_graph
        self.last_ids: Optional[torch.Tensor] = None           # greedy phoneme id(s) of the last emitted frame (fast form), i32 [B] on the device
        self._graph = None
        self._beam = None
        if beam_width is not None:
            if not 1 <= int(nbest) <= int(beam_width):
                raise NsdError(f"nbest={nbest} outside [1, beam_width={beam_width}]")
            self._nbest = int(nbest)
            self._beam = CtcBeamSearch(self.B, model.fc_decoder_out.weight.shape[0], beam_width, max_frames, 0, lm, lm_weight,
                                       insertion_bonus, device=self.dev)
        self.reset()

    def hypotheses(self):
        """N-best of the frames emitted so far: (hyps i64 [B,nbest,max_frames], hyp_len i32 [B,nbest], score f32 [B,nbest],
        acoustic f32 [B,nbest]) on the device (``CtcBeamSearch.nbest``)."""
        if self._beam is None:
            raise NsdError("hypotheses() needs StreamingDecoder(..., beam_width=W)")
        return self._beam.nbest(self._nbest)

    def _emit_and_advance(self, j0: int, j1: int, r1: int) -> torch.Tensor:
        """``_emit`` and, with a beam, its advance on the returned logits; the frame budget is checked before either runs."""
        if self._beam is not None:
            self._beam.reserve(j1 - j0 + 1)
        out = self._emit(j0, j1, r1)
        if self._beam is not None:
            self._beam.enqueue(out.permute(1, 0, 2), None, True)
        return out

    def reset(self) -> None:
        m = self.m
        if getattr(self, "hs", None) is None:
            self.hs = torch.zeros(m.layer_dim, self.B, m.hidden_dim, device=self.dev)   # fp32 state of every layer, carried between calls
        else:
            self.hs.zero_()            # in place: a captured graph of the fast form holds this buffer's address
        self.hist = torch.empty(self.B, 0, self.N, device=self.dev)
        self.hist_start = 0            # absolute bin index of hist[:, 0]
        self.n_bins = 0                # bins received so far
        self.next_frame = 0            # first frame not yet emitted
        self._steady = False           # fast form engaged: the last bins live in the static window instead of ``hist``
        if self._beam is not None:
            self._beam.reset()         # in place, like ``hs``

    # ------------------------------------------------------------------------------------------------------------ fast form
    RING = 64                          # raw bins kept on the device (>= halo + K + right + S: enough to fall back to the exact form)

    def _fast_setup(self, extra: int) -> None:
        """Device state of the fast form (allocated once; ``extra`` = bins received beyond the newest frame's look-ahead,
        constant while every push is one stride long -- it is a kernel argument, so a change re-captures the graph)."""
        m, B = self.m, self.B
        if getattr(self, "_extra", None) != extra:
            self._graph = None
        self._extra = extra
        if getattr(self, "_rawring", None) is not None:
            return
        L, H, F0 = m.layer_dim, m.hidden_dim, self.N * self.K
        C = m.fc_decoder_out.weight.shape[0]
        dev = self.dev
        self._bins_in = torch.zeros(B, self.S, self.N, device=dev)
        self._rawring = torch.zeros(B, self.RING, self.N, device=dev)
        self._x0buf = torch.zeros(2, B, F0, device=dev, dtype=torch.bfloat16)
        self._nbins_dev = torch.zeros(1, device=dev, dtype=torch.int32)
        self._hbf = torch.zeros(L, B, H, device=dev, dtype=torch.bfloat16)
        self._logits = torch.zeros(B, C, device=dev)
        self.last_ids = torch.zeros(B, dtype=torch.int32, device=dev)
        self._logits_host = torch.zeros(B, C).pin_memory()
        self._ids_host = torch.zeros(B, dtype=torch.int32).pin_memory()
        nbytes = _lib.lib().nsd_stream_push_workspace(B, F0, H, L)
        self._ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        gw = m._gru_weights()
        self._w_ih = [m._shadows.stacked(("ih", l), [gw[4 * l]]) for l in range(L)]
        self._w_hh = [m._shadows.stacked(("hh", l), [gw[4 * l + 1]]) for l in range(L)]
        self._b_ih = [gw[4 * l + 2].detach().contiguous() for l in range(L)]
        self._b_hh = [gw[4 * l + 3].detach().contiguous() for l in range(L)]
        self._fc_w = m._shadows.stacked(("fc", 0), [m.fc_decoder_out.weight])
        self._fc_b = m.fc_decoder_out.bias.detach().contiguous()
        self._taps = m.gaussianSmoother.weight[0, 0].contiguous()
        self._day_w = m.dayWeights.detach().contiguous()
        self._day_b = m.dayBias.detach().contiguous()

    def refresh_weights(self) -> None:
        """Call after the model's parameters changed (optimizer step, ``load_state_dict``): the fast form holds the addresses of the
        bf16 weight copies it was set up with (and so does its captured graph); this re-derives them and drops the graph.  The per-push
        path deliberately does not check parameter versions (it would cost a tenth of the push latency)."""
        if getattr(self, "_rawring", None) is None:
            return
        m, L = self.m, self.m.layer_dim
        gw = m._gru_weights()
        self._w_ih = [m._shadows.stacked(("ih", l), [gw[4 * l]]) for l in range(L)]
        self._w_hh = [m._shadows.stacked(("hh", l), [gw[4 * l + 1]]) for l in range(L)]
        self._b_ih = [gw[4 * l + 2].detach().contiguous() for l in range(L)]
        self._b_hh = [gw[4 * l + 3].detach().contiguous() for l in range(L)]
        self._fc_w = m._shadows.stacked(("fc", 0), [m.fc_decoder_out.weight])
        self._fc_b = m.fc_decoder_out.bias.detach().contiguous()
        self._day_w = m.dayWeights.detach().contiguous()
        self._day_b = m.dayBias.detach().contiguous()
        self._graph = None

    def _fast_state(self):
        st = [self.hs, self._hbf, self._rawring, self._x0buf, self._nbins_dev]
        return st if self._beam is None else st + [self._beam.state, self._beam.err_flag]

    def _fast_launch(self) -> None:
        """One launch for the whole push + the read-back of logits and greedy ids into pinned host memory: the unit that is
        captured as a CUDA graph."""
        ops.stream_push(self._bins_in, self._rawring, self.day, self._day_w, self._day_b, self._taps, self._x0buf, self._nbins_dev,
                        self._extra, self.K, self.S, self._w_ih, self._w_hh, self._b_ih, self._b_hh, self.hs, self._hbf, self._fc_w,
                        self._fc_b, self._logits, self.last_ids, self.m._err_flag, self._ws)
        if self._beam is not None:         # T = 1 frame of logits, log-softmaxed inside the beam kernel
            self._beam.enqueue(self._logits.unsqueeze(0), None, True)
        self._ids_host.copy_(self.last_ids, non_blocking=True)
        self._logits_host.copy_(self._logits, non_blocking=True)

    def _fast_step(self, bins: torch.Tensor) -> None:
        if self._beam is not None:
            self._beam.reserve(1)
        self._bins_in.copy_(bins, non_blocking=True)               # pinned host (fastest), pageable host or device source
        if self.use_graph and self._graph is None:
            snap = [t.clone() for t in self._fast_state()]
            try:                                               # warm up on a side stream, then capture (torch's capture protocol)
                side = torch.cuda.Stream(self.dev)
                side.wait_stream(torch.cuda.current_stream(self.dev))
                with torch.cuda.stream(side):
                    self._fast_launch()
                torch.cuda.current_stream(self.dev).wait_stream(side)
                for t, v in zip(self._fast_state(), snap):
                    t.copy_(v)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._fast_launch()
                self._graph = g                                # capture does not execute; the warm-up did and was undone above
            except Exception as e:                             # noqa: BLE001 -- capture unsupported: stay eager (still one launch per push)
                self._graph, self.use_graph = None, False
                self._graph_error = repr(e)
                torch.cuda.synchronize(self.dev)
                for t, v in zip(self._fast_state(), snap):
                    t.copy_(v)
        if self._graph is not None:
            self._graph.replay()
        else:
            self._fast_launch()
        self.n_bins += self.S
        self.next_frame += 1

    def _enter_fast(self, j: int) -> None:
        """Engage the fast form after frame j went through the exact form: ring <- the last raw bins, patch row of frame j,
        bf16 copy of the carried states, stream position."""
        n, R = self.n_bins, self.RING
        self._fast_setup(n - (self.S * j + self.K + self.right))
        self._ring_from = max(self.hist_start, n - R)              # oldest bin the ring really holds
        a = torch.arange(self._ring_from, n, device=self.dev)
        self._rawring.zero_()
        self._rawring[:, a % R] = self.hist[:, a - self.hist_start]
        self._x0buf[j & 1].copy_(self._last_patch)
        self._hbf.copy_(self.hs)
        self._nbins_dev.fill_(n)
        self._steady = True
        self.hist = None

    def _leave_fast(self) -> None:
        n, R = self.n_bins, self.RING
        self.hist_start = max(self._ring_from, n - R)
        a = torch.arange(self.hist_start, n, device=self.dev)
        self.hist = self._rawring[:, a % R].contiguous()
        self._steady = False

    @torch.no_grad()
    def push_decode(self, bins: torch.Tensor) -> Optional[torch.Tensor]:
        """``push`` + greedy phoneme ids on the host: int32 CPU tensor [B, f] for the f frames that became complete (None if
        f == 0).  In the steady fast form this is the low-latency call: one graph replay (H2D of the bins is enqueued in front
        of it, the ids come back through pinned memory), one stream synchronisation.  The returned tensor is reused by the
        next call."""
        if self._steady and bins.dim() == 3 and bins.shape == (self.B, self.S, self.N):
            with torch.cuda.device(self.dev):
                self._fast_step(bins)
                torch.cuda.current_stream(self.dev).synchronize()
            return self._ids_host.unsqueeze(1)
        out = self.push(bins)
        return None if out is None else out.argmax(-1).to(torch.int32).cpu()

    # ------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def _emit(self, j0: int, j1: int, r1: int) -> torch.Tensor:
        """Frames j0..j1 (inclusive) from bins [r0, r1): r0 re-reads ``halo`` bins of left context so that the frames
        we keep see the true smoothing history; frames computed from the window's padded edges are discarded."""
        m, B, K, S = self.m, self.B, self.K, self.S
        r0, skip = window_for(j0, S, self.halo)
        x = self.hist[:, r0 - self.hist_start:r1 - self.hist_start].contiguous()
        k = j1 - j0 + 1
        taps = m.gaussianSmoother.weight[0, 0].contiguous()
        patches, _, _ = ops.frontend_fwd(x, self.day, m.dayWeights.detach().contiguous(), m.dayBias.detach().contiguous(), taps,
                                         K, S, torch.bfloat16, m._err_flag if m._err_flag is not None else None)
        inp = patches[skip * B:(skip + k) * B]                  # time-major rows: a contiguous block of frames
        self._last_patch = patches[(skip + k - 1) * B:(skip + k) * B]   # bf16 [B, N*K]: the fast form slides it from here on
        H, L = m.hidden_dim, m.layer_dim
        M = k * B
        gw = m._gru_weights()
        for l in range(L):
            w_ih, w_hh, b_ih, b_hh = gw[4 * l:4 * l + 4]
            w_ih_bf = m._shadows.stacked(("ih", l), [w_ih])
            w_hh_bf = m._shadows.stacked(("hh", l), [w_hh])
            gi = torch.empty((M, 3 * H), device=self.dev, dtype=torch.float32)
            in_l = inp.shape[1]
            ops.gemm(False, True, M, 3 * H, in_l, inp, in_l, w_ih_bf, in_l, gi, 3 * H, bias=b_ih.detach().contiguous())
            hseq, hseq_bf, _ = ops.gru_fwd_bf16(gi, w_hh_bf, b_hh.detach().contiguous(), k, B, H, 1, False, False, h0=self.hs[l])
            self.hs[l].copy_(hseq[(k - 1) * B:])                # fp32 state carried to the next call
            inp = hseq_bf
        fc = m.fc_decoder_out
        C = fc.weight.shape[0]
        fc_bf = m._shadows.stacked(("fc", 0), [fc.weight])
        logits_tm = torch.empty((M, C), device=self.dev, dtype=torch.float32)
        ops.gemm(False, True, M, C, H, inp, H, fc_bf, H, logits_tm, C, bias=fc.bias.detach().contiguous())
        return ops.swap01(logits_tm.view(k, B, C))

    def _trim(self) -> None:
        keep_from = max(0, self.S * self.next_frame - self.halo)
        if keep_from > self.hist_start:
            self.hist = self.hist[:, keep_from - self.hist_start:].contiguous()
            self.hist_start = keep_from

    @torch.no_grad()
    def push(self, bins: torch.Tensor) -> Optional[torch.Tensor]:
        """bins [B, n, N] (n >= 0 new 20 ms bins) -> logits [B, f, C] of the f frames that became complete (None if f == 0)."""
        if bins.dim() != 3 or bins.shape[0] != self.B or bins.shape[2] != self.N:
            raise RuntimeError(f"bins must be [{self.B}, n, {self.N}], got {tuple(bins.shape)}")
        if self.m._err_flag is None:
            self.m._err_flag = torch.zeros(1, dtype=torch.int32, device=self.dev)
        if self._steady:
            if bins.shape[1] == self.S:
                with torch.cuda.device(self.dev):
                    self._fast_step(bins)
                    return self._logits.clone().unsqueeze(1)
            self._leave_fast()
        self.hist = torch.cat([self.hist, bins.to(self.dev, torch.float32)], dim=1)
        self.n_bins += bins.shape[1]
        # frame j needs smoothed bins up to S*j+K-1, i.e. raw bins up to S*j+K-1+right
        j1 = complete_frames(self.n_bins, self.K, self.S, self.right) - 1
        if j1 < self.next_frame:
            return None
        with torch.cuda.device(self.dev):
            out = self._emit_and_advance(self.next_frame, j1, self.S * j1 + self.K + self.right)
            if self.fast and bins.shape[1] == self.S and j1 == self.next_frame and self.S * j1 >= self.halo:
                # steady streaming: one stride per push, one new frame per push -> the single-launch push from here on
                self.next_frame = j1 + 1
                self._trim()
                self._enter_fast(j1)
                self.last_ids.copy_(out[:, -1].argmax(-1))
                return out
        self.next_frame = j1 + 1
        self._trim()
        return out

    @torch.no_grad()
    def finish(self) -> Optional[torch.Tensor]:
        """End of utterance: the frames the offline forward still produces (it zero-pads the smoothing past the last bin)."""
        if self._steady:
            self._leave_fast()
        if self.n_bins < self.K:
            if self.next_frame == 0 and self.n_bins > 0:
                raise RuntimeError(f"utterance shorter than kernelLen={self.K} bins")     # the reference raises too (nn.Unfold)
            return None
        j1 = (self.n_bins - self.K) // self.S
        if j1 < self.next_frame:
            return None
        with torch.cuda.device(self.dev):
            out = self._emit_and_advance(self.next_frame, j1, self.n_bins)
        self.next_frame = j1 + 1
        self._trim()
        return out


INT_MAX = 2 ** 31 - 1


class StreamingSessions:
    """Independent streaming sessions on one GPU: ``slots`` (<= 8) batch rows, each with its own utterance clock, recording
    day, carried state and beam.  Sessions start (``open``), push one stride of bins at a time while active, pause (inactive
    pushes leave every byte of a slot's state as it is) and end (``finish``) independently; a freed slot takes the next
    utterance.  Every push is one launch of ``nsd_stream_push_slots`` (the single-launch push of ``StreamingDecoder``'s fast
    form with a counter, an active flag and a last frame per slot), replayed as a CUDA graph with the beam advance and the
    read-back of the greedy ids.  There is no exact form: the warm-up before a session's first frame runs inside the kernel.

    A session's logits are the same bits whatever the slot count, the other sessions and when the session started -- the
    bits of the utterance streamed alone through ``StreamingSessions(model, 1)`` -- and agree with the offline forward up to
    fp32 summation order.  Frame j is emitted by the push that brings the session to S*j + K + right bins (right = the
    smoothing's look-ahead, 10 bins for the 20 taps of augmentations.py:91); ``finish`` flushes the frames the offline forward
    still produces by zero padding past the end of the utterance.  The weights are read at construction."""

    RING = StreamingDecoder.RING

    def __init__(self, model, slots: int, *, beam_width: Optional[int] = None, nbest: int = 1, lm: Optional[torch.Tensor] = None,
                 lm_weight: float = 0.0, insertion_bonus: float = 0.0, max_frames: int = 4096, use_graph: bool = True):
        if model.bidirectional:
            raise NsdError("streaming needs the unidirectional GRUDecoder (the reverse direction reads the future)")
        if model.precision != "bf16":
            raise NsdError("StreamingSessions runs the bf16 tensor-core path (set_default_precision('bf16'))")
        B = int(slots)
        self.K, self.S, self.N = model.kernelLen, model.strideLen, model.neural_dim
        taps = model.gaussianSmoother.weight[0, 0]
        ntaps = taps.numel()
        self.right = ntaps - 1 - (ntaps - 1) // 2
        L, H, F0 = model.layer_dim, model.hidden_dim, self.N * self.K
        if not (1 <= B <= 8 and H % 512 == 0 and F0 % 512 == 0 and self.N % 32 == 0 and L <= 8 and self.S <= 8 and self.K > self.S
                and ntaps <= 32 and ntaps - 1 + 2 * self.S <= self.RING):
            raise NsdError("StreamingSessions needs 1..8 slots, hidden size and neural_dim*kernelLen multiples of 512, neural_dim a "
                           "multiple of 32, stride <= 8 and < kernelLen, <= 8 layers, <= 32 smoothing taps")
        if int(max_frames) < 1:
            raise NsdError(f"max_frames={max_frames} must be positive")
        self.m, self.slots, self.max_frames, self.use_graph = model, B, int(max_frames), use_graph
        dev = self.dev = next(model.parameters()).device
        C = self.C = model.fc_decoder_out.weight.shape[0]
        i32 = dict(device=dev, dtype=torch.int32)
        # per-slot state: open() writes a slot's h, counter, last frame and day; the kernel never reads a ring row or a patch row
        # the slot's current utterance has not written, so those need no clearing
        self._bins_in = torch.zeros(B, self.S, self.N, device=dev)
        self._rawring = torch.empty(B, self.RING, self.N, device=dev)
        self._x0buf = torch.empty(2, B, F0, device=dev, dtype=torch.bfloat16)
        self._h = torch.empty(L, B, H, device=dev)
        self._hbf = torch.empty(L, B, H, device=dev, dtype=torch.bfloat16)
        self._day = torch.empty(B, device=dev, dtype=torch.int64)
        self._n_bins = torch.zeros(B, **i32)
        self._last = torch.full((B,), INT_MAX, **i32)
        self._active = torch.zeros(B, **i32)
        self._emitted = torch.zeros(B, **i32)
        self._logits = torch.empty(B, C, device=dev)
        self._ids = torch.empty(B, **i32)
        self._active_host = torch.zeros(B, dtype=torch.int32).pin_memory()
        self._ids_host = torch.zeros(B, dtype=torch.int32).pin_memory()
        self._ws = torch.empty(_lib.lib().nsd_stream_push_workspace(B, F0, H, L), device=dev, dtype=torch.uint8)
        gw = model._gru_weights()
        self._w_ih = [model._shadows.stacked(("ih", l), [gw[4 * l]]) for l in range(L)]
        self._w_hh = [model._shadows.stacked(("hh", l), [gw[4 * l + 1]]) for l in range(L)]
        self._b_ih = [gw[4 * l + 2].detach().contiguous() for l in range(L)]
        self._b_hh = [gw[4 * l + 3].detach().contiguous() for l in range(L)]
        self._fc_w = model._shadows.stacked(("fc", 0), [model.fc_decoder_out.weight])
        self._fc_b = model.fc_decoder_out.bias.detach().contiguous()
        self._taps = taps.detach().contiguous()
        self._day_w = model.dayWeights.detach().contiguous()
        self._day_b = model.dayBias.detach().contiguous()
        if model._err_flag is None:
            model._err_flag = torch.zeros(1, **i32)
        self._beam = None
        if beam_width is not None:
            if not 1 <= int(nbest) <= int(beam_width):
                raise NsdError(f"nbest={nbest} outside [1, beam_width={beam_width}]")
            self._nbest = int(nbest)
            self._beam = CtcBeamSearch(B, C, beam_width, self.max_frames, 0, lm, lm_weight, insertion_bonus, device=dev)
            self._mask = torch.zeros(B, **i32)
        self._open = [False] * B
        self._n = [0] * B              # bins of each slot's utterance, counted on the host
        self._frames = [0] * B         # frames each slot's utterance emitted
        self._graph = None

    # ------------------------------------------------------------------------------------------------------------ sessions
    def _slot(self, slot) -> int:
        s = int(slot)
        if not 0 <= s < self.slots:
            raise NsdError(f"slot {slot} outside [0, {self.slots})")
        return s

    @torch.no_grad()
    def open(self, slot: int, day: int) -> None:
        """Start a new utterance in ``slot`` (ending whatever it held) recorded on ``day``: zero state, counter 0, empty beam, in
        place in the device buffers the captured graph reads.  Other slots are untouched.  A day out of range sets the model's
        error flag at the next push, as the offline forward's front end does."""
        s = self._slot(slot)
        with torch.cuda.device(self.dev):
            self._h[:, s].zero_()
            self._hbf[:, s].zero_()
            self._n_bins[s].fill_(0)
            self._last[s].fill_(INT_MAX)
            self._day[s].fill_(int(day))
            if self._beam is not None:
                self._mask.zero_()
                self._mask[s].fill_(1)
                self._beam.reset_utterances(self._mask)
        self._open[s], self._n[s], self._frames[s] = True, 0, 0

    def _emits(self, s: int, last: int = INT_MAX) -> bool:
        """Whether the next push of slot ``s`` emits a frame (the kernel's rule, on the host counters)."""
        n = self._n[s] + self.S
        return n >= self.K + self.right and (n - self.K - self.right) // self.S <= last

    def _check_push(self, bins: torch.Tensor, active) -> List[bool]:
        if bins.dim() != 3 or tuple(bins.shape) != (self.slots, self.S, self.N):
            raise NsdError(f"bins must be [{self.slots}, {self.S}, {self.N}], got {tuple(bins.shape)}")
        act = torch.as_tensor(active)
        if tuple(act.shape) != (self.slots,) or act.is_floating_point() or act.is_complex():
            raise NsdError(f"active must be a bool or integer [{self.slots}] vector, got {act.dtype} {tuple(act.shape)}")
        act = [bool(a) for a in act.tolist()]
        for s, a in enumerate(act):
            if a and not self._open[s]:
                raise NsdError(f"slot {s} is not open")
            if a and self._emits(s) and self._frames[s] + 1 > self.max_frames:
                raise NsdError(f"slot {s}: the session would pass max_frames={self.max_frames}")
        return act

    def _commit(self, act: List[bool], last: int = INT_MAX) -> List[bool]:
        """Advance the host counters of the slots a push moved; -> which slots emitted."""
        em = [False] * self.slots
        for s, a in enumerate(act):
            if a:
                em[s] = self._emits(s, last)
                self._n[s] += self.S
                self._frames[s] += int(em[s])
        return em

    def _launch(self) -> None:
        """One push for every slot, the beam advance on the rows that emitted, the read-back of the greedy ids into pinned
        memory: the unit captured as a CUDA graph."""
        ops.stream_push_slots(self._bins_in, self._rawring, self._day, self._day_w, self._day_b, self._taps, self._x0buf, self._n_bins,
                              self._active, self._last, self._emitted, self.K, self.S, self._w_ih, self._w_hh, self._b_ih, self._b_hh,
                              self._h, self._hbf, self._fc_w, self._fc_b, self._logits, self._ids, self.m._err_flag, self._ws)
        if self._beam is not None:          # T = 1 frame; lens = emitted leaves the other utterances untouched
            self._beam.enqueue(self._logits.unsqueeze(0), self._emitted, True)
        self._ids_host.copy_(self._ids, non_blocking=True)

    def _step(self) -> None:
        if self.use_graph and self._graph is None:
            try:                            # a push with no slot active changes no state: it is the warm-up before the capture
                saved = self._active.clone()
                self._active.zero_()
                side = torch.cuda.Stream(self.dev)
                side.wait_stream(torch.cuda.current_stream(self.dev))
                with torch.cuda.stream(side):
                    self._launch()
                torch.cuda.current_stream(self.dev).wait_stream(side)
                self._active.copy_(saved)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._launch()
                self._graph = g
            except Exception as e:          # noqa: BLE001 -- capture unsupported: stay eager (still one launch per push)
                self._graph, self.use_graph = None, False
                self._graph_error = repr(e)
                torch.cuda.synchronize(self.dev)
                self._active.copy_(saved)
        if self._graph is not None:
            self._graph.replay()
        else:
            self._launch()

    @torch.no_grad()
    def push(self, bins: torch.Tensor, active):
        """bins [slots, S, N] (row s: the next S bins of slot s's session), active [slots] (bool or int) -> (logits f32
        [slots, C], emitted bool [slots]) on the device; rows of the slots that did not emit hold no new frame."""
        act = self._check_push(bins, active)
        with torch.cuda.device(self.dev):
            self._bins_in.copy_(bins, non_blocking=True)
            self._active.copy_(torch.tensor(act, dtype=torch.int32), non_blocking=True)
            self._step()
            self._commit(act)
            return self._logits.clone(), self._emitted != 0

    @torch.no_grad()
    def push_decode(self, bins: torch.Tensor, active) -> torch.Tensor:
        """``push`` that returns greedy phoneme ids on the host: int32 CPU tensor [slots], -1 for the slots that emitted no
        frame.  The low-latency call: the bins (pinned host memory is fastest) and the active flags go up in front of one graph
        replay, the ids come back through pinned memory, one stream synchronisation.  The returned tensor is reused."""
        act = self._check_push(bins, active)
        with torch.cuda.device(self.dev):
            self._bins_in.copy_(bins, non_blocking=True)
            self._active_host.copy_(torch.tensor(act, dtype=torch.int32))
            self._active.copy_(self._active_host, non_blocking=True)
            self._step()
            torch.cuda.current_stream(self.dev).synchronize()
        self._commit(act)
        return self._ids_host

    @torch.no_grad()
    def finish(self, slot: int, tail: torch.Tensor) -> torch.Tensor:
        """End slot ``slot``'s utterance with its last ``tail`` [r, N] bins (r >= 0) -> logits [f, C] of every frame the offline
        forward of the whole utterance produces beyond those already emitted (frames j <= (n_total - K) // S): the tail and then
        zero bins, exactly the offline zero padding, are pushed with the slot's last frame set.  The slot is closed; its
        hypotheses stay readable until it is opened again."""
        s = self._slot(slot)
        if not self._open[s]:
            raise NsdError(f"slot {s} is not open")
        if tail.dim() != 2 or tail.shape[1] != self.N:
            raise NsdError(f"tail must be [r, {self.N}], got {tuple(tail.shape)}")
        r, K, S = tail.shape[0], self.K, self.S
        n_total = self._n[s] + r
        if n_total < K:
            self._open[s] = False
            raise RuntimeError(f"utterance shorter than kernelLen={K} bins")     # the reference raises too (nn.Unfold)
        last = (n_total - K) // S
        f = last + 1 - self._frames[s]
        if self._frames[s] + f > self.max_frames:
            raise NsdError(f"slot {s}: the session would pass max_frames={self.max_frames}")
        outs = []
        if f > 0:
            pushes = max(-(-r // S), -(-(S * last + K + self.right - self._n[s]) // S))
            pad = torch.zeros(pushes * S, self.N, device=self.dev)
            pad[:r] = tail
            act = [i == s for i in range(self.slots)]
            with torch.cuda.device(self.dev):
                self._last[s].fill_(last)
                self._active.copy_(torch.tensor(act, dtype=torch.int32), non_blocking=True)
                for i in range(pushes):
                    self._bins_in[s].copy_(pad[i * S:(i + 1) * S])
                    self._step()
                    if self._commit(act, last)[s]:
                        outs.append(self._logits[s].clone())
        self._open[s] = False
        return torch.stack(outs) if outs else torch.zeros(0, self.C, device=self.dev)

    def hypotheses(self, slot: int):
        """N-best of slot ``slot``'s session so far: (hyps i64 [nbest, max_frames], hyp_len i32 [nbest], score f32 [nbest],
        acoustic f32 [nbest]) on the device (``CtcBeamSearch.nbest``)."""
        s = self._slot(slot)
        if self._beam is None:
            raise NsdError("hypotheses() needs StreamingSessions(..., beam_width=W)")
        hyps, hyp_len, score, acoustic = self._beam.nbest(self._nbest)
        return hyps[s], hyp_len[s], score[s], acoustic[s]
