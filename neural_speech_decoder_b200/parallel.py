"""Batch-sharded data parallelism for the training step (SURVEY.md section 8e; new work -- the reference is
single-GPU).  One process per GPU; every rank holds the full weights and a slice of the batch; the only
exchange is the gradient all-reduce, issued bucket by bucket from INSIDE the hand-written backward as each
layer's weight gradients become final, so NCCL (NVLink 5 / NVSwitch) runs under the remaining
backward-through-time.  The 1/world average is folded into the Adam kernel's ``grad_scale``.

Exactness: the reference loss is mean_b nll_b / len_b over the global batch; with equal per-rank batches,
per-rank "mean" followed by gradient averaging reproduces it exactly.
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.distributed as dist


class GradSync:
    def __init__(self, world_size: Optional[int] = None, group=None, reserve_sms: int = 0, tail_sms: int = 0):
        """``reserve_sms``: SMs the persistent GEMMs leave to NCCL between ``begin()`` and ``finish()`` (pair it with
        ``NCCL_MAX_CTAS=<reserve_sms>`` in the environment before the process group is created); 0 = share all SMs.
        ``tail_sms``: the targeted form -- only the LAST GRU bucket (layer 0: 226 MB, final when nothing but the layer-0 dgrad GEMM and
        the front-end backward are left to hide it) is released before its dgrad GEMM, and only that GEMM leaves ``tail_sms`` SMs to
        NCCL (again with ``NCCL_MAX_CTAS=<tail_sms>``); every other GEMM keeps all SMs."""
        self.group = group
        self.world = world_size if world_size is not None else (dist.get_world_size(group) if dist.is_initialized() else 1)
        self.handles: List = []
        self._storages: List = []
        self.bytes = 0
        self.reserve_sms = int(reserve_sms) if self.world > 1 else 0
        self.tail_sms = int(tail_sms) if self.world > 1 else 0
        self.timeline = None           # set to [] to record, per bucket, (bytes, ready event, done event) of the coming step (diagnostics)
        self._t0 = None

    @property
    def grad_scale(self) -> float:
        return 1.0 / self.world

    def begin(self) -> None:
        self.handles, self.bytes = [], 0
        self._storages = []            # per handle: (storage address, bytes) of the bucket -- tells which parameters' gradients it holds
        if self.timeline is not None:
            self.timeline.clear()
            self._t0 = torch.cuda.Event(enable_timing=True)
            self._t0.record()
        if self.reserve_sms:
            from ._lib import call
            call("nsd_set_gemm_sm_reserve", self.reserve_sms)

    def bucket_ready(self, flat: torch.Tensor):
        """Called by the backward with a flat buffer whose gradients are final.  The collective is enqueued on
        NCCL's own stream behind the work already queued on the current stream and overlaps what follows.
        Returns the collective's work handle (None when ``world <= 1``)."""
        if self.world <= 1:
            return None
        self.bytes += flat.numel() * flat.element_size()
        ready = None
        if self.timeline is not None:
            ready = torch.cuda.Event(enable_timing=True)
            ready.record()                                  # on the compute stream: the bucket's last wgrad has been enqueued before this point
        h = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        self.handles.append(h)
        self._storages.append((flat.untyped_storage().data_ptr(), flat.numel() * flat.element_size()))
        if self.timeline is not None:
            side = torch.cuda.Stream(flat.device)           # a stream that waits for THIS collective only: its event is the collective's end
            done = torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(side):
                h.wait()
                done.record()
            self.timeline.append((flat.numel() * flat.element_size(), ready, done))
        return h

    def finish_early(self, tail_bytes: int = 32 << 20) -> set:
        """Make the current stream wait for every collective EXCEPT the tail of the queue: the last bucket of at least
        ``tail_bytes`` (layer 0's 226 MB, final when only its dgrad GEMM and the front-end backward are left to hide it) and the
        small ones released after it.  Returns the storage addresses of the buckets still in flight, so that the caller can
        update the parameters of the finished buckets while the tail is on the wire (trainer.train_step does; measured timeline:
        profiles/r02_allreduce_timeline_2gpu.json) and then call ``finish()``.  NCCL runs the collectives of one communicator in
        order, so waiting for handle k covers every earlier one."""
        n = len(self.handles)
        cut = n
        for i in range(n - 1, -1, -1):
            cut = i
            if self._storages[i][1] >= tail_bytes:
                break
        if n == 0 or self._storages[cut][1] < tail_bytes:
            cut = n                                          # no big bucket: nothing worth deferring
        for h in self.handles[:cut]:
            h.wait()
        pending = {a for a, _ in self._storages[cut:]}
        self.handles, self._storages = self.handles[cut:], self._storages[cut:]
        return pending

    def finish(self) -> None:
        for h in self.handles:
            h.wait()                      # current stream waits for the collective; no host block on NCCL
        self.handles, self._storages = [], []
        if self.timeline is not None:
            self._t1 = torch.cuda.Event(enable_timing=True)
            self._t1.record()                               # compute stream: backward enqueued and every collective waited for
        if self.reserve_sms:
            from ._lib import call
            call("nsd_set_gemm_sm_reserve", 0)

    def timeline_ms(self):
        """After a synchronize: [(bytes, ready_ms, done_ms)] per bucket relative to begin(), and the time at which the compute stream
        got past the last wait."""
        return [(b, self._t0.elapsed_time(r), self._t0.elapsed_time(d)) for b, r, d in self.timeline], self._t0.elapsed_time(self._t1)
