"""Where the bf16 train step issues its optimizer updates, relative to the BPTT launches.

Each in-backward update must be the launch directly behind a ``nsd_gru_bwd_bf16`` (the late-wait Adam triple
``nsd_set_adam_late_wait(1) / nsd_adam_step / nsd_set_adam_late_wait(0)``): that adjacency is what lets it run on the SMs the
recurrence leaves idle.  The tests record the library's entry points, in order, by wrapping the loaded library object.

The data-parallel case runs this file as a two-rank worker (gloo, both ranks on one GPU):
    python -m torch.distributed.run --nproc-per-node 2 tests/test_gpu_update_schedule.py
"""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

L = 3
KW = dict(neural_dim=32, n_classes=10, hidden_dim=64, layer_dim=L, nDays=4, dropout=0.3, strideLen=4, kernelLen=16,
          gaussianSmoothWidth=2.0, bidirectional=True)
LATE_ON, LATE_OFF = ("nsd_set_adam_late_wait", 1), ("nsd_set_adam_late_wait", 0)


class _Recorder:
    """Stands in for the loaded library: forwards every entry point and records (name, detail) in call order.  The detail is
    the flag of ``nsd_set_adam_late_wait`` and, for ``nsd_adam_step``, the sorted buckets ("fc", "l<layer>", "day") of the
    parameters it updates."""

    def __init__(self, lib, bucket_of_ptr):
        self._lib, self._bucket = lib, bucket_of_ptr
        self.calls = []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def rec(*args):
            detail = None
            if name == "nsd_set_adam_late_wait":
                detail = int(args[0])
            elif name == "nsd_adam_step":
                detail = tuple(sorted(self._bucket[p] for p in list(args[1])[:args[0]]))
            self.calls.append((name, detail))
            return fn(*args)
        return rec


def _bucket_of(name):
    if name.startswith("fc_decoder_out."):
        return "fc"
    if name.startswith("day"):
        return "day"
    return "l" + name.split("_l")[-1].split("_")[0]          # gru_decoder.weight_ih_l2_reverse -> l2


def _record_step(grad_sync=None, seed=0):
    """Train two steps of a bf16 model with dropout and input noise; return the calls of the second and the bucket sizes."""
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200 import _lib
    from neural_speech_decoder_b200.synthetic import fill_trained_like_, make_batch
    nsd.set_default_precision("bf16")
    try:
        torch.manual_seed(0)
        m = nsd.GRUDecoder(device="cuda", **KW)
    finally:
        nsd.set_default_precision("fp32")
    fill_trained_like_(m, seed=3)
    m = m.cuda().train()
    batch = [t.cuda() for t in make_batch(6, 90, n_feat=32, n_days=4, n_classes=10, seed=7 + seed, ragged=True, min_tgt=2,
                                          max_tgt=6, kernel_len=16, stride_len=4)]
    opt, sched = nsd.make_optimizer(m, dict(lrStart=0.02, lrEnd=0.01, nBatch=10, l2_decay=1e-5))
    trained = {n: _bucket_of(n) for n, p in m.named_parameters() if not n.startswith("inpLayer")}
    sizes = {}
    for b in trained.values():
        sizes[b] = sizes.get(b, 0) + 1
    bucket_of_ptr = {p.data_ptr(): trained[n] for n, p in m.named_parameters() if n in trained}
    nsd.train_step(m, opt, *batch, scheduler=sched, grad_sync=grad_sync, white_noise_sd=0.3)
    real = _lib.lib()
    rec = _Recorder(real, bucket_of_ptr)
    _lib._lib = rec
    try:
        nsd.train_step(m, opt, *batch, scheduler=sched, grad_sync=grad_sync, white_noise_sd=0.3)
    finally:
        _lib._lib = real
    torch.cuda.synchronize()
    return rec.calls, sizes


def _adam(sizes, *buckets):
    return "nsd_adam_step", tuple(sorted(b for b in buckets for _ in range(sizes[b])))


def _bptt_positions(calls):
    pos = [i for i, (n, _) in enumerate(calls) if n == "nsd_gru_bwd_bf16"]
    assert len(pos) == L, calls
    return pos                                              # BPTT(L-1), ..., BPTT(0)


def _after_backward(calls):
    """The calls after the front-end backward, the last kernel of the backward."""
    last = max(i for i, (n, _) in enumerate(calls) if n == "nsd_frontend_bwd")
    return calls[last + 1:]


def test_single_gpu_updates_each_bucket_behind_the_next_bptt(monkeypatch):
    monkeypatch.setenv("NSD_STEP_IN_BACKWARD", "1")
    calls, sizes = _record_step()
    pos = _bptt_positions(calls)
    behind = ["fc"] + [f"l{l + 1}" for l in range(L - 2, -1, -1)]          # fc behind BPTT(L-1), layer l+1 behind BPTT(l)
    for i, b in zip(pos, behind):
        assert calls[i + 1:i + 4] == [LATE_ON, _adam(sizes, b), LATE_OFF], (b, calls[i:i + 4])
    assert sum(c == LATE_ON for c in calls) == L
    tail = _after_backward(calls)
    assert [c for c in tail if c[0] in ("nsd_adam_step", "nsd_set_adam_late_wait")] == [_adam(sizes, "l0", "day")]


def test_classic_order_without_step_in_backward(monkeypatch):
    monkeypatch.setenv("NSD_STEP_IN_BACKWARD", "0")
    calls, sizes = _record_step()
    assert not any(n == "nsd_set_adam_late_wait" for n, _ in calls)
    assert [c for c in calls if c[0] == "nsd_adam_step"] == [_adam(sizes, *sizes)]
    assert _after_backward(calls)[-1] == _adam(sizes, *sizes)


def test_data_parallel_updates_each_bucket_one_bptt_later():
    """Two ranks share one GPU through gloo.  A bucket released in front of BPTT(l) is all-reduced under it and updated behind
    BPTT(l-1); layer 1, layer 0 and the day weights are updated after the backward."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.abspath(__file__)], capture_output=True, text=True, timeout=900,
                       env={**os.environ, "NSD_STEP_IN_BACKWARD": "1"})
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("CALLS ")]
    assert r.returncode == 0 and len(lines) == 1, r.stdout[-3000:] + r.stderr[-3000:]
    ranks = json.loads(lines[0][len("CALLS "):])
    assert len(ranks) == 2
    for rank, (calls, sizes) in enumerate(ranks):
        calls = [(n, tuple(d) if isinstance(d, list) else d) for n, d in calls]
        pos = _bptt_positions(calls)
        assert calls[pos[0] + 1][0] not in ("nsd_set_adam_late_wait", "nsd_adam_step"), (rank, calls[pos[0]:pos[0] + 4])
        behind = ["fc"] + [f"l{l + 2}" for l in range(L - 3, -1, -1)]       # fc behind BPTT(L-2), layer l+1 behind BPTT(l-1)
        for i, b in zip(pos[1:], behind):
            assert calls[i + 1:i + 4] == [LATE_ON, _adam(sizes, b), LATE_OFF], (rank, b, calls[i:i + 4])
        assert sum(c == LATE_ON for c in calls) == L - 1, rank
        tail = [c for c in _after_backward(calls) if c[0] in ("nsd_adam_step", "nsd_set_adam_late_wait")]
        assert all(n == "nsd_adam_step" for n, _ in tail), (rank, tail)
        assert sorted(b for _, d in tail for b in d) == sorted(_adam(sizes, "l1", "l0", "day")[1]), (rank, tail)


def _worker():
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    from neural_speech_decoder_b200.parallel import GradSync
    every = [None] * world
    dist.all_gather_object(every, _record_step(GradSync(world), seed=rank))
    if rank == 0:
        print("CALLS " + json.dumps(every), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    _worker()
