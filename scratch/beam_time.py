"""K5b prefix beam search timing: one JSON line per measurement, GPU name and power limit first.

Offline: ``ctc_beam_search`` (state set-up + advance over every frame + N-best read-out, the whole call) at B=64/T'=118/C=41
for W in {1, 16, 64, 128} with the bigram prior off and on, ``greedy_decode`` at the same shape for comparison, and
B=256/T'=493 at W=16/64; CUDA events over ``--reps`` calls after ``--warmup`` calls.  Streaming: wall-clock latency per
4-bin push at B=1 with ``push_decode`` (pinned bins in, ids out, synchronised: the protocol of ``bench.py --mode stream``)
without and with ``beam_width=16``.  ``--profile-dir DIR`` also writes a torch.profiler kernel table of one W=16 call.

    python scratch/beam_time.py [--reps 50] [--warmup 10] [--profile-dir DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neural_speech_decoder_b200 as nsd  # noqa: E402
from neural_speech_decoder_b200.ctc import ctc_beam_search  # noqa: E402


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def inputs(T, B, C, seed=0):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(T, B, C, generator=g) * 6.0
    logits[:, :, 0] += 2.0
    lens = torch.randint(T // 2, T + 1, (B,), generator=g)
    lens[0] = T
    lm = torch.randn(C, C, generator=g).log_softmax(-1)
    return logits.cuda().log_softmax(-1), lens.cuda(), lm.cuda()


def time_call(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    samples = []
    for _ in range(3):
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        samples.append(e0.elapsed_time(e1) / reps)
    return sorted(samples)[1], max(samples) - min(samples)


def offline(a):
    C = 41
    for B, T, widths in ((64, 118, (1, 16, 64, 128)), (256, 493, (16, 64))):
        lp, lens, lm = inputs(T, B, C)
        ms, spread = time_call(lambda: nsd.greedy_decode(lp, lens), a.reps, a.warmup)
        print(json.dumps({"what": "greedy_decode", "B": B, "T": T, "C": C, "ms_per_call": round(ms, 4), "spread_ms": round(spread, 4)}), flush=True)
        for W in widths:
            for prior in (False, True):
                kw = dict(lm=lm, lm_weight=0.5, insertion_bonus=0.5) if prior else {}
                ms, spread = time_call(lambda: ctc_beam_search(lp, lens, W, min(4, W), **kw), a.reps, a.warmup)
                print(json.dumps({"what": "ctc_beam_search", "B": B, "T": T, "C": C, "W": W, "prior": prior, "ms_per_call": round(ms, 4),
                                  "us_per_frame": round(ms * 1e3 / T, 2), "spread_ms": round(spread, 4)}), flush=True)


def streaming(a):
    from neural_speech_decoder_b200.synthetic import make_batch
    kw = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, strideLen=4, kernelLen=32, gaussianSmoothWidth=2.0,
              dropout=0.0)
    nsd.set_default_precision("bf16")
    torch.manual_seed(0)
    model = nsd.GRUDecoder(device="cuda", bidirectional=False, **kw).cuda().eval()
    T = 2000
    X, _, _, _, day = make_batch(1, T, seed=2)
    X = X.pin_memory()
    results = {}
    for rep in range(2):                              # alternate the two forms twice; report the second round
        for beam in (None, 16):
            sd = nsd.StreamingDecoder(model, 1, day, beam_width=beam, max_frames=T // 4 + 8)
            for _ in range(2):                        # first pass warms up and captures the graph
                sd.reset()
                lat = []
                for pos in range(0, T, 4):
                    t0 = time.perf_counter()
                    ids = sd.push_decode(X[:, pos:pos + 4])
                    if ids is None:
                        torch.cuda.synchronize()
                    lat.append(time.perf_counter() - t0)
                sd.finish()
            steady = sorted(lat[len(lat) // 4:])
            results[beam] = (steady[len(steady) // 2] * 1e6, steady[int(len(steady) * 0.99) - 1] * 1e6, sd._graph is not None)
    for beam, (med, p99, graph) in results.items():
        print(json.dumps({"what": "stream push_decode", "B": 1, "beam_width": beam, "us_per_push_median": round(med, 1),
                          "us_per_push_p99": round(p99, 1), "graph": graph}), flush=True)


def profile(a):
    lp, lens, lm = inputs(118, 64, 41)
    for _ in range(3):
        ctc_beam_search(lp, lens, 16, 4, lm=lm, lm_weight=0.5, insertion_bonus=0.5)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA, torch.profiler.ProfilerActivity.CPU]) as prof:
        for _ in range(10):
            ctc_beam_search(lp, lens, 16, 4, lm=lm, lm_weight=0.5, insertion_bonus=0.5)
        torch.cuda.synchronize()
    os.makedirs(a.profile_dir, exist_ok=True)
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=20)
    with open(os.path.join(a.profile_dir, "beam_profile.txt"), "w") as f:
        f.write(json.dumps(gpu_line()) + "\n10 calls of ctc_beam_search(B=64, T'=118, C=41, W=16, nbest=4, prior on)\n" + table)
    print(table, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--profile-dir", default=None)
    ap.add_argument("--skip-stream", action="store_true")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    print(json.dumps(gpu_line()), flush=True)
    offline(a)
    if not a.skip_stream:
        streaming(a)
    if a.profile_dir:
        profile(a)


if __name__ == "__main__":
    main()
