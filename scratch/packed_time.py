"""Cost of packed-sequence semantics on the benchmark shape (bf16, bidirectional 5 x 1024, B = 64, T = 500, ragged batch).

  (a) train_step with packed=False and packed=True, alternated step by step, each step timed with CUDA events around it (the
      step ends in a device synchronise); median and spread of --steps steps each after --warmup of each.
  (b) K3 alone: nsd_gru_fwd_bf16 and nsd_gru_bwd_bf16 of one layer (both directions), with and without frame counts, CUDA
      events around --reps launches.
The card's name and power limit are read in the same run and written beside the numbers, one JSON line per measurement.
Usage: python scratch/packed_time.py --out profiles/packed_time.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import neural_speech_decoder_b200 as nsd  # noqa: E402
from neural_speech_decoder_b200 import ops, trainer  # noqa: E402
from neural_speech_decoder_b200.synthetic import fill_trained_like_, make_batch  # noqa: E402

COMP = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, dropout=0.4, strideLen=4, kernelLen=32,
            gaussianSmoothWidth=2.0, bidirectional=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2]
    return dict(gpu=name, power_limit=power)


def stats(ms):
    ms = np.asarray(ms)
    return dict(median_ms=float(np.median(ms)), p10_ms=float(np.percentile(ms, 10)), p90_ms=float(np.percentile(ms, 90)), n=len(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/packed_time.jsonl")
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = card()
    lines = []
    torch.manual_seed(0)
    m = nsd.GRUDecoder(device="cuda", **COMP)
    fill_trained_like_(m, seed=1)
    m.precision = "bf16"
    m = m.to(dev).train()
    opt, sched = trainer.make_optimizer(m, dict(lrStart=0.02, lrEnd=0.02, nBatch=10 ** 6, l2_decay=1e-5))
    B, T = 64, 500
    X, y, X_len, y_len, day = (t.to(dev) for t in make_batch(B, T, seed=3, ragged=True))
    times = {False: [], True: []}
    for i in range(2 * (a.warmup + a.steps)):
        packed = bool(i % 2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        trainer.train_step(m, opt, X, y, X_len, y_len, day, scheduler=sched, white_noise_sd=0.8, constant_offset_sd=0.2, packed=packed)
        e1.record()
        torch.cuda.synchronize()
        if i >= 2 * a.warmup:
            times[packed].append(e0.elapsed_time(e1))
    for packed in (False, True):
        lines.append(dict(what="train_step", packed=packed, B=B, T=T, arch="bi 5x1024 bf16, dropout 0.4, noise", **stats(times[packed]), **info))
    # (b) one layer of K3 alone
    H, D = 1024, 2
    Tp = (T - 32) // 4 + 1
    g = torch.Generator(device=dev).manual_seed(5)
    gi = torch.randn((Tp * B, D * 3 * H), device=dev, generator=g) * 0.5
    w = (torch.randn((D * 3 * H, H), device=dev, generator=g) / 32).bfloat16()
    wT = torch.stack([w[d * 3 * H:(d + 1) * 3 * H].t() for d in range(D)]).reshape(D * H, 3 * H).contiguous()
    b_hh = torch.zeros(D * 3 * H, device=dev)
    nf = ops.frame_counts(X_len.to(torch.int64).contiguous(), T, 32, 4)
    dh = torch.randn((Tp * B, D * H), device=dev, generator=g)
    for packed in (False, True):
        kw = dict(n_frames=nf) if packed else {}
        for what in ("gru_fwd_bf16", "gru_bwd_bf16"):
            hseq, _, saves = ops.gru_fwd_bf16(gi, w, b_hh, Tp, B, H, D, False, True, **kw)
            run = (lambda: ops.gru_fwd_bf16(gi, w, b_hh, Tp, B, H, D, False, True, **kw)) if what == "gru_fwd_bf16" else \
                  (lambda: ops.gru_bwd_bf16(dh, hseq, saves, wT, Tp, B, H, D, False, **kw))
            for _ in range(3):
                run()
            torch.cuda.synchronize()
            ms = []
            for _ in range(a.reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run()
                e1.record()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1))
            lines.append(dict(what=what, packed=packed, B=B, Tp=Tp, H=H, D=D, **stats(ms), us_per_step=float(np.median(ms)) * 1e3 / Tp, **info))
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
            print(json.dumps(ln))


if __name__ == "__main__":
    main()
