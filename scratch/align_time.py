"""K5c forced alignment timing: one JSON line per measurement, GPU name and power limit first.

``ctc_forced_align`` on logits (``is_logits=True``) at B=64/T'=118/C=41 with targets padded to 60 and to 500, and at B=256/T'=493
padded to 500 (target lengths up to ~160); both with ``check=True`` (the default: one flag read, a host synchronisation) and
``check=False`` (launch only, the graph-capturable form).  Beside them ``ctc_loss_from_logits`` (K4) at the same shapes, with the
gradient (the training step's form) and without.  CUDA events around ``--reps`` calls, median of 3 such windows after ``--warmup``
calls.  Last, the loop users run today: one ``torchaudio.functional.forced_align`` per utterance with a ``.cpu()`` of its result
(on the GPU if this torchaudio build runs there, else on the CPU from log-probs already copied to the host; the line says which),
timed with a host clock over one batch.

    python scratch/align_time.py [--reps 20] [--warmup 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neural_speech_decoder_b200 as nsd  # noqa: E402
from neural_speech_decoder_b200.ctc import ctc_forced_align, log_softmax_tbc  # noqa: E402


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def inputs(T, B, C, Smax, lo, hi, seed=0):
    """Logits [B,T,C] (the GRU's layout) shaped like a trained decoder's, ragged lengths, targets [B,Smax] with lengths in [lo, hi]."""
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(B, T, C, generator=g) * 6.0
    logits[:, :, 0] += 2.0
    lens = torch.randint(T // 2, T + 1, (B,), generator=g)
    lens[0] = T
    tl = torch.minimum(torch.randint(lo, hi + 1, (B,), generator=g), lens // 3)
    tgt = torch.randint(1, C, (B, Smax), generator=g, dtype=torch.int32)
    return logits.cuda(), lens.cuda(), tgt.cuda(), tl.cuda()


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


def torchaudio_loop(logits, lens, tgt, tl):
    import torchaudio.functional as F
    lp = log_softmax_tbc(logits)                                       # [T,B,C]
    B = lp.shape[1]
    dev = "cuda"
    try:
        F.forced_align(lp[:, 0].unsqueeze(0).contiguous(), tgt[:1, :int(tl[0])], lens[:1], tl[:1], blank=0)
        torch.cuda.synchronize()
    except Exception as e:                                             # no kernel for this GPU in the build
        dev = f"cpu ({type(e).__name__}: {str(e).splitlines()[0][:80]})"
    lens_h, tl_h = lens.cpu().tolist(), tl.cpu().tolist()
    if dev == "cuda":
        src, tg = lp, tgt
    else:
        src, tg = lp.cpu(), tgt.cpu()

    def run():
        for b in range(B):
            il, L = lens_h[b], tl_h[b]
            if L == 0:
                continue
            lab, sc = F.forced_align(src[:il, b].unsqueeze(0).contiguous(), tg[b:b + 1, :L], torch.tensor([il], device=src.device),
                                     torch.tensor([L], device=src.device), blank=0)
            lab.cpu(), sc.cpu()
    run()
    ms = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run()
        torch.cuda.synchronize()
        ms.append((time.perf_counter() - t0) * 1e3)
    return sorted(ms)[1], max(ms) - min(ms), dev


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    print(json.dumps(gpu_line()), flush=True)
    C = 41
    for B, T, Smax, lo, hi in ((64, 118, 60, 20, 60), (64, 118, 500, 20, 60), (256, 493, 500, 80, 200)):
        logits, lens, tgt, tl = inputs(T, B, C, Smax, lo, hi)
        shape = {"B": B, "T": T, "C": C, "max_tgt": Smax, "max_tgt_len": int(tl.max())}
        tbc = logits.permute(1, 0, 2)
        for check in (True, False):
            ms, spread = time_call(lambda: ctc_forced_align(tbc, tgt, lens, tl, is_logits=True, check=check), a.reps, a.warmup)
            print(json.dumps({"what": "ctc_forced_align", **shape, "check": check, "ms_per_call": round(ms, 4),
                              "spread_ms": round(spread, 4)}), flush=True)
        for grad in (True, False):
            x = logits.detach().requires_grad_(grad)
            ms, spread = time_call(lambda: nsd.ctc_loss_from_logits(x, tgt, lens, tl), a.reps, a.warmup)
            print(json.dumps({"what": "ctc_loss_from_logits", **shape, "grad": grad, "ms_per_call": round(ms, 4),
                              "spread_ms": round(spread, 4)}), flush=True)
        if Smax == 60 or B == 256:
            ms, spread, dev = torchaudio_loop(logits, lens, tgt, tl)
            print(json.dumps({"what": "torchaudio.forced_align per utterance + .cpu()", **shape, "device": dev, "ms_per_batch": round(ms, 3),
                              "spread_ms": round(spread, 3)}), flush=True)


if __name__ == "__main__":
    main()
