"""Input-gradient timing: one JSON line per measurement, GPU name and power limit first.  B=64, T=500, N=256, K=32, S=4, the
bidirectional 5x1024 GRUDecoder in bf16.

  (a) nsd_frontend_bwd_input alone (bf16 and f32 dpatches) beside nsd_frontend_bwd at the same shape: CUDA events around --reps
      launches, median of 3 windows; achieved GB/s over the bytes it must move (dpatches + z read, dx written) against the 6,544.7 GB/s
      copy peak.  The 190 MB working set is larger than the 126 MB L2, so consecutive launches do not run from L2.
  (b) the model's backward (loss.backward() after a forward, CUDA events around the backward only): every parameter trainable and X
      without grad, against frozen parameters with X.requires_grad.
  (c) input_attribution(..., "integrated_gradients", steps=32) over the B=64 batch (2,048 utterance forward+backward passes in batches
      of 256), host clock around the call ending in a synchronise: utterance-steps per second.

    python scratch/attrib_time.py [--reps 20] [--warmup 3] [--out FILE]
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
from neural_speech_decoder_b200 import ops  # noqa: E402
from neural_speech_decoder_b200.synthetic import fill_trained_like_, make_batch  # noqa: E402

COPY_PEAK_GBS = 6544.7
COMP = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, dropout=0.0, strideLen=4, kernelLen=32,
            gaussianSmoothWidth=2.0, bidirectional=True)


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def time_call(fn, reps, warmup):
    """Median over 3 windows of the CUDA-event time per call, ms."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    samples = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        samples.append(e0.elapsed_time(e1) / reps)
    return sorted(samples)[1], samples


def kernel_lines(reps, warmup):
    B, T, N, K, S = 64, 500, 256, 32, 4
    Tp = (T - K) // S + 1
    g = torch.Generator().manual_seed(0)
    z = torch.tanh(torch.randn(B, T, N, generator=g)).cuda()
    ys = torch.randn(B, T, N, generator=g).cuda()
    day = torch.randint(0, 24, (B,), generator=g).cuda()
    W = (torch.randn(24, N, N, generator=g) / 16).cuda()
    taps = nsd.model.gaussian_kernel_1d(20, 2.0).cuda()
    out = []
    for dt in (torch.bfloat16, torch.float32):
        dp = torch.randn(Tp * B, N * K, generator=g).to(dt).cuda()
        nbytes = dp.numel() * dp.element_size() + 2 * z.numel() * 4
        ms, samples = time_call(lambda: ops.frontend_bwd_input(dp, z, day, W, taps, K, S), reps, warmup)
        gbs = nbytes / ms / 1e6
        out.append(dict(what="nsd_frontend_bwd_input", dpatches=str(dt).split(".")[-1], B=B, T=T, N=N, K=K, S=S, ms=ms, windows_ms=samples,
                        bytes=nbytes, achieved_GBs=gbs, hbm_bound_ms=nbytes / COPY_PEAK_GBS / 1e6, share_of_copy_peak=gbs / COPY_PEAK_GBS))
        ms, samples = time_call(lambda: ops.frontend_bwd(dp, ys, z, day, 24, K, S), reps, warmup)
        out.append(dict(what="nsd_frontend_bwd", dpatches=str(dt).split(".")[-1], B=B, T=T, N=N, K=K, S=S, ms=ms, windows_ms=samples))
    return out


def model_and_batch():
    nsd.set_default_precision("bf16")
    try:
        torch.manual_seed(0)
        m = nsd.GRUDecoder(device="cuda", **COMP)
    finally:
        nsd.set_default_precision("fp32")
    fill_trained_like_(m, seed=7)
    m = m.cuda().eval()
    batch = [t.cuda() for t in make_batch(64, 500, seed=11, ragged=True)]
    return m, batch


def backward_lines(m, batch, reps, warmup):
    X, y, X_len, y_len, day = batch
    lens = nsd.out_lens(X_len, m.kernelLen, m.strideLen)
    out = []
    for frozen in (False, True):
        m.requires_grad_(not frozen)
        times = []
        for i in range(warmup + reps):
            m.zero_grad(set_to_none=True)
            Xi = X.clone().requires_grad_(frozen)
            loss = nsd.ctc_loss_from_logits(m(Xi, day), y, lens, y_len)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss.backward()
            e1.record()
            e1.synchronize()
            if i >= warmup:
                times.append(e0.elapsed_time(e1))
        times.sort()
        out.append(dict(what="model_backward", params="frozen, X.requires_grad" if frozen else "trainable, X without grad",
                        median_ms=times[len(times) // 2], min_ms=times[0], max_ms=times[-1], reps=reps))
    m.requires_grad_(True)
    return out


def ig_line(m, batch, steps=32, max_batch=256, reps=3):
    X, y, X_len, y_len, day = batch
    nsd.input_attribution(m, X, y, X_len, y_len, day, method="integrated_gradients", steps=steps, max_batch=max_batch)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        nsd.input_attribution(m, X, y, X_len, y_len, day, method="integrated_gradients", steps=steps, max_batch=max_batch)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    t = sorted(times)[len(times) // 2]
    return dict(what="input_attribution", method="integrated_gradients", steps=steps, B=X.shape[0], max_batch=max_batch, median_s=t,
                all_s=times, utterance_steps_per_s=steps * X.shape[0] / t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attrib_time.py measures on the GPU; no CUDA device found")
    lines = [gpu_line()] + kernel_lines(a.reps, a.warmup)
    m, batch = model_and_batch()
    lines += backward_lines(m, batch, a.reps, a.warmup)
    lines.append(ig_line(m, batch))
    lines.append(gpu_line())
    text = "\n".join(json.dumps(x) for x in lines) + "\n"
    print(text, end="")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text)


if __name__ == "__main__":
    main()
