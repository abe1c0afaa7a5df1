#!/usr/bin/env python
"""Headline benchmark: train utterances/sec of the GRUDecoder + CTC step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|fp32] [--dump-outputs DIR]

One "step" = noise augmentation (trainer:194-201) -> forward -> out_lens -> log-softmax + CTC -> backward -> (gradient all-reduce) -> Adam step on one
synthetic batch of the competition shape (256 features, 24 days, 41 classes; B=64 per GPU, T=500), i.e.
neural_decoder_trainer.py:208-218, 242, 251-260.  Workload = BASELINE.json configs[1]: bidirectional 5x1024
GRUDecoder, dropout 0.4, batch-sharded data parallel (weak scaling: 64 utterances per GPU).

Our arm prints one JSON line with
  value         utt/s, inputs resident in HBM, CUDA events, max over ranks
  e2e           utt/s through the public API with HOST (pinned) inputs: H2D copies (BatchPrefetcher) + a D2H read of the step's loss every step
                (LossReader: the read waits for the forward's loss, not for the backward behind it); wall clock between two barriers, K steps,
                measured 3 times back to back -- the fastest is reported, every sample is in the line
  roofline      the dominant kernel (K2 GEMM, tensor-bound): algorithmic FLOP / CUDA-event time measured in the timed region
  cpu_baseline  the torch-operator port of the reference (oracle/torch_port.py) on this box's host cores (rank 0, N=1)
``--impl reference`` times the reference's CPU path alone on the FULL batch: the reference's own ``GRUDecoder`` module,
byte-compiled from /root/reference into oracle/_ref by oracle/build_ref.py ("kind": "reference"), or -- when oracle/_ref has
not been built -- the torch-operator port oracle/torch_port.py ("kind": "port"); the trainer's loss / Adam lines are
restated in oracle/torch_port.py:train_step in both cases.  ``--impl reference-cuda`` (secondary, never the headline
ratio) runs the same reference module on the GPU (cuDNN GRU, fp32/TF32 and bf16 autocast): the "beat-this" bar of SURVEY 2a.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "train utterances/sec (GRUDecoder, B=64, T=500)"      # BASELINE.json's metric; metric_name() restates B and T when they are overridden


def metric_name(a):
    return METRIC if (a.batch == 64 and a.T == 500) else f"train utterances/sec (GRUDecoder, B={a.batch}, T={a.T})"
UNIT = "utterances/s"
E2E_REPEATS = 3                                                # samples of the host-timed end-to-end region (K steps each)
NOISE = dict(white_noise_sd=0.8, constant_offset_sd=0.2)     # scripts/train_model.py:17-18 (whiteNoiseSD, constantOffsetSD)
K1_SAVED_TENSORS = 2          # [B,T,N] f32 tensors K1's forward writes for its own backward (ys, z)
MODEL_KW = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, dropout=0.4, strideLen=4,
                kernelLen=32, gaussianSmoothWidth=2.0)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--precision", default=os.environ.get("NSD_PRECISION", "bf16"), choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--T", type=int, default=500)
    ap.add_argument("--uni", action="store_true", help="unidirectional GRU (class default) instead of the training default")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--strong", action="store_true", help="strong scaling: --batch is the GLOBAL batch, split evenly over the GPUs (default: weak, --batch per GPU)")
    ap.add_argument("--nccl-ctas", type=int, default=int(os.environ.get("NSD_NCCL_CTAS", "0")),
                    help="N > 1 GPUs: cap NCCL at this many CTAs (NCCL_MAX_CTAS) and keep as many SMs free of the persistent GEMMs during the backward; 0 = off")
    ap.add_argument("--graph", action="store_true", help="--mode conformer: replay the whole training step as one captured CUDA graph (GraphedConformerStep)")
    ap.add_argument("--tail-ctas", type=int, default=int(os.environ.get("NSD_TAIL_CTAS", "0")),
                    help="N > 1 GPUs: cap NCCL at this many CTAs and let ONLY the layer-0 dgrad GEMM leave as many SMs free, so the last (226 MB) "
                         "bucket's all-reduce runs under it; 0 = off")
    ap.add_argument("--timeline", default="", help="N > 1: write rank 0's per-bucket all-reduce timeline of one step (ready / done times relative to the start of the backward) to this JSON file")
    ap.add_argument("--breakdown", action="store_true", help="also print a per-entry-point time table to stderr")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="train step of --impl ours: after the timed steps, write what the last of them computed to DIR/<name>.npy (float32): "
                         "the loss it returned, and per parameter the values it left and the gradient it computed (see dump_outputs)")
    ap.add_argument("--mode", default="train", choices=["train", "infer", "stream", "conformer"],
                    help="infer: BASELINE configs[3] -- unidirectional GRUDecoder forward + greedy CTC decode latency at B=1 and B=32; "
                         "stream: the same model fed 4 bins (80 ms) at a time through StreamingDecoder")
    return ap.parse_args()


def baseline_config_name(a):
    """Which BASELINE.json configs[] entry the flags select."""
    if a.T == 500 and a.batch == 64 and not a.strong:
        return "BASELINE configs[0] (class default: unidirectional)" if a.uni else "BASELINE configs[1]"
    if a.T == 2000 and a.batch == 256:
        return "BASELINE configs[4] (long-sequence sweep)"
    return "non-BASELINE shape"


def config_dict(a, n_gpus, impl_note=""):
    bi = not a.uni
    return {"workload": f"GRUDecoder {'bi' if bi else 'uni'}directional 5x1024, 256 feats, 24 days, k32/s4, 41 classes, "
                        f"dropout 0.4, white noise 0.8 + constant offset 0.2; train step augment+fwd+CTC+bwd+Adam; B={a.batch}/GPU T={a.T} ({baseline_config_name(a)})",
            "global_batch": a.batch * n_gpus, "T": a.T, "frames": (a.T - 32) // 4 + 1,
            "parallelism": f"dp{n_gpus}" if n_gpus > 1 else "single",
            "l2": "working set (0.54 GB weights + >1 GB activations per step) far exceeds the 126 MB L2; no flush needed"}


# ----------------------------------------------------------------------------------------------------------
# CPU baseline: the torch-operator port of the reference on the host cores
# ----------------------------------------------------------------------------------------------------------
def reference_model(a, device="cpu"):
    """(module, kind): the reference's own GRUDecoder from oracle/_ref ("reference"), else the torch-operator port ("port")."""
    import torch
    from oracle import torch_port as P
    from oracle.build_ref import load_reference_decoder
    torch.manual_seed(0)
    Ref = load_reference_decoder()
    if Ref is not None:
        return Ref(device=device, bidirectional=not a.uni, **MODEL_KW), "reference"
    return P.PortGRUDecoder(bidirectional=not a.uni, **MODEL_KW), "port"


def cpu_reference_run(a, steps, warmup, budget_s=200.0):
    """Reference train step on the host cores, FULL batch (same config as our arm), all host threads.  The number of timed
    steps is bounded so the whole run stays within ``budget_s``; the batch is never reduced."""
    import torch
    from oracle import torch_port as P
    from neural_speech_decoder_b200.synthetic import make_batch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    m, kind = reference_model(a)
    m.train()
    opt = P.make_adam(m)
    batch = make_batch(a.batch, a.T, seed=1)
    t0 = time.perf_counter()
    P.train_step(m, opt, *batch, **NOISE)                     # first step: also the probe that sizes the run
    t_first = time.perf_counter() - t0
    warm = max(0, min(warmup - 1, int(budget_s * 0.25 / max(t_first, 1e-3))))
    for _ in range(warm):
        P.train_step(m, opt, *batch, **NOISE)
    n = max(1, min(steps, int((budget_s - (warm + 1) * t_first) / max(t_first, 1e-3))))
    times = []
    for _ in range(n):
        t0 = time.perf_counter()
        P.train_step(m, opt, *batch, **NOISE)
        times.append(time.perf_counter() - t0)
    t_step = sum(times) / len(times)
    sample = (f"full batch B={a.batch} T={a.T} per step, {len(times)} timed steps after {warm + 1} warm-up, torch {cores} threads"
              + ("" if len(times) == steps else f" (bounded from {steps} steps to stay under {budget_s:.0f} s)"))
    return a.batch / t_step, cores, t_step, kind, sample, len(times), warm + 1


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    val, cores, t_step, kind, sample, n_timed, n_warm = cpu_reference_run(a, a.steps, a.warmup)
    line = {"metric": metric_name(a), "value": round(val, 3), "unit": UNIT, "n_gpus": a.gpus, "steps": n_timed, "warmup": n_warm,
            "ms_per_step": round(t_step * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference", "config": config_dict(a, a.gpus),
            "cpu_baseline": {"value": round(val, 3), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": round(val, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_reference_cuda(a):
    """SECONDARY line (SURVEY 2a "beat-this" bar): the unmodified reference module on the GPU -- torch + cuDNN GRU + cuBLAS,
    none of this repo's kernels -- for the same train step.  Never the headline ratio."""
    import torch
    from oracle import torch_port as P
    from neural_speech_decoder_b200.synthetic import make_batch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    for mode in ("fp32 (cudnn.allow_tf32 default)", "bf16 autocast"):
        m, kind = reference_model(a, device="cuda")
        m = m.to(dev).train()
        opt = P.make_adam(m)
        batch = [t.to(dev) for t in make_batch(a.batch, a.T, seed=1)]

        def step():
            if mode.startswith("bf16"):
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    return P.train_step(m, opt, *batch, **NOISE)
            return P.train_step(m, opt, *batch, **NOISE)

        for _ in range(max(a.warmup, 3)):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            loss = step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.steps
        print(json.dumps({"metric": metric_name(a), "value": round(a.batch / (ms * 1e-3), 2), "unit": UNIT, "n_gpus": 1, "steps": a.steps,
                          "warmup": max(a.warmup, 3), "ms_per_step": round(ms, 3), "higher_is_better": True, "impl": "reference-cuda",
                          "kind": kind, "dtype": mode, "data": "synthetic", "config": config_dict(a, 1), "loss": float(loss),
                          "note": "secondary: reference module on the GPU through torch/cuDNN/cuBLAS (no repo kernels); not the headline ratio"}),
              flush=True)
        del m, opt


# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([c.strip() for c in ln.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        hot = [v for v in sm if v >= 0.5 * (mx or 1)] or sm
        return {"sm_mhz": hot[len(hot) // 2] if hot else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def gemm_flops_per_step(a, frames):
    """Algorithmic FLOPs of the K2 launches of one train step (fwd + dgrad + wgrad of the time-batched W_ih
    projections and the output layer, plus the time-batched W_hh wgrad); DESIGN.md section 'K2'."""
    D = 1 if a.uni else 2
    H, L, C, F0 = 1024, 5, 41, 256 * 32
    M = a.batch * frames
    fl = 0
    for l in range(L):
        in_l = F0 if l == 0 else H * D
        fl += 3 * 2 * M * (3 * H) * in_l * D                  # fwd, dgrad, wgrad of W_ih (both directions)
        fl += 2 * (M - a.batch) * (3 * H) * H * D             # W_hh wgrad (time-batched)
    fl += 3 * 2 * M * C * H * D                               # output layer fwd, dgrad, wgrad
    return fl


DUMP_SAMPLE = 1 << 16          # entries --dump-outputs keeps of a tensor (all of a smaller one): 18 MB for the benchmark's model


def dump_outputs(d, loss, model):
    """What the last timed train step computed, as ``d/<name>.npy`` in float32: ``loss`` (the value train_step returned) and, for
    every parameter, ``param.<name>`` (its values after the step's optimizer update) and ``grad.<name>`` (the step's gradient).
    A tensor of more than DUMP_SAMPLE entries is sampled at DUMP_SAMPLE sorted flat indices drawn from a generator seeded with
    the parameter's name and size: the same indices in every run, so that two builds can be compared file by file."""
    import zlib
    import numpy as np
    import torch
    os.makedirs(d, exist_ok=True)
    out = {"loss": loss.detach().reshape(1)}
    for name, p in model.named_parameters():
        for tag, t in (("param", p), ("grad", p.grad)):
            if t is None:
                continue
            flat = t.detach().reshape(-1)
            if flat.numel() > DUMP_SAMPLE:
                rng = np.random.default_rng([zlib.crc32(name.encode()), flat.numel()])
                idx = np.sort(rng.choice(flat.numel(), DUMP_SAMPLE, replace=False))
                flat = flat[torch.from_numpy(idx).to(flat.device)]
            out[f"{tag}.{name}"] = flat
    for k, v in out.items():
        np.save(os.path.join(d, k + ".npy"), v.float().cpu().numpy())


def run_ours(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (ours): no CUDA device -- this package has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if a.nccl_ctas > 0 or a.tail_ctas > 0:
            os.environ["NCCL_MAX_CTAS"] = str(a.nccl_ctas or a.tail_ctas)
        dist.init_process_group("nccl", device_id=dev)
    if a.strong:
        if a.batch % world:
            raise SystemExit(f"--strong: global batch {a.batch} is not divisible by {world} GPUs")
        a.batch //= world                                  # per-GPU share of the fixed global batch
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200 import _lib
    from neural_speech_decoder_b200.parallel import GradSync
    from neural_speech_decoder_b200.synthetic import make_batch

    nsd.set_default_precision(a.precision)
    torch.manual_seed(0)
    model = nsd.GRUDecoder(device="cuda", bidirectional=not a.uni, **MODEL_KW).to(dev)
    model.train()
    gs = GradSync(world, reserve_sms=a.nccl_ctas, tail_sms=a.tail_ctas) if world > 1 else None
    opt, sched = nsd.make_optimizer(model, dict(lrStart=0.02, lrEnd=0.02, nBatch=10000, l2_decay=1e-5))
    if gs is not None:
        opt.grad_scale = gs.grad_scale
        for p in model.parameters():                       # identical start on every rank
            dist.broadcast(p.data, 0)
        model.invalidate_weight_copies()                    # .data writes are invisible to autograd's version counters
    host = [t.pin_memory() for t in make_batch(a.batch, a.T, seed=1 + rank)]
    devb = [t.to(dev) for t in host]
    frames = (a.T - 32) // 4 + 1

    def step_resident():
        return nsd.train_step(model, opt, *devb, scheduler=sched, grad_sync=gs, **NOISE)

    def host_batches():                                     # every step copies its own inputs from pinned host memory
        while True:
            yield host

    feed = nsd.BatchPrefetcher(host_batches(), dev)         # the copy of step i+1 runs under the kernels of step i

    reader = nsd.LossReader(dev)                            # the step's loss lands in pinned host memory as soon as the forward has produced it

    def step_e2e():
        b = next(feed)
        nsd.train_step(model, opt, *b, scheduler=sched, grad_sync=gs, loss_reader=reader, **NOISE)
        return reader.item()                                # D2H read of this step's loss, every step (4 bytes)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(a.warmup, 3)):
        step_resident()
    barrier()
    # ---- timed region 1: device-resident inputs.  EXACTLY K steps between two barriers, nothing but the product's own launches in the
    # stream: CUDA events between kernels (the per-entry-point timers below) would break the programmatic-dependent-launch adjacency the
    # step relies on (the optimizer of a finished bucket runs UNDER the next BPTT kernel only if it is the launch right behind it).
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.lib().nsd_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps):
        loss = step_resident()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = (_lib.lib().nsd_launch_count() - l0) // a.steps
    if a.dump_outputs and rank == 0:                       # before the passes below move the parameters on
        dump_outputs(a.dump_outputs, loss, model)
    # ---- instrumented pass (roofline): the same K steps again with CUDA events around every entry point of interest, the optimizer in
    # its classic place after the backward, so that every kernel's time is its own (no overlap).  Not part of `value`.
    os.environ["NSD_STEP_IN_BACKWARD"], sib = "0", os.environ.get("NSD_STEP_IN_BACKWARD")
    _lib.profile_begin({"nsd_gemm_bf16", "nsd_gemm_bf16_x2", "nsd_gemm_f32", "nsd_adam_step", "nsd_frontend_fwd", "nsd_frontend_bwd",
                        "nsd_gru_fwd_bf16", "nsd_gru_bwd_bf16"})
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    p0.record()
    for _ in range(a.steps):
        step_resident()
    p1.record()
    barrier()
    prof_ms = p0.elapsed_time(p1)                            # duration of the instrumented pass (denominator of share_of_step)
    prof = _lib.profile_end()
    if sib is None:
        del os.environ["NSD_STEP_IN_BACKWARD"]
    else:
        os.environ["NSD_STEP_IN_BACKWARD"] = sib
    clocks = sampler.stop() if rank == 0 else None
    # ---- timed region 2: host inputs through the public API
    # The host is in this loop (wall clock, a read-back every step), so a single scheduling hiccup of the box's CPU moves a 10-step sample
    # by 10-20 %: the region is measured E2E_REPEATS times back to back (K steps each, max over ranks each) and the fastest is reported;
    # every sample is kept in the line (e2e.samples_ms_per_step).
    step_e2e()
    e2e_samples = []
    for _ in range(E2E_REPEATS):
        barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            lv = step_e2e()
        barrier()
        e2e_samples.append((time.perf_counter() - t0) * 1e3)
    tt = torch.tensor([ms] + e2e_samples, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms, e2e_samples = tt.tolist()[0], tt.tolist()[1:]
    e2e_ms = min(e2e_samples)
    if a.timeline and gs is not None:
        gs.timeline = []
        step_resident()
        torch.cuda.synchronize()
        buckets, t_end = gs.timeline_ms()
        gs.timeline = None
        if rank == 0:
            names = ["fc_decoder_out"] + [f"gru layer {l}" for l in range(4, -1, -1)] + ["dayWeights/dayBias"]
            json.dump({"n_gpus": world, "note": "one training step, rank 0; ms relative to the start of loss.backward(); ready = the bucket's last wgrad GEMM has been "
                       "enqueued on the compute stream and reached, done = its NCCL all-reduce has finished; compute_stream_past_last_wait = when the optimizer may start",
                       "ms_per_step": round(ms / a.steps, 3),
                       "buckets": [{"bucket": names[i] if i < len(names) else str(i), "MB": round(b / 1e6, 1), "ready_ms": round(r, 3), "done_ms": round(d, 3),
                                    "allreduce_ms": round(d - r, 3)} for i, (b, r, d) in enumerate(buckets)],
                       "compute_stream_past_last_wait_ms": round(t_end, 3)}, open(a.timeline, "w"), indent=1)
    if a.breakdown and rank == 0:
        os.environ["NSD_STEP_IN_BACKWARD"], sib = "0", os.environ.get("NSD_STEP_IN_BACKWARD")     # every kernel's time its own (see above)
        _lib.profile_begin(None)
        step_resident()
        torch.cuda.synchronize()
        if sib is None:
            del os.environ["NSD_STEP_IN_BACKWARD"]
        else:
            os.environ["NSD_STEP_IN_BACKWARD"] = sib
        for k, (n, t) in sorted(_lib.profile_end().items(), key=lambda kv: -kv[1][1]):
            print(f"  {k:28s} calls {n:5d}  {t:9.3f} ms", file=sys.stderr)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = a.batch * world * a.steps / (ms * 1e-3)
    e2e = a.batch * world * a.steps / (e2e_ms * 1e-3)
    gemm_calls = sum(n for k, (n, _) in prof.items() if k.startswith("nsd_gemm"))
    gemm_ms = sum(t for k, (_, t) in prof.items() if k.startswith("nsd_gemm"))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    ach = gemm_flops_per_step(a, frames) * a.steps / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
    traffic, traffic_note = None, "no ncu capture found under profiles/"
    try:
        cands = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_gemm_traffic.json"))
        tj = json.load(open(os.path.join(ROOT, "profiles", cands[-1])))
        traffic = tj["dram_bytes"]
        traffic_note = (f"ncu --set full, {tj['launch']}: dram read+write {tj['dram_bytes'] / 1e6:.0f} MB vs "
                        f"{tj['algorithmic_bytes'] / 1e6:.0f} MB algorithmic operand+result bytes of that launch")
    except Exception:
        pass
    roofline = {"kernel": "K2 time-batched GEMMs (nsd_gemm_%s)" % a.precision, "bound": "tensor",
                "achieved": round(ach, 2) if ach else None, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": round(ach / peak_tf, 4) if ach else None, "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained",
                "launches_per_step": gemm_calls // max(1, a.steps), "share_of_step": round(gemm_ms / prof_ms, 4),
                "timing": "CUDA events around every nsd_gemm_bf16* call in a second, instrumented pass over the same K steps "
                          f"({prof_ms / a.steps:.3f} ms per step with the events in the stream and the optimizer after the backward); "
                          "the value region carries no events"}
    if ach and peaks.get("bf16_tflops"):       # the GEMMs run at ~1/3 duty inside the step: the burst figure is the stricter denominator, quoted beside it
        roofline["peak_burst"] = peaks["bf16_tflops"]
        roofline["frac_vs_burst"] = round(ach / peaks["bf16_tflops"], 4)
    # the other kernels of the step against their own bounds (DESIGN.md section 4)
    hbm = peaks.get("hbm_gbs", 6650.0)
    others = []
    n_upd = sum(p.numel() for p in model.parameters() if p.grad is not None)
    if "nsd_adam_step" in prof:
        t_ms = prof["nsd_adam_step"][1] / a.steps
        gbs = n_upd * (30 if a.precision == "bf16" else 28) / (t_ms * 1e-3) / 1e9
        others.append({"kernel": "Adam (nsd_adam_step)", "bound": "hbm", "achieved": round(gbs, 1), "peak": hbm, "unit": "GB/s",
                       "frac": round(gbs / hbm, 4), "ms_per_step": round(t_ms, 3), "bytes_per_param": 30 if a.precision == "bf16" else 28})
    esz = 2 if a.precision == "bf16" else 4
    if "nsd_frontend_fwd" in prof:
        # SURVEY 8d: algorithmic bytes per utterance = read X (T*N*4) + write patches (T'*N*K*e); what the kernel saves for its
        # own backward is its choice and is listed as extra traffic, not counted as achieved bandwidth
        t_ms = prof["nsd_frontend_fwd"][1] / a.steps
        byt = a.batch * (a.T * 256 * 4 + frames * 8192 * esz)
        gbs = byt / (t_ms * 1e-3) / 1e9
        others.append({"kernel": "K1 front end forward (nsd_frontend_fwd)", "bound": "hbm", "achieved": round(gbs, 1), "peak": hbm, "unit": "GB/s",
                       "frac": round(gbs / hbm, 4), "ms_per_step": round(t_ms, 3), "algorithmic_bytes": byt,
                       "extra_bytes_saved_for_backward": a.batch * K1_SAVED_TENSORS * a.T * 256 * 4})
    if "nsd_frontend_bwd" in prof:
        t_ms = prof["nsd_frontend_bwd"][1] / a.steps
        byt = a.batch * frames * 8192 * esz                   # read dPatches (the dW/db outputs are 6.3 MB, L2-sized)
        gbs = byt / (t_ms * 1e-3) / 1e9
        others.append({"kernel": "K1 front end backward (nsd_frontend_bwd)", "bound": "hbm", "achieved": round(gbs, 1), "peak": hbm, "unit": "GB/s",
                       "frac": round(gbs / hbm, 4), "ms_per_step": round(t_ms, 3), "algorithmic_bytes": byt})
    for k, nm in (("nsd_gru_fwd_bf16", "K3 recurrence forward"), ("nsd_gru_bwd_bf16", "K3 recurrence BPTT")):
        if k in prof:
            t_ms = prof[k][1] / a.steps
            others.append({"kernel": nm, "bound": "latency", "us_per_timestep": round(t_ms * 1e3 / (5 * frames), 3), "ms_per_step": round(t_ms, 3),
                           "note": "both directions, all batch groups; 5 layers x %d sequential timesteps" % frames})
    h2d = sum(t.numel() * t.element_size() for t in host)
    line = {"metric": metric_name(a), "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": round(ms / a.steps, 3), "higher_is_better": True, "scaling": "strong" if a.strong else "weak", "vs_baseline": None,
            "dtype": a.precision, "data": "synthetic", "config": config_dict(a, world), "clocks": clocks,
            "e2e": {"value": round(e2e, 2), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "samples_ms_per_step": [round(x / a.steps, 3) for x in e2e_samples], "reported": "fastest of the samples"},
            "gpu_launches": int(launches), "roofline": roofline, "rooflines_other": others, "loss": float(lv)}
    if world == 1 and not a.no_cpu_baseline:
        val, cores, t_step, kind, sample, _, _ = cpu_reference_run(a, 3, 1, budget_s=30.0)     # same protocol as --impl reference, bounded to ~30 s
        line["cpu_baseline"] = {"value": round(val, 3), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_infer(a):
    """BASELINE configs[3]: unidirectional GRUDecoder inference, batch 1 and batch 32, T=500 bins (10 s of 20 ms bins):
    eval-mode forward -> log-softmax -> greedy CTC decode on the device, host inputs, decoded ids read back.  Secondary
    lines (not the headline contract): latency per call, per output frame (4 bins) and per 20 ms bin."""
    import torch
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200.synthetic import make_batch
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    frames = (a.T - 32) // 4 + 1
    for precision in ("bf16", "fp32"):
        nsd.set_default_precision(precision)
        torch.manual_seed(0)
        model = nsd.GRUDecoder(device="cuda", bidirectional=False, **{**MODEL_KW, "dropout": 0.0}).to(dev).eval()
        for B in (1, 32):
            X, y, X_len, y_len, day = [t.pin_memory() for t in make_batch(B, a.T, seed=2)]

            @torch.no_grad()
            def call():
                x, xl, dd = X.to(dev, non_blocking=True), X_len.to(dev, non_blocking=True), day.to(dev, non_blocking=True)
                logits = model.forward(x, dd)
                lens = nsd.out_lens(xl, model.kernelLen, model.strideLen)
                dec, dec_len = nsd.greedy_decode(nsd.ctc.log_softmax_tbc(logits), lens)
                return dec.cpu(), dec_len.cpu()

            for _ in range(max(a.warmup, 3)):
                call()
            torch.cuda.synchronize()
            ts = []
            for _ in range(a.steps):
                t0 = time.perf_counter()
                call()
                ts.append(time.perf_counter() - t0)
            ts.sort()
            med = ts[len(ts) // 2]
            print(json.dumps({"metric": "inference latency, unidirectional GRUDecoder + greedy CTC decode (host in, decoded ids out)",
                              "batch": B, "T_bins": a.T, "frames": frames, "dtype": precision, "ms_per_call": round(med * 1e3, 3),
                              "us_per_output_frame": round(med * 1e6 / frames, 2), "us_per_20ms_bin": round(med * 1e6 / a.T, 2),
                              "utterances_per_s": round(B / med, 1), "calls": a.steps, "impl": "ours", "data": "synthetic"}), flush=True)
    nsd.set_default_precision("bf16")
    if not a.no_cpu_baseline:
        cpu_infer_reference(a, frames)


def cpu_infer_reference(a, frames):
    """The reference's eval lines on the host cores for the same inference call (trainer:299-320: forward -> log_softmax ->
    per-utterance argmax / unique_consecutive / drop blank), unidirectional model, B=1 and B=32."""
    import torch
    from neural_speech_decoder_b200.synthetic import make_batch
    a.uni = True
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    m, kind = reference_model(a)
    m.eval()
    for B in (1, 32):
        X, y, X_len, y_len, day = make_batch(B, a.T, seed=2)

        @torch.no_grad()
        def call():
            pred = m.forward(X, day)                                                         # trainer:299
            lens = ((X_len - m.kernelLen) / m.strideLen).to(torch.int32)                     # trainer:300
            pred = pred.log_softmax(2)
            out = []
            for i in range(pred.shape[0]):                                                   # trainer:313-320
                d = torch.argmax(pred[i, 0:int(lens[i]), :], dim=-1)
                d = torch.unique_consecutive(d, dim=-1).numpy()
                out.append(d[d != 0])
            return out

        call()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        med = sorted(ts)[1]
        print(json.dumps({"metric": "inference latency, unidirectional GRUDecoder + greedy CTC decode (host in, decoded ids out)",
                          "batch": B, "T_bins": a.T, "frames": frames, "dtype": "f32", "ms_per_call": round(med * 1e3, 3),
                          "us_per_output_frame": round(med * 1e6 / frames, 2), "us_per_20ms_bin": round(med * 1e6 / a.T, 2),
                          "utterances_per_s": round(B / med, 1), "calls": 3, "impl": "reference", "kind": kind, "cores": cores,
                          "data": "synthetic"}), flush=True)


def run_stream(a):
    """BASELINE configs[3], streaming form: 4 new 20 ms bins per call (one output frame), host bins in, argmax id out.
    Reported per call = per 80 ms of signal; per-bin = /4.  Real-time factor = 80 ms / latency."""
    import torch
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200.synthetic import make_batch
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    nsd.set_default_precision("bf16")
    torch.manual_seed(0)
    model = nsd.GRUDecoder(device="cuda", bidirectional=False, **{**MODEL_KW, "dropout": 0.0}).to(dev).eval()
    for B in (1, 8, 32):
        X, y, X_len, y_len, day = make_batch(B, a.T, seed=2)
        X = X.pin_memory()
        sd = nsd.StreamingDecoder(model, B, day)
        lat, dev_us = [], []
        for rep in range(2):                                    # first pass warms up (and captures the graph)
            sd.reset()
            lat = []
            for pos in range(0, a.T, 4):
                t0 = time.perf_counter()
                ids = sd.push_decode(X[:, pos:pos + 4])         # pinned host bins in -> greedy ids on the host (synchronises)
                if ids is None:
                    torch.cuda.synchronize()
                lat.append(time.perf_counter() - t0)
            sd.finish()
        if sd.fast and sd._graph is not None:                   # device time of one replay (the push kernel + the two read-backs)
            sd.reset()
            for pos in range(0, a.T, 4):
                steady = sd._steady
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                if steady:
                    sd._bins_in.copy_(X[:, pos:pos + 4], non_blocking=True)
                    e0.record(); sd._graph.replay(); e1.record()
                    sd.n_bins += 4; sd.next_frame += 1
                    torch.cuda.synchronize()
                    dev_us.append(e0.elapsed_time(e1) * 1e3)
                else:
                    sd.push(X[:, pos:pos + 4])
            sd.finish()
        steady = sorted(lat[len(lat) // 4:])
        med, p99 = steady[len(steady) // 2], steady[int(len(steady) * 0.99) - 1]
        line = {"metric": "streaming inference latency per 4-bin (80 ms) push, unidirectional GRUDecoder, greedy id out",
                "batch": B, "dtype": "bf16", "us_per_push_median": round(med * 1e6, 1), "us_per_push_p99": round(p99 * 1e6, 1),
                "us_per_20ms_bin": round(med * 1e6 / 4, 1), "real_time_factor": round(0.080 / med, 1),
                "lookahead_bins": 10, "pushes": len(steady), "impl": "ours", "data": "synthetic",
                "protocol": "pinned host bins -> H2D -> push -> greedy ids D2H -> stream synchronise, wall clock per push",
                "form": ("nsd_stream_push: one launch per push (front end + 5-layer stack + logits + argmax), CUDA graph replay"
                         if (sd.fast and sd._graph is not None) else
                         "nsd_stream_push: one launch per push" if sd.fast else "time-batched kernels (exact form)")}
        if dev_us:
            dev_us.sort()
            line["device_us_per_push_median"] = round(dev_us[len(dev_us) // 2], 1)
            line["weights_streamed_mb_per_push"] = round(sum(w.numel() * 2 for w in sd._w_ih + sd._w_hh) / 1e6, 1)
            line["weight_stream_gbps"] = round(line["weights_streamed_mb_per_push"] * 1e-3 / (line["device_us_per_push_median"] * 1e-6), 0)
        print(json.dumps(line), flush=True)


def _conformer_batch(a, seed=1):
    import torch
    g = torch.Generator().manual_seed(seed)
    B, T = a.batch, a.T
    X = torch.randn(B, T, 256, generator=g)
    day = torch.randint(0, 24, (B,), generator=g)
    X_len = torch.full((B,), T, dtype=torch.int32)
    y_len = torch.randint(10, 50, (B,), generator=g).to(torch.int32)
    y = torch.zeros(B, int(y_len.max()), dtype=torch.int32)
    for b in range(B):
        y[b, :y_len[b]] = torch.randint(1, 41, (int(y_len[b]),), generator=g).to(torch.int32)
    return X, y, X_len, y_len, day


CONFORMER_TRAIN = dict(lr=4e-4, eps=1e-6, weight_decay=1e-3, label_smoothing=0.1, interctc_weight=0.3, max_norm=1.0)   # scripts/train_conformer.py


def _conformer_port_step_fn(a, device, autocast_bf16=False):
    """The reference's Conformer train step restated over torch operators (oracle/conformer_port.py; regularisers are the identity
    there) + torch.optim.AdamW + clip_grad_norm_ (trainer:144-151, 255-259) on ``device``."""
    import torch
    import neural_speech_decoder_b200 as nsd
    from oracle import conformer_port as CP
    torch.manual_seed(0)
    shell = nsd.NeuralTransformerCTCModel(n_channels=256, n_classes=41, n_days=24, device="cpu")      # parameter container only (same init as the reference)
    sd = {k: v.detach().clone().to(device) for k, v in shell.state_dict().items()}
    params = {k: sd[k].requires_grad_(True) for k, _ in shell.named_parameters()}
    opt = torch.optim.AdamW(list(params.values()), lr=CONFORMER_TRAIN["lr"], betas=(0.9, 0.999), eps=CONFORMER_TRAIN["eps"], weight_decay=CONFORMER_TRAIN["weight_decay"])
    X, y, X_len, y_len, day = [t.to(device) for t in _conformer_batch(a)]
    cfg = dict(n_layers=8, n_heads=8, temporal_kernel=32, temporal_stride=4, conv_kernel=31)

    def step():
        Xn = X + torch.randn(X.shape, device=device) * NOISE["white_noise_sd"] + torch.randn([X.shape[0], 1, X.shape[2]], device=device) * NOISE["constant_offset_sd"]
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16, enabled=autocast_bf16):
            lp, olen, inter = CP.forward({**sd, **params}, Xn, day, X_len, training=True, **cfg)
        loss = CP.training_loss(lp.float(), inter.float(), y, olen, y_len, label_smoothing=CONFORMER_TRAIN["label_smoothing"], interctc_weight=CONFORMER_TRAIN["interctc_weight"])
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(list(params.values()), max_norm=CONFORMER_TRAIN["max_norm"])
        opt.step()
        return loss
    return step


def run_conformer(a):
    """BASELINE configs[2]: Conformer (transformer_ctc.py) train step, synthetic B=64 T=500: our CUDA path (device-resident and
    host-in end to end), the torch-operator port on the host cores (bounded) and, with --impl reference-cuda, the port on the GPU."""
    import torch
    import neural_speech_decoder_b200 as nsd
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    metric = f"train utterances/sec (Conformer CTC 8x1024, B={a.batch}, T={a.T})"
    workload = ("NeuralTransformerCTCModel 256 feats, 24 days, d=1024, 8 blocks x 8 heads, FF 2048, conv k31, k32/s4, 41 classes, dropout 0.3, "
                "DropPath 0.1, SpecAugment, InterCTC 0.3, label smoothing 0.1; train step noise+fwd+CTC+bwd+clip+AdamW; "
                f"B={a.batch} T={a.T} (BASELINE configs[2])")
    if a.impl == "reference-cuda":
        for tag, ac in (("fp32 (TF32 allowed)", False), ("bf16 autocast", True)):
            torch.backends.cuda.matmul.allow_tf32 = True
            step = _conformer_port_step_fn(a, dev, ac)
            for _ in range(a.warmup):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                step()
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.steps
            print(json.dumps({"metric": metric, "impl": "reference-cuda", "note": "torch-operator port of the reference on the GPU (cuBLAS / SDPA-free explicit attention / torch kernels); "
                              "regularisers off in the port; the beat-this bar, never the headline ratio", "precision": tag, "value": round(a.batch / ms * 1e3, 1),
                              "unit": "utterances/s", "ms_per_step": round(ms, 3), "steps": a.steps, "warmup": a.warmup, "config": {"workload": workload}}), flush=True)
        return
    nsd.set_default_precision(a.precision)
    torch.manual_seed(0)
    model = nsd.NeuralTransformerCTCModel(n_channels=256, n_classes=41, n_days=24, device="cuda").to(dev)
    model.check_day_ids = False
    opt = nsd.FusedAdamW(model.parameters(), lr=CONFORMER_TRAIN["lr"], betas=(0.9, 0.999), eps=CONFORMER_TRAIN["eps"], weight_decay=CONFORMER_TRAIN["weight_decay"],
                         max_grad_norm=CONFORMER_TRAIN["max_norm"])
    opt.attach_shadows(model._shadows)
    host = _conformer_batch(a)
    pinned = [t.pin_memory() for t in host]
    X, y, X_len, y_len, day = [t.to(dev) for t in host]

    graphed = None
    if a.graph:
        graphed = nsd.GraphedConformerStep(model, opt, a.batch, a.T, int(host[1].shape[1]), label_smoothing=CONFORMER_TRAIN["label_smoothing"],
                                           interctc_weight=CONFORMER_TRAIN["interctc_weight"], white_noise_sd=NOISE["white_noise_sd"],
                                           constant_offset_sd=NOISE["constant_offset_sd"], base_lr=CONFORMER_TRAIN["lr"], warmup_steps=1000, total_steps=15000)

    def step(batch, i):
        if graphed is not None:
            return graphed.step(*batch)
        return nsd.conformer_train_step(model, opt, *batch, label_smoothing=CONFORMER_TRAIN["label_smoothing"], interctc_weight=CONFORMER_TRAIN["interctc_weight"],
                                        white_noise_sd=NOISE["white_noise_sd"], constant_offset_sd=NOISE["constant_offset_sd"], noise_seed=1000 + i)
    for i in range(a.warmup):
        step((X, y, X_len, y_len, day), i)
    torch.cuda.synchronize()
    clocks = ClockSampler(0); clocks.start()
    n0 = nsd.lib().nsd_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(a.steps):
        loss = step((X, y, X_len, y_len, day), a.warmup + i)
    e1.record()
    host_ms = (time.perf_counter() - t0) * 1e3 / a.steps       # host time to enqueue the steps (before the synchronisation)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    launches = graphed.kernels_per_replay if graphed is not None else (nsd.lib().nsd_launch_count() - n0) // a.steps
    # end to end: pinned host batch -> H2D -> step -> loss read back, every step
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(a.steps):
        batch = [t.to(dev, non_blocking=True) for t in pinned]
        lv = step(batch, 2 * a.warmup + a.steps + i).item()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / a.steps
    ck = clocks.stop()
    line = {"metric": metric, "value": round(a.batch / ms * 1e3, 1), "unit": "utterances/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(ms, 3),
            "host_enqueue_ms_per_step": round(host_ms, 3), "higher_is_better": True, "dtype": a.precision, "data": "synthetic", "config": {"workload": workload},
            "clocks": ck, "e2e": {"value": round(a.batch / e2e_ms * 1e3, 1), "unit": "utterances/s", "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in pinned)),
                                  "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches), "loss": round(float(lv), 5), "impl": "ours",
            "form": "one captured CUDA graph per step (GraphedConformerStep)" if graphed is not None else "eager: one C-ABI call per kernel from Python autograd"}
    if a.breakdown:
        from neural_speech_decoder_b200 import _lib
        _lib.profile_begin(None)
        step((X, y, X_len, y_len, day), 9999)
        torch.cuda.synchronize()
        tot = 0.0
        for k, (n, t) in sorted(_lib.profile_end().items(), key=lambda kv: -kv[1][1]):
            print(f"  {k:28s} calls {n:5d}  {t:9.3f} ms", file=sys.stderr)
            tot += t
        print(f"  {'sum of entry points':28s}              {tot:9.3f} ms", file=sys.stderr)
    if not a.no_cpu_baseline:
        import copy
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        a2 = copy.copy(a); a2.batch = min(a.batch, 16)
        cstep = _conformer_port_step_fn(a2, torch.device("cpu"))
        cstep()
        t0 = time.perf_counter(); cstep(); dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": round(a2.batch / dt, 2), "unit": "utterances/s", "cores": cores, "kind": "port",
                                "sample": f"1 timed step (after 1 warm-up) on {a2.batch} of the {a.batch} utterances, T={a.T}, torch {cores} threads; regularisers off in the port"}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    args = parse()
    if args.dump_outputs and (args.mode != "train" or args.impl != "ours"):
        raise SystemExit("--dump-outputs: only the train step of --impl ours is dumped")
    if args.mode == "conformer":
        run_conformer(args)
    elif args.mode == "stream":
        run_stream(args)
    elif args.mode == "infer":
        run_infer(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-cuda":
        run_reference_cuda(args)
    else:
        run_ours(args)
