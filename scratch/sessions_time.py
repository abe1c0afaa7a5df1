"""StreamingSessions timing at the competition architecture (unidirectional 5x1024, N=256, K=32, S=4): one JSON line per
measurement, GPU name and power limit first.

  * per-push latency with every slot active, at 1, 4 and 8 slots: host to host (``push_decode``: pinned bins in, ids out, one
    graph replay and one synchronisation; median and p90 over ``--pushes`` calls) and device time per replay (CUDA events
    around ``--pushes`` back-to-back replays of the captured push);
  * the same two numbers for ``StreamingDecoder``'s fast form at B = 1 and 8, measured in the same rounds, alternating;
  * a replay of ``--utts`` synthetic utterances (200..600 bins = 4..12 s) through 8 slots, each free slot taking the next
    utterance at once: pushes, wall time, utterances per second, real-time factor (wall time over audio time, 20 ms bins).

    python scratch/sessions_time.py [--out profiles/stream_sessions_time.jsonl] [--pushes 300] [--rounds 3] [--utts 240]
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
from neural_speech_decoder_b200.synthetic import fill_trained_like_  # noqa: E402

KW = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, strideLen=4, kernelLen=32, gaussianSmoothWidth=2.0)
S, N = 4, 256


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"what": "gpu", "gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


class Sessions:
    """All slots active on one long utterance each (opened again before max_frames)."""

    def __init__(self, m, B, X):
        self.ss, self.B, self.X, self.pos = nsd.StreamingSessions(m, B), B, X, 0
        for s in range(B):
            self.ss.open(s, s)
        self.act = [True] * B

    def push_decode(self):
        if self.ss._frames[0] + 1 >= self.ss.max_frames:
            for s in range(self.B):
                self.ss.open(s, s)
        self.ss.push_decode(self.X[self.pos % len(self.X)], self.act)
        self.pos += 1

    def replay(self):
        self.ss._graph.replay()


class Decoder:
    """StreamingDecoder's fast form (engaged after the exact-form warm-up)."""

    def __init__(self, m, B, X):
        self.sd, self.X, self.pos = nsd.StreamingDecoder(m, B, torch.arange(B, device="cuda")), X, 0
        while not self.sd._steady:
            self.push_decode()

    def push_decode(self):
        self.sd.push_decode(self.X[self.pos % len(self.X)])
        self.pos += 1

    def replay(self):
        self.sd._graph.replay()


def latency(obj, pushes):
    host = []
    for _ in range(pushes):
        t0 = time.perf_counter()
        obj.push_decode()
        host.append(time.perf_counter() - t0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(pushes):
        obj.replay()
    e1.record()
    torch.cuda.synchronize()
    h = np.array(host) * 1e6
    return float(np.median(h)), float(np.percentile(h, 90)), e0.elapsed_time(e1) * 1e3 / pushes


def replay_set(m, n_utts, out):
    g = torch.Generator().manual_seed(1)
    lens = torch.randint(200, 601, (n_utts,), generator=g).tolist()
    utts = [torch.randn(T, N, generator=g) for T in lens]
    days = torch.randint(0, KW["nDays"], (n_utts,), generator=g).tolist()
    B = 8
    ss = nsd.StreamingSessions(m, B)
    bins = torch.zeros(B, S, N).pin_memory()
    # warm-up: capture the graph on one short utterance
    ss.open(0, 0)
    ss.push_decode(bins, [True] + [False] * (B - 1))
    ss.finish(0, torch.zeros(40, N, device="cuda"))
    torch.cuda.synchronize()
    slot_u, slot_pos, queue, pushes, frames = [None] * B, [0] * B, list(range(n_utts)), 0, 0
    t0 = time.perf_counter()
    while queue or any(u is not None for u in slot_u):
        active = [False] * B
        for s in range(B):
            if slot_u[s] is None and queue:
                slot_u[s], slot_pos[s] = queue.pop(0), 0
                ss.open(s, days[slot_u[s]])
            u = slot_u[s]
            if u is None:
                continue
            X = utts[u]
            if X.shape[0] - slot_pos[s] < S:
                frames += ss.finish(s, X[slot_pos[s]:].cuda(non_blocking=True)).shape[0]
                slot_u[s] = None
                continue
            bins[s].copy_(X[slot_pos[s]:slot_pos[s] + S])
            active[s] = True
            slot_pos[s] += S
        if any(active):
            ids = ss.push_decode(bins, active)
            frames += int((ids >= 0).sum())
            pushes += 1
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    audio = sum(lens) * 0.02
    out({"what": "replay_8_slots", "utterances": n_utts, "bins": sum(lens), "audio_s": round(audio, 2), "frames": frames, "pushes": pushes,
         "wall_s": round(wall, 3), "utt_per_s": round(n_utts / wall, 2), "rtf": round(wall / audio, 5),
         "us_per_push": round(wall * 1e6 / pushes, 1)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/stream_sessions_time.jsonl")
    ap.add_argument("--pushes", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--utts", type=int, default=240)
    a = ap.parse_args()
    f = open(a.out, "w")

    def out(d):
        line = json.dumps(d)
        print(line, flush=True)
        f.write(line + "\n")

    out(gpu_line())
    nsd.set_default_precision("bf16")
    torch.manual_seed(0)
    m = nsd.GRUDecoder(device="cuda", bidirectional=False, dropout=0.0, **KW)
    nsd.set_default_precision("fp32")
    fill_trained_like_(m, seed=5)
    m = m.cuda().eval()
    g = torch.Generator().manual_seed(0)
    forms = []
    for B in (1, 4, 8):
        X = [torch.randn(B, S, N, generator=g).pin_memory() for _ in range(64)]
        forms.append(("sessions", B, Sessions(m, B, X)))
        if B in (1, 8):
            forms.append(("decoder_fast", B, Decoder(m, B, X)))
    for _, _, obj in forms:                 # warm every form (graph captured, modules loaded)
        latency(obj, 20)
    res = {(w, B): [] for w, B, _ in forms}
    for _ in range(a.rounds):               # alternate the forms round by round
        for w, B, obj in forms:
            res[(w, B)].append(latency(obj, a.pushes))
    for (w, B), r in res.items():
        r = np.array(r)
        out({"what": "push_latency_all_active", "form": w, "B": B, "pushes": a.pushes, "rounds": a.rounds,
             "host_to_host_us_median": round(float(np.median(r[:, 0])), 1), "host_to_host_us_p90": round(float(np.median(r[:, 1])), 1),
             "device_us_per_replay": round(float(np.median(r[:, 2])), 1),
             "device_us_per_replay_rounds": [round(float(v), 1) for v in r[:, 2]]})
    replay_set(m, a.utts, out)
    f.close()


if __name__ == "__main__":
    main()
