"""Streaming push latency with live word decoding, at the competition architecture (unidirectional 5x1024, N=256, K=32, S=4): one
JSON line per measurement, GPU name and power limit first.

Three decoders follow ``StreamingSessions`` with every slot active, at 1, 4 and 8 slots: no beam (greedy ids only), K5b at W=16
(phoneme beam, no prior), and K5d at W=16 (word beam over a 10 k-word lexicon with a 3-gram of about 1 M entries, built as in
scratch/word_beam_time.py), whose push also runs the live read-out and copies it to pinned memory.  The protocol of
profiles/stream_sessions_time.jsonl: host to host (``push_decode``: pinned bins in, ids out and, for K5d, the transcript taken in;
one graph replay and one synchronisation; median and p90 over ``--pushes`` calls) and device time per replay (CUDA events around
``--pushes`` back-to-back replays).  The decoders are alternated round by round; the median round is reported.

    python scratch/stream_words_time.py [--out profiles/stream_words_time.jsonl] [--pushes 300] [--rounds 3]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import neural_speech_decoder_b200 as nsd  # noqa: E402
from neural_speech_decoder_b200.ctc import Lexicon  # noqa: E402
from neural_speech_decoder_b200.synthetic import fill_trained_like_  # noqa: E402
from sessions_time import KW, N, S, gpu_line, latency  # noqa: E402
from word_beam_time import C, lexicon_pairs, trigram_lm  # noqa: E402


class Sessions:
    """All slots active on one long utterance each (opened again before max_frames)."""

    def __init__(self, m, B, X, **beam):
        self.ss, self.B, self.X, self.pos = nsd.StreamingSessions(m, B, **beam), B, X, 0
        for s in range(B):
            self.ss.open(s, s)
        self.act = [True] * B
        self.words = beam.get("lexicon") is not None

    def push_decode(self):
        if self.ss._frames[0] + 1 >= self.ss.max_frames:
            for s in range(self.B):
                self.ss.open(s, s)
        self.ss.push_decode(self.X[self.pos % len(self.X)], self.act)
        if self.words:
            self.ss.transcript(0)
        self.pos += 1

    def replay(self):
        self.ss._graph.replay()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/stream_words_time.jsonl")
    ap.add_argument("--pushes", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_words_time.py measures on a GPU; none is visible")
    f = open(a.out, "w")

    def out(d):
        line = json.dumps(d)
        print(line, flush=True)
        f.write(line + "\n")

    out({"what": "gpu", **gpu_line()})
    rng = np.random.default_rng(0)
    lex = Lexicon.from_pronunciations(lexicon_pairs(rng, 10_000), C)
    lm = trigram_lm(np.random.default_rng(10_000), lex.words, 450_000, 600_000)
    lm_entries = len(lm.p1) + len(lm.p2) + len(lm.p3)
    nsd.set_default_precision("bf16")
    torch.manual_seed(0)
    m = nsd.GRUDecoder(device="cuda", bidirectional=False, dropout=0.0, **KW)
    nsd.set_default_precision("fp32")
    fill_trained_like_(m, seed=5)
    m = m.cuda().eval()
    decoders = {"greedy": {}, "k5b_w16": dict(beam_width=16), "k5d_w16": dict(beam_width=16, lexicon=lex, lm=lm, lm_weight=0.8, word_bonus=0.5)}
    g = torch.Generator().manual_seed(0)
    forms = []
    for B in (1, 4, 8):
        X = [torch.randn(B, S, N, generator=g).pin_memory() for _ in range(64)]
        for name, beam in decoders.items():
            forms.append((name, B, Sessions(m, B, X, **beam)))
    for _, _, obj in forms:                 # warm every form (graph captured, modules loaded)
        latency(obj, 20)
    res = {(w, B): [] for w, B, _ in forms}
    for _ in range(a.rounds):               # alternate the decoders round by round
        for w, B, obj in forms:
            res[(w, B)].append(latency(obj, a.pushes))
    words = {}
    for w, B, obj in forms:
        if obj.words:
            words[B] = sum(len(obj.ss.transcript(s)[0]) for s in range(B))
    for (w, B), r in res.items():
        r = np.array(r)
        rec = {"what": "push_latency_all_active", "form": "sessions", "decoder": w, "B": B, "pushes": a.pushes, "rounds": a.rounds,
               "host_to_host_us_median": round(float(np.median(r[:, 0])), 1), "host_to_host_us_p90": round(float(np.median(r[:, 1])), 1),
               "device_us_per_replay": round(float(np.median(r[:, 2])), 1),
               "device_us_per_replay_rounds": [round(float(v), 1) for v in r[:, 2]]}
        if w == "k5d_w16":
            rec.update({"lexicon_words": len(lex.words), "lm_entries": lm_entries, "committed_words_at_end": words[B]})
        out(rec)
    f.close()


if __name__ == "__main__":
    main()
