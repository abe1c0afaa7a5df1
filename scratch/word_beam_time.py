"""K5d word beam search timing beside K5b: one JSON line per configuration, GPU name and power limit first.

Each timed call is the device work of decoding one batch with a reused decoder: ``reset`` + ``advance`` over every frame (logits,
log-softmaxed in the kernel) + the 4-best read-out (``final=True`` for K5d).  Shapes B=64/T'=118 and B=256/T'=493, C=41, W=16 and
64; K5d with a synthetic lexicon of 10 k and of 100 k words (pronunciations of 3-8 random phones, 5 % homophones), each without an
LM and with a seeded 3-gram of about 1 M entries over its words; K5b (no prior) on the same logits.  The logits spell random
words of the 100 k lexicon with separators, so hypotheses stay inside the lexicon and finish words.  Configurations of a shape are
alternated over ``--rounds`` rounds; the median round is reported with the spread.

    python scratch/word_beam_time.py [--reps 20] [--warmup 3] [--rounds 3] [--out profiles/k5d_word_beam_time.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from neural_speech_decoder_b200.ctc import CtcBeamSearch, Lexicon, NgramLM, WordBeamSearch  # noqa: E402

C, SEP = 41, 40


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def lexicon_pairs(rng, n):
    lens = rng.integers(3, 9, n)
    phones = rng.integers(1, 40, (n, 8))
    pairs = [(f"W{i}", phones[i, :lens[i]].tolist()) for i in range(n)]
    for k, i in enumerate(rng.integers(0, n, n // 20)):
        pairs.append((f"H{k}", pairs[int(i)][1]))
    return pairs


def trigram_lm(rng, words, n2, n3):
    """About n2 bigrams and n3 trigrams over <s>, </s>, <unk> + words, natural-log values, built directly as NgramLM."""
    vocab = ["<s>", "</s>", "<unk>"] + list(words)
    V = len(vocab)
    p1 = -rng.uniform(2.0, 12.0, V)
    p1[0] = -99.0
    bo1 = -rng.uniform(0.0, 2.0, V)
    big = np.unique(np.stack([np.where(rng.random(n2) < 0.02, 0, rng.integers(2, V, n2)), rng.integers(1, V, n2)], 1), axis=0)
    bigrams = {(int(a), int(w)): (float(p), float(b)) for (a, w), p, b in zip(big, -rng.uniform(0.2, 7.0, len(big)), -rng.uniform(0, 2, len(big)))}
    hist = big[big[:, 1] != 1]
    tri = np.unique(np.concatenate([hist[rng.integers(len(hist), size=n3)], rng.integers(1, V, (n3, 1))], 1), axis=0)
    trigrams = {(int(a), int(b), int(w)): float(p) for (a, b, w), p in zip(tri, -rng.uniform(0.1, 6.0, len(tri)))}
    return NgramLM(vocab, p1, bo1, bigrams, trigrams)


def spelled_logits(rng, pairs, T, B):
    logits = rng.standard_normal((T, B, C)).astype(np.float32) * 2.5
    for b in range(B):
        t = 0
        while t < T:
            for c in pairs[int(rng.integers(len(pairs)))][1] + [SEP]:
                for _ in range(int(rng.integers(1, 3))):
                    if t < T:
                        logits[t, b, c] += 5.0
                        t += 1
                if t < T and rng.random() < 0.4:
                    logits[t, b, 0] += 5.0
                    t += 1
    lens = rng.integers(T // 2, T + 1, B)
    lens[0] = T
    return torch.from_numpy(logits).cuda(), torch.from_numpy(lens).cuda().to(torch.int32)


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "k5d_word_beam_time.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("word_beam_time.py measures on a GPU; none is visible")
    rng = np.random.default_rng(0)
    big_pairs = lexicon_pairs(rng, 100_000)
    models = {}
    for n in (10_000, 100_000):
        pairs = big_pairs[:n] + big_pairs[100_000:100_000 + n // 20]
        lex = Lexicon.from_pronunciations(pairs, C)
        lm = trigram_lm(np.random.default_rng(n), lex.words, 450_000, 600_000)
        models[n] = (lex, lm, len(lm.p1) + len(lm.p2) + len(lm.p3))
    lines = [gpu_line()]
    print(json.dumps(lines[0]), flush=True)
    for B, T in ((64, 118), (256, 493)):
        act, lens = spelled_logits(np.random.default_rng(B), big_pairs, T, B)
        for W in (16, 64):
            configs = [("k5b", None, False)] + [(f"k5d_{n // 1000}k", n, use_lm) for n in (10_000, 100_000) for use_lm in (False, True)]
            runners = {}
            for name, n, use_lm in configs:
                if n is None:
                    bs = CtcBeamSearch(B, C, W, T)
                    fn = (lambda bs=bs: (bs.reset(), bs.advance(act, lens, True), bs.nbest(4)))
                else:
                    lex, lm, _ = models[n]
                    bs = WordBeamSearch(B, lex, lm if use_lm else None, W, T, 0.8 if use_lm else 0.0, 0.5)
                    fn = (lambda bs=bs: (bs.reset(), bs.advance(act, lens, True), bs.nbest(4, final=True)))
                runners[(name, use_lm)] = fn
            samples = {k: [] for k in runners}
            for _ in range(a.rounds):
                for k, fn in runners.items():
                    samples[k].append(timed(fn, a.reps, a.warmup))
            base = sorted(samples[("k5b", False)])[len(samples[("k5b", False)]) // 2]
            for (name, use_lm), s in samples.items():
                ms = sorted(s)[len(s) // 2]
                rec = {"what": name, "B": B, "T": T, "C": C, "W": W, "ms_per_call": round(ms, 4), "spread_ms": round(max(s) - min(s), 4),
                       "vs_k5b": round(ms / base, 3)}
                if name != "k5b":
                    n = 10_000 if name.endswith("10k") else 100_000
                    lex, lm, entries = models[n]
                    rec.update({"lexicon_words": len(lex.words), "lexicon_nodes": int(lex.nodes.shape[0]),
                                "lm_entries": entries if use_lm else 0})
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
