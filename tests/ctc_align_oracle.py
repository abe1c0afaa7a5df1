"""float64 reference of CTC forced alignment (K5c, ``nsd_ctc_align``).

It implements the semantics of include/nsd_b200.h literally, tie rules included, vectorised over the lattice states of one
frame, and reports how close each decision of the chosen path came to a tie.  It lives beside the tests rather than in
``oracle/``, which holds the reference of the training path."""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

NEG_INF = -np.inf


def lattice(target, L: int, blank: int) -> Tuple[np.ndarray, np.ndarray]:
    """-> (ext [2L+1], skip [2L+1] bool: the s-2 predecessor counts)."""
    S = 2 * L + 1
    ext = np.full(S, blank, dtype=np.int64)
    ext[1::2] = np.asarray(target[:L], dtype=np.int64)
    skip = np.zeros(S, dtype=bool)
    skip[3::2] = ext[3::2] != ext[1:-2:2]
    return ext, skip


def min_frames(target, L: int) -> int:
    """L plus the number of adjacent equal target pairs: the fewest frames any path of the lattice needs."""
    t = np.asarray(target[:L])
    return L + int((t[1:] == t[:-1]).sum())


def ctc_viterbi(lp: np.ndarray, target, il: int, L: int, blank: int = 0) -> Tuple[float, Optional[np.ndarray], float]:
    """lp: [T, C] log-probs of one utterance; frames t < il, the first L targets.

    Returns ``(score, states, margin)``: the best path's log-probability, its lattice state per frame ([il] int64, None when no
    path exists; score is then -inf, or 0 for il = L = 0) and the smallest gap, over every decision of the backtrace and the
    final-state choice, between the chosen candidate and the best other finite candidate (inf if there never was one)."""
    lp = np.asarray(lp, dtype=np.float64)
    ext, skip = lattice(target, L, blank)
    S = 2 * L + 1
    if il == 0:
        return (0.0 if L == 0 else NEG_INF), None, np.inf
    if il < min_frames(target, L):
        return NEG_INF, None, np.inf
    delta = np.full((il, S), NEG_INF)
    code = np.zeros((il, S), dtype=np.int8)
    delta[0, 0] = lp[0, blank]
    if L > 0:
        delta[0, 1] = lp[0, ext[1]]
    for t in range(1, il):
        p = delta[t - 1]
        pp = np.concatenate([[NEG_INF, NEG_INF], p])      # two -inf guard cells in front
        c1 = pp[1:-1]
        c2 = np.where(skip, pp[:-2], NEG_INF)
        best = p.copy()
        k = np.zeros(S, dtype=np.int8)
        up = c1 > best                                  # strict: a tie stays
        best[up], k[up] = c1[up], 1
        up = c2 > best
        best[up], k[up] = c2[up], 2
        delta[t] = best + lp[t, ext]
        code[t] = k
    s = S - 1
    if S > 1 and delta[il - 1, S - 2] > delta[il - 1, S - 1]:
        s = S - 2
    score = float(delta[il - 1, s])
    if not score > NEG_INF:
        return score, None, np.inf
    margin = np.inf
    if S > 1:
        other = delta[il - 1, S - 1 if s == S - 2 else S - 2]
        if other > NEG_INF:
            margin = score - other
    states = np.zeros(il, dtype=np.int64)
    for t in range(il - 1, 0, -1):
        states[t] = s
        cands = [(s, 0)] + ([(s - 1, 1)] if s >= 1 else []) + ([(s - 2, 2)] if skip[s] else [])
        chosen = s - int(code[t, s])
        others = [delta[t - 1, q] for q, _ in cands if q != chosen and delta[t - 1, q] > NEG_INF]
        if others:
            margin = min(margin, delta[t - 1, chosen] - max(others))
        s = chosen
    states[0] = s
    return score, states, float(margin)


def align_batch(lp: np.ndarray, targets: np.ndarray, in_lens, tgt_lens, blank: int = 0):
    """lp: [T, B, C]; targets [B, S] padded.  -> dict of the kernel's outputs (float64) plus ``margin`` [B], with the header's
    clamping of the lengths and its handling of bad targets and infeasible utterances."""
    T, B, C = lp.shape
    Smax = targets.shape[1]
    out = dict(labels=np.full((B, T), -1, dtype=np.int64), frame_logp=np.zeros((B, T)), spans=np.full((B, Smax, 2), -1, dtype=np.int64),
               token_logp=np.zeros((B, Smax)), score=np.zeros(B), margin=np.full(B, np.inf), bad=np.zeros(B, dtype=bool))
    for b in range(B):
        il = min(max(int(in_lens[b]), 0), T)
        L = min(max(int(tgt_lens[b]), 0), Smax)
        tg = np.asarray(targets[b, :L], dtype=np.int64)
        if ((tg == blank) | (tg < 0) | (tg >= C)).any():
            out["bad"][b] = True
            out["score"][b] = NEG_INF
            continue
        score, states, margin = ctc_viterbi(lp[:, b], tg, il, L, blank)
        out["score"][b], out["margin"][b] = score, margin
        if states is None:
            continue
        ext, _ = lattice(tg, L, blank)
        lab = ext[states]
        out["labels"][b, :il] = lab
        fl = lp[np.arange(il), b, lab].astype(np.float64)
        out["frame_logp"][b, :il] = fl
        for k in range(L):
            fr = np.nonzero(states == 2 * k + 1)[0]
            out["spans"][b, k] = (fr[0], fr[-1])
            out["token_logp"][b, k] = fl[fr[0]:fr[-1] + 1].sum()
    return out
