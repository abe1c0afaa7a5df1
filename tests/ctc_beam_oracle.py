"""float64 reference of the CTC prefix beam search with a phoneme-bigram prior (K5b, ``nsd_ctc_beam_*``).

It implements the semantics of include/nsd_b200.h literally, tie-break rule included, vectorised over the candidates of
one frame.  It lives beside the tests rather than in ``oracle/``, which holds the reference of the training path."""
from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np

NEG_INF = -np.inf


def ctc_prefix_beam_search(lp: np.ndarray, length: int, W: int, blank: int = 0, lm: Optional[np.ndarray] = None,
                           alpha: float = 0.0, beta: float = 0.0) -> Tuple[List[Tuple[Tuple[int, ...], float, float]], float]:
    """lp: [T, C] log-probs of one utterance; frames t < length are decoded with beam width W.

    Returns ``(beam, gap)``: ``beam`` is the final beam in rank order, a list of ``(labels, total, acoustic)`` with
    ``acoustic = Pb (+) Pnb`` and ``total = acoustic + alpha * sum lm + beta * len``; ``gap`` is the smallest difference
    between the last kept and the first dropped candidate's total over all frames (inf if nothing was ever dropped)."""
    lp = np.asarray(lp, dtype=np.float64)
    C = lp.shape[1]
    use_lm = lm is not None and alpha != 0.0
    lm64 = np.asarray(lm, dtype=np.float64) if use_lm else None
    beam: List[Tuple[int, ...]] = [()]
    pb = np.array([0.0])
    pnb = np.array([NEG_INF])
    prior = np.array([0.0])
    gap = np.inf
    cols = np.arange(C)
    with np.errstate(invalid="ignore"):
        for t in range(max(0, min(int(length), lp.shape[0]))):
            y = lp[t]
            n = len(beam)
            index = {l: i for i, l in enumerate(beam)}
            last = np.array([l[-1] if l else -1 for l in beam], dtype=np.int64)
            par = np.array([index.get(l[:-1], -1) if l else -1 for l in beam], dtype=np.int64)
            both = np.logaddexp(pb, pnb)
            # stay
            pb_s = both + y[blank]
            pnb_s = np.where(last >= 0, pnb + y[np.maximum(last, 0)], NEG_INF)
            merged = np.zeros((n, C), dtype=bool)
            for j in np.nonzero(par >= 0)[0]:
                q, c = par[j], last[j]
                ext = (pb[q] if last[q] == c else both[q]) + y[c]
                pnb_s[j] = np.logaddexp(pnb_s[j], ext)
                merged[q, c] = True
            tot_s = np.logaddexp(pb_s, pnb_s) + prior
            # extend by every c
            pnb_e = np.where(cols[None, :] == last[:, None], pb[:, None], both[:, None]) + y[None, :]
            ctx = np.where(last >= 0, last, blank)
            inc = alpha * lm64[ctx] + beta if use_lm else np.full((n, C), float(beta))
            prior_e = prior[:, None] + inc
            tot_e = pnb_e + prior_e
            tot_e[:, blank] = NEG_INF
            tot_e[merged] = NEG_INF
            totals = np.concatenate([tot_s[:, None], tot_e], axis=1).ravel()       # key i*(C+1) + r
            keys = np.arange(totals.size)
            valid = totals > NEG_INF
            order = np.lexsort((keys, -totals))
            order = order[valid[order]]
            if order.size > W:
                gap = min(gap, totals[order[W - 1]] - totals[order[W]])
            keep = order[:W]
            nb, npb, npnb, nprior = [], [], [], []
            for k in keep.tolist():
                i, r = divmod(k, C + 1)
                if r == 0:
                    nb.append(beam[i]); npb.append(pb_s[i]); npnb.append(pnb_s[i]); nprior.append(prior[i])
                else:
                    c = r - 1
                    nb.append(beam[i] + (c,)); npb.append(NEG_INF); npnb.append(pnb_e[i, c]); nprior.append(prior_e[i, c])
            beam, pb, pnb, prior = nb, np.array(npb), np.array(npnb), np.array(nprior)
    acoustic = np.logaddexp(pb, pnb) if len(beam) else np.zeros(0)
    total = acoustic + prior
    return [(tuple(int(c) for c in l), float(s), float(a)) for l, s, a in zip(beam, total, acoustic)], float(gap)


def prior_of(labels, blank: int, lm: Optional[np.ndarray], alpha: float, beta: float) -> float:
    """alpha * sum of lm[previous token (blank at the start), token] + beta * len(labels)."""
    s, prev = 0.0, blank
    if lm is not None and alpha != 0.0:
        for c in labels:
            s += alpha * float(lm[prev, c])
            prev = c
    return s + beta * len(labels)
