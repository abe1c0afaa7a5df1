"""float64 reference of the lexicon-constrained CTC beam search with a word n-gram LM (K5d, ``nsd_ctc_word_beam_*``).

The loop is ``ctc_beam_oracle.ctc_prefix_beam_search``'s (same stay / merge / rank rules and keep/drop gap); what changes is
the per-candidate prior and which extensions are candidates, as include/nsd_b200.h states them.  The lexicon is a dict
{pronunciation tuple: word ids} and the LM a dict of tuples {n-gram of words: (log10 p, log10 backoff)} queried with ARPA
backoff here, written independently of the library's Lexicon and NgramLM.  The seeded generators of lexicons and ARPA files
used by the tests live here too."""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

NEG_INF = -np.inf
LN10 = math.log(10.0)


# ------------------------------------------------------------------------------------------------ LM as a dict of tuples
def lm_logp(lm: Dict[tuple, Tuple[float, float]], w: str, h: Sequence[str]) -> float:
    """Natural-log lm(w | h) with ARPA backoff over the last two words of h (h non-empty)."""
    h = tuple(h)[-2:]
    if len(h) == 2:
        if h + (w,) in lm:
            return lm[h + (w,)][0] * LN10
        bo = lm[h][1] * LN10 if h in lm else 0.0
        return bo + lm_logp(lm, w, h[1:])
    if h + (w,) in lm:
        return lm[h + (w,)][0] * LN10
    return lm[h][1] * LN10 + lm[(w,)][0] * LN10


def lm_token(lm, word: str) -> str:
    return word if (word,) in lm else "<unk>"


def random_lm(rng: np.random.Generator, words: Sequence[str], order: int, n2: int, n3: int, unk: bool = True,
              backoffs: bool = True) -> Dict[tuple, Tuple[float, float]]:
    """A seeded ARPA-like LM over ``words`` + <s>, </s> (and <unk>): every unigram, up to n2 bigrams and n3 trigrams whose
    prefixes exist; some backoffs absent (0).  Values in log10."""
    vocab = ["<s>", "</s>"] + (["<unk>"] if unk else []) + list(words)
    lm = {}
    for w in vocab:
        lm[(w,)] = (-99.0 if w == "<s>" else float(-rng.uniform(0.5, 4.0)),
                    float(-rng.uniform(0.0, 1.0)) if backoffs and order > 1 and rng.random() < 0.8 else 0.0)
    hist = [w for w in vocab if w != "</s>"]
    succ = [w for w in vocab if w != "<s>"]
    if order >= 2:
        for _ in range(n2):
            k = (hist[rng.integers(len(hist))], succ[rng.integers(len(succ))])
            lm[k] = (float(-rng.uniform(0.1, 3.0)), float(-rng.uniform(0.0, 1.0)) if backoffs and order > 2 and rng.random() < 0.8 else 0.0)
    if order >= 3:
        bigrams = [k for k in lm if len(k) == 2 and k[1] != "</s>"]
        for _ in range(n3):
            a, b = bigrams[rng.integers(len(bigrams))]
            lm[(a, b, succ[rng.integers(len(succ))])] = (float(-rng.uniform(0.05, 2.5)), 0.0)
    return lm


def write_arpa(path: str, lm: Dict[tuple, Tuple[float, float]]) -> None:
    by = {n: [(k, v) for k, v in lm.items() if len(k) == n] for n in (1, 2, 3)}
    order = max(n for n in by if by[n])
    with open(path, "w") as f:
        f.write("\n\\data\\\n")
        for n in range(1, order + 1):
            f.write(f"ngram {n}={len(by[n])}\n")
        for n in range(1, order + 1):
            f.write(f"\n\\{n}-grams:\n")
            for k, (p, bo) in by[n]:
                f.write(f"{p:.6f}\t{' '.join(k)}" + (f"\t{bo:.6f}" if n < order and bo != 0.0 else "") + "\n")
        f.write("\n\\end\\\n")


def read_back(lm):
    """The values as write_arpa stores them (6 decimals), so an oracle over the dict sees what the file holds."""
    return {k: (float(f"{p:.6f}"), float(f"{bo:.6f}")) for k, (p, bo) in lm.items()}


def random_lexicon(rng: np.random.Generator, n_words: int, phones: Sequence[int], min_len: int = 1, max_len: int = 6,
                   homophones: int = 0, prefixes: int = 0) -> List[Tuple[str, Tuple[int, ...]]]:
    """Seeded (word, pronunciation) pairs over ``phones``: distinct random words, plus ``homophones`` words sharing another's
    pronunciation and ``prefixes`` words whose pronunciation is a proper prefix of another's."""
    pairs, seen = [], set()
    while len(pairs) < n_words:
        p = tuple(int(x) for x in rng.choice(phones, rng.integers(min_len, max_len + 1)))
        if p in seen:
            continue
        seen.add(p)
        pairs.append((f"W{len(pairs)}", p))
    for k in range(homophones):
        pairs.append((f"H{k}", pairs[int(rng.integers(n_words))][1]))
    for k in range(prefixes):
        long = [p for _, p in pairs if len(p) > 1]
        if long:
            p = long[int(rng.integers(len(long)))]
            pairs.append((f"P{k}", p[:int(rng.integers(1, len(p)))]))
    return pairs


# ------------------------------------------------------------------------------------------------ the beam
class Words:
    """The lexicon and LM side of the rules: which extension is a candidate and what it adds to the prior."""

    def __init__(self, pairs, sep: int, lm=None, alpha: float = 0.0, beta: float = 0.0):
        self.word_id, self.prons = {}, {}
        for w, p in pairs:
            self.word_id.setdefault(w, len(self.word_id))
            self.prons.setdefault(tuple(p), set()).add(self.word_id[w])
        self.words = list(self.word_id)
        self.prons = {p: sorted(ws) for p, ws in self.prons.items()}
        self.prefixes = {p[:k] for p in self.prons for k in range(1, len(p) + 1)}
        self.sep, self.lm, self.alpha, self.beta = sep, lm, alpha, beta

    def best_word(self, pron, hist) -> Tuple[int, float]:
        """(w*, separator increment) for a word spelled ``pron`` after LM history ``hist``."""
        ws = self.prons[pron]
        if self.lm is None:
            return ws[0], self.beta
        vals = [lm_logp(self.lm, lm_token(self.lm, self.words[w]), hist) for w in ws]
        k = int(np.argmax(vals))                    # first maximum: the smaller word id
        return ws[k], self.alpha * vals[k] + self.beta

    def state(self, labels):
        """(pronunciation since the last sep, word ids, LM history, prior) of a label sequence, or None if it is not valid."""
        cur, words, hist, prior = (), [], ("<s>",), 0.0
        for c in labels:
            if c == self.sep:
                if cur not in self.prons:
                    return None
                w, inc = self.best_word(cur, hist)
                prior += inc
                words.append(w)
                hist = (hist + (lm_token(self.lm, self.words[w]) if self.lm is not None else self.words[w],))[-2:]
                cur = ()
            else:
                cur = cur + (c,)
                if cur not in self.prefixes:
                    return None
        return cur, tuple(words), hist, prior

    def end(self, labels) -> Tuple[float, Optional[int]]:
        """The final read-out's end term and pending word of a valid label sequence (-inf: not at a word boundary)."""
        cur, _, hist, _ = self.state(labels)
        pend, term = None, 0.0
        if cur:
            if cur not in self.prons:
                return NEG_INF, None
            pend, term = self.best_word(cur, hist)
            hist = (hist + (lm_token(self.lm, self.words[pend]) if self.lm is not None else "",))[-2:]
        if self.lm is not None:
            term += self.alpha * lm_logp(self.lm, "</s>", hist)
        return term, pend


def word_beam_search(lp: np.ndarray, length: int, W: int, lex: Words, blank: int = 0):
    """lp: [T, C] log-probs of one utterance; frames t < length are decoded with beam width W under ``lex``.

    Returns ``(beam, gap)``: ``beam`` in rank order, a list of ``(labels, words, total, acoustic)``; ``gap`` as in
    ``ctc_beam_oracle``: the smallest keep/drop difference of totals over all frames (inf if nothing was ever dropped)."""
    lp = np.asarray(lp, dtype=np.float64)
    C = lp.shape[1]
    sep = lex.sep
    beam: List[Tuple[int, ...]] = [()]
    info = {(): lex.state(())}
    pb, pnb, prior = np.array([0.0]), np.array([NEG_INF]), np.array([0.0])
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
            pb_s = both + y[blank]
            pnb_s = np.where(last >= 0, pnb + y[np.maximum(last, 0)], NEG_INF)
            merged = np.zeros((n, C), dtype=bool)
            for j in np.nonzero(par >= 0)[0]:
                q, c = par[j], last[j]
                ext = (pb[q] if last[q] == c else both[q]) + y[c]
                pnb_s[j] = np.logaddexp(pnb_s[j], ext)
                merged[q, c] = True
            tot_s = np.logaddexp(pb_s, pnb_s) + prior
            pnb_e = np.where(cols[None, :] == last[:, None], pb[:, None], both[:, None]) + y[None, :]
            prior_e = np.repeat(prior[:, None], C, axis=1)
            allowed = np.zeros((n, C), dtype=bool)
            for i, l in enumerate(beam):
                cur, _, hist, _ = info[l]
                for c in range(C):
                    if c == blank:
                        continue
                    if c == sep:
                        if cur and cur in lex.prons:
                            allowed[i, c] = True
                            prior_e[i, c] += lex.best_word(cur, hist)[1]
                    elif cur + (c,) in lex.prefixes:
                        allowed[i, c] = True
            tot_e = pnb_e + prior_e
            tot_e[~allowed] = NEG_INF
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
                    l = beam[i] + (c,)
                    if l not in info:
                        info[l] = lex.state(l)
                    nb.append(l); npb.append(NEG_INF); npnb.append(pnb_e[i, c]); nprior.append(prior_e[i, c])
            beam, pb, pnb, prior = nb, np.array(npb), np.array(npnb), np.array(nprior)
    acoustic = np.logaddexp(pb, pnb) if len(beam) else np.zeros(0)
    total = acoustic + prior
    return [(tuple(int(c) for c in l), info[l][1], float(s), float(a)) for l, s, a in zip(beam, total, acoustic)], float(gap)


def finalize(beam, lex: Words):
    """The final read-out: end terms added, re-ranked by total (ties -> beam order); entries inside an unfinished word get
    -inf and are listed last with no labels or words.  -> list of (labels, words, total, acoustic)."""
    out = []
    for k, (labels, words, total, ac) in enumerate(beam):
        term, pend = lex.end(labels)
        if term == NEG_INF:
            out.append(((), (), NEG_INF, NEG_INF, k))
        else:
            out.append((labels, words + ((pend,) if pend is not None else ()), total + term, ac, k))
    out.sort(key=lambda e: (-e[2] if e[2] > NEG_INF else np.inf, e[4]))
    return [e[:4] for e in out]
