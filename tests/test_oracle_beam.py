"""The float64 prefix beam search (tests/ctc_beam_oracle.py) against brute force: exact CTC probabilities of every label
sequence, the prior added term by term, and greedy decoding on peaky inputs.  CPU only."""
import itertools

import numpy as np
import pytest

from ctc_beam_oracle import ctc_prefix_beam_search, prior_of
from oracle import nsd_oracle as O


def log_probs(rng, T, C, scale=2.0):
    return O.log_softmax(rng.standard_normal((T, C)) * scale)


def all_label_seqs(C, blank, max_len):
    labels = [c for c in range(C) if c != blank]
    for n in range(max_len + 1):
        yield from itertools.product(labels, repeat=n)


def neg_nll(lp, labels, blank):
    nll, _, _ = O.ctc_alpha_beta(lp, np.array(labels, dtype=np.int64), lp.shape[0], len(labels), blank)
    return -nll


EXHAUSTIVE = [(4, T) for T in range(1, 5)] + [(3, T) for T in range(1, 7)]


@pytest.mark.parametrize("C,T", EXHAUSTIVE)
@pytest.mark.parametrize("prior", [False, True])
def test_exhaustive_against_alpha_beta(C, T, prior):
    rng = np.random.default_rng(100 * C + T + (7 if prior else 0))
    blank = int(rng.integers(C)) if prior else 0
    lp = log_probs(rng, T, C)
    lm = O.log_softmax(rng.standard_normal((C, C))) if prior else None
    alpha, beta = (0.7, -0.4) if prior else (0.0, 0.0)
    beam, _ = ctc_prefix_beam_search(lp, T, 128, blank, lm, alpha, beta)
    seqs = list(all_label_seqs(C, blank, T))
    assert len(seqs) <= 128
    # every prefix reachable in T frames survives (nothing is pruned), each exactly once
    reachable = {s for s in seqs if neg_nll(lp, s, blank) > -np.inf}
    assert {l for l, _, _ in beam} == reachable and len(beam) == len(reachable)
    for labels, total, acoustic in beam:
        assert abs(acoustic - neg_nll(lp, labels, blank)) < 1e-10
        assert abs(total - (acoustic + prior_of(labels, blank, lm, alpha, beta))) < 1e-10
    scores = {s: neg_nll(lp, s, blank) + prior_of(s, blank, lm, alpha, beta) for s in seqs}
    assert beam[0][0] == max(scores, key=scores.get)
    assert all(beam[i][1] >= beam[i + 1][1] for i in range(len(beam) - 1))


@pytest.mark.parametrize("W", [1, 3, 16])
@pytest.mark.parametrize("blank", [0, 5])
def test_peaky_equals_greedy(W, blank):
    rng = np.random.default_rng(W + blank)
    T, C = 60, 9
    ids = rng.integers(0, C, T)
    ids[rng.random(T) < 0.4] = blank
    lp = np.full((T, C), -30.0) - rng.random((T, C)) * 5
    lp[np.arange(T), ids] = -1e-6
    for length in (0, 1, 37, T):
        beam, _ = ctc_prefix_beam_search(lp, length, W, blank)
        want = O.greedy_decode(lp[:, None, :], np.array([length]), blank)[0]
        assert list(beam[0][0]) == want


def test_empty_utterance():
    beam, gap = ctc_prefix_beam_search(np.zeros((3, 4)), 0, 4)
    assert beam == [((), 0.0, 0.0)] and gap == np.inf


def test_pruned_beam_keeps_the_best_and_reports_the_gap():
    rng = np.random.default_rng(3)
    lp = log_probs(rng, 40, 6, scale=1.5)
    full, _ = ctc_prefix_beam_search(lp, 40, 1, 0)
    beam, gap = ctc_prefix_beam_search(lp, 40, 4, 0)
    assert len(beam) == 4 and gap > 0
    assert all(beam[i][1] >= beam[i + 1][1] for i in range(3))
    assert len({l for l, _, _ in beam}) == 4
    # the acoustic score of a surviving prefix never exceeds its exact probability (pruning only loses paths)
    for labels, _, acoustic in beam + full:
        assert acoustic <= neg_nll(lp, labels, 0) + 1e-9
