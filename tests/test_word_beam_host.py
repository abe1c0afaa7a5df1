"""K5d's host half without a GPU: ARPA loading (``NgramLM``) against the dict-of-tuples LM of tests/ctc_word_beam_oracle.py, the
pronunciation ``Lexicon`` and the arrays the kernel reads, transcript <-> word-id helpers, the constructor guards that need no
device, and an exhaustive check of the fp64 oracle against a brute-force sum over CTC paths."""
import itertools
import os

import numpy as np
import pytest
import torch

from ctc_word_beam_oracle import (LN10, NEG_INF, Words, finalize, lm_logp, random_lexicon, random_lm, read_back, word_beam_search,
                                  write_arpa)

import neural_speech_decoder_b200 as nsd
from neural_speech_decoder_b200.ctc import PHONEMES, SIL, Lexicon, NgramLM


# ------------------------------------------------------------------------------------------------ ARPA
@pytest.mark.parametrize("order,unk,backoffs", [(1, True, True), (2, False, True), (3, True, True), (3, True, False), (3, False, True)])
def test_arpa_matches_dict_lm(tmp_path, order, unk, backoffs):
    rng = np.random.default_rng(order * 10 + unk)
    words = [f"W{i}" for i in range(30)]
    lm = read_back(random_lm(rng, words, order, 150, 200, unk=unk, backoffs=backoffs))
    path = str(tmp_path / "lm.arpa")
    write_arpa(path, lm)
    m = NgramLM.from_arpa(path)
    assert m.order == order and sorted(m.vocab) == sorted(k[0] for k in lm if len(k) == 1)
    assert m.p1[m.index["W3"]] == np.float32(lm[("W3",)][0] * LN10)          # log10 -> natural log
    # every n-gram, queried with its own history, and random (mostly backed-off) queries
    queries = [(k[-1], k[:-1]) for k in lm if len(k) > 1] + [(k[0], ("<s>",)) for k in lm if len(k) == 1 and k[0] != "<s>"]
    vocab = [k[0] for k in lm if len(k) == 1 and k[0] != "<s>"]
    for _ in range(300):
        h = tuple(vocab[i] for i in rng.integers(len(vocab), size=int(rng.integers(1, 3))))
        queries.append((vocab[rng.integers(len(vocab))], h))
    for w, h in queries:
        assert abs(m.logp(w, h) - lm_logp(lm, w, h)) <= 1e-5 * max(1.0, abs(lm_logp(lm, w, h))), (w, h)
    if unk:
        assert m.logp("NOT-A-WORD", ("<s>",)) == m.logp("<unk>", ("<s>",))
        assert m.logp("W1", ("NOT-A-WORD",)) == m.logp("W1", ("<unk>",))
    else:
        with pytest.raises(KeyError):
            m.logp("NOT-A-WORD")


def _arpa_lines(lm):
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "x.arpa")
        write_arpa(p, lm)
        return open(p).read().splitlines()


def _load(tmp_path, lines):
    p = str(tmp_path / "bad.arpa")
    open(p, "w").write("\n".join(lines) + "\n")
    return NgramLM.from_arpa(p)


def test_arpa_malformed_raises(tmp_path):
    rng = np.random.default_rng(3)
    lm = read_back(random_lm(rng, ["A", "B", "C"], 3, 6, 4))
    lines = _arpa_lines(lm)
    _load(tmp_path, lines)                                     # the unmodified file loads
    i2 = lines.index("ngram 2=" + str(sum(len(k) == 2 for k in lm)))
    bad = list(lines)
    bad[i2] = "ngram 2=" + str(sum(len(k) == 2 for k in lm) + 1)
    with pytest.raises(ValueError, match="2-grams"):           # count mismatch
        _load(tmp_path, bad)
    first_bigram = lines.index("\\2-grams:") + 1
    dup = list(lines)
    dup.insert(first_bigram, lines[first_bigram])
    dup[i2] = "ngram 2=" + str(sum(len(k) == 2 for k in lm) + 1)
    with pytest.raises(ValueError, match="duplicate"):
        _load(tmp_path, dup)
    i3 = [k for k, l in enumerate(lines) if l.startswith("ngram 3=")][0]
    orphan = list(lines)
    missing = next((a, b) for a in ("A", "B", "C") for b in ("A", "B", "C") if (a, b) not in lm)
    orphan.insert(lines.index("\\3-grams:") + 1, f"-0.5\t{missing[0]} {missing[1]} C")
    orphan[i3] = "ngram 3=" + str(sum(len(k) == 3 for k in lm) + 1)
    with pytest.raises(ValueError, match="prefix"):
        _load(tmp_path, orphan)
    four = list(lines)
    four.insert(four.index("\\end\\"), "\\4-grams:")
    with pytest.raises(ValueError, match="order 4"):
        _load(tmp_path, four)


# ------------------------------------------------------------------------------------------------ lexicon
def _walk(lex: Lexicon, pron):
    """Follow a pronunciation through the kernel's arrays: child(c) = first child + popcount(mask below c)."""
    nodes = lex.nodes.view(np.uint32).astype(np.int64)
    u = 0
    for c in pron:
        mask = sum(int(nodes[u, k]) << (32 * k) for k in range(4))
        assert (mask >> c) & 1, (pron, c)
        u = int(nodes[u, 4]) + bin(mask & ((1 << c) - 1)).count("1")
    return u


def test_lexicon_arrays_homophones_and_prefixes():
    rng = np.random.default_rng(0)
    pairs = random_lexicon(rng, 200, [1, 2, 3, 5, 7, 33, 39], homophones=20, prefixes=20)
    pairs.append(("W0", (39, 39, 39, 39, 39, 39, 39, 39)))    # a second pronunciation of an existing word
    lex = Lexicon.from_pronunciations(pairs, 41)
    assert lex.words[0] == "W0" and len(lex.prons[0]) == 2
    by_pron = {}
    for w, p in pairs:
        by_pron.setdefault(tuple(p), set()).add(lex.word_index[w])
    for p, ws in by_pron.items():
        u = _walk(lex, p)
        first, count = int(lex.nodes[u, 5]), int(lex.nodes[u, 6])
        assert list(lex.entries[first:first + count]) == sorted(ws)          # homophones, ascending id
    assert any(len(ws) > 1 for ws in by_pron.values())
    assert any(p[:k] in by_pron for p in by_pron for k in range(1, len(p)))  # a word that is a prefix of another
    assert lex.nodes[0, 6] == 0                                              # the root holds no word
    n = lex.nodes.shape[0]
    assert n == 1 + len({p[:k] for p in by_pron for k in range(1, len(p) + 1)})
    assert ((lex.nodes[:, 4] >= 0) & (lex.nodes[:, 4] < n)).all()


def test_lexicon_from_cmudict_file(tmp_path):
    p = tmp_path / "dict.txt"
    p.write_text(";;; comment line\nHELLO  HH AH0 L OW1\nHELLO(2)  HH EH0 L OW1\nWORLD W ER1 L D\nWERLD W ER0 L D\n\nA AH0\n")
    lex = Lexicon.from_file(str(p))
    assert lex.num_classes == 41 and lex.blank == 0 and lex.sep == SIL == 40
    ph = {q: i + 1 for i, q in enumerate(PHONEMES)}
    assert lex.words == ["HELLO", "WORLD", "WERLD", "A"]
    assert lex.prons[0] == [[ph["HH"], ph["AH"], ph["L"], ph["OW"]], [ph["HH"], ph["EH"], ph["L"], ph["OW"]]]
    u = _walk(lex, [ph["W"], ph["ER"], ph["L"], ph["D"]])
    assert list(lex.entries[lex.nodes[u, 5]:lex.nodes[u, 5] + lex.nodes[u, 6]]) == [1, 2]    # homophones
    assert len(PHONEMES) == 39 and PHONEMES[0] == "AA" and PHONEMES[-1] == "ZH"


@pytest.mark.parametrize("pairs,match", [
    ([("X", ["QQ"])], "unknown phone"),
    ([("X", [1, 0, 2])], "blank / sep"),
    ([("X", [1, 40])], "blank / sep"),
    ([("X", [])], "empty"),
    ([("X", [41])], "outside"),
])
def test_lexicon_rejects(pairs, match):
    with pytest.raises(ValueError, match=match):
        Lexicon.from_pronunciations(pairs, 41)


def test_lexicon_rejects_sep_equal_blank():
    with pytest.raises(ValueError):
        Lexicon.from_pronunciations([("X", [1])], 5, blank=0, sep=0)


def test_words_to_ids_and_back():
    lex = Lexicon.from_pronunciations([("A", [1]), ("B", [2]), ("C", [1, 2])], 5, sep=4)
    ids, lens = nsd.words_to_ids(["A C", "B ZZZ A", ""], lex)
    assert ids.dtype == torch.int32 and lens.tolist() == [2, 3, 0]
    assert ids.tolist() == [[0, 2, -1], [1, -1, 0], [-1, -1, -1]]
    assert nsd.ids_to_words(ids[0], lex) == ["A", "C"]


def test_constructor_guards_without_device(tmp_path):
    lex = Lexicon.from_pronunciations([("A", [1]), ("B", [2])], 5, sep=4)
    with pytest.raises(nsd.NsdError, match="phoneme-bigram"):
        nsd.WordBeamSearch(2, lex, lm=torch.zeros(5, 5))
    lm = read_back(random_lm(np.random.default_rng(1), ["A"], 2, 3, 0, unk=False))
    path = str(tmp_path / "lm.arpa")
    write_arpa(path, lm)
    with pytest.raises(nsd.NsdError, match="<unk>"):
        nsd.WordBeamSearch(2, lex, lm=NgramLM.from_arpa(path))                  # "B" is not in the LM, which has no <unk>
    with pytest.raises(nsd.NsdError, match="differ"):
        nsd.WordBeamSearch(2, lex, sep=3)


# ------------------------------------------------------------------------------------------------ oracle, exhaustively
def _collapse(path, blank):
    out, prev = [], None
    for c in path:
        if c != prev and c != blank:
            out.append(c)
        prev = c
    return tuple(out)


@pytest.mark.parametrize("T,seed,use_lm,sep", [(T, s, u, sep) for T in range(1, 7) for s, u, sep in ((0, True, 4), (1, False, 4), (2, True, 2))])
def test_oracle_equals_brute_force(T, seed, use_lm, sep):
    """C = 5: every CTC path is enumerated; the beam (wide enough that nothing is dropped) holds exactly the lexicon-valid
    label sequences, each with the exact path sum as acoustic and the word prior."""
    C, blank = 5, 0
    rng = np.random.default_rng(100 * seed + T)
    phones = [c for c in range(1, C) if c != sep]
    pairs = [("A", (phones[0],)), ("B", (phones[1], phones[0])), ("C", (phones[1],)), ("D", (phones[1],)), ("E", (phones[2], phones[2]))]
    lm = read_back(random_lm(rng, ["A", "B", "C"], 3, 12, 10)) if use_lm else None   # D and E are <unk>
    lex = Words(pairs, sep, lm, alpha=0.7, beta=-0.4)
    lp = np.log(rng.dirichlet(np.ones(C) * 0.7, size=T))
    beam, gap = word_beam_search(lp, T, 128, lex, blank)
    assert gap == np.inf
    sums = {}
    for path in itertools.product(range(C), repeat=T):
        l = _collapse(path, blank)
        s = float(sum(lp[t, c] for t, c in enumerate(path)))
        sums[l] = np.logaddexp(sums.get(l, NEG_INF), s)
    valid = {l: a for l, a in sums.items() if lex.state(l) is not None}
    assert {e[0] for e in beam} == set(valid)
    for labels, words, total, ac in beam:
        _, w, _, prior = lex.state(labels)
        assert words == w
        assert abs(ac - valid[labels]) <= 1e-9 and abs(total - (ac + prior)) <= 1e-9
    # the final read-out: end terms, -inf inside a word, ranked by total
    fin = finalize(beam, lex)
    tot = [e[2] for e in fin]
    assert tot == sorted(tot, reverse=True)
    for labels, words, total, ac in fin:
        if total > NEG_INF:
            cur = lex.state(labels)[0]
            assert not cur or cur in lex.prons
            assert len(words) == len(lex.state(labels)[1]) + (1 if cur else 0)
        else:
            assert labels == () and words == () and ac == NEG_INF
