"""K5d lexicon-constrained CTC beam search with a word n-gram LM (``nsd_ctc_word_beam_*``, ``WordBeamSearch``,
``word_beam_search``, ``word_error_rate``, ``trainer.eval_batch_words``) against the float64 oracle
(tests/ctc_word_beam_oracle.py) and itself: parity, spelling, resumability, batch independence, graph replay, guards and WER.

Parity cases are drawn only where the oracle's smallest keep/drop gap, and the gap between adjacent final totals, exceed 1e-3
(asserted), so that fp32 rounding cannot legitimately change which hypotheses survive.  Tolerances are K5b's."""
import os

import numpy as np
import pytest
import torch

from ctc_word_beam_oracle import NEG_INF, Words, finalize, random_lexicon, random_lm, read_back, word_beam_search, write_arpa
from oracle import nsd_oracle as O

import neural_speech_decoder_b200 as nsd
from neural_speech_decoder_b200 import _lib
from neural_speech_decoder_b200.ctc import Lexicon, NgramLM, WordBeamSearch

pytestmark = pytest.mark.gpu

DEV = "cuda"
GAP = 1e-3
TOL_REAL = 1.5e-4          # K5b's (tests/test_gpu_ctc_beam.py)


@pytest.fixture
def poisoned(monkeypatch):
    real_empty, real_empty_like = torch.empty, torch.empty_like

    def poison(t):
        if t.is_cuda and t.numel() > 0:
            if t.is_floating_point():
                t.fill_(float("nan"))
            elif t.dtype == torch.bool:
                t.fill_(True)
            else:
                t.fill_(-1 if t.dtype.is_signed else 0xFF)
        return t

    monkeypatch.setattr(torch, "empty", lambda *a, **k: poison(real_empty(*a, **k)))
    monkeypatch.setattr(torch, "empty_like", lambda *a, **k: poison(real_empty_like(*a, **k)))


def kernels_launched(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " ".join(e.name.replace(" ", "") for e in prof.events())


# ------------------------------------------------------------------------------------------------ cases
def make_case(seed, T, B, C, sep, order, tmpdir, n_words=60, blank=0, scale=5.0, ragged=True):
    """A seeded lexicon (homophones, words that prefix others), an LM of ``order`` (0: none) missing some lexicon words (they
    map to <unk>), and logits [T,B,C] that spell random words of the lexicon with separators, plus noise."""
    rng = np.random.default_rng(seed)
    phones = [c for c in range(1, C) if c not in (blank, sep)]
    pairs = random_lexicon(rng, n_words, phones, 1, 4, homophones=max(2, n_words // 8), prefixes=max(2, n_words // 8))
    lex = Lexicon.from_pronunciations(pairs, C, blank, sep)
    words = lex.words
    ngram = lm = None
    if order:
        lm = read_back(random_lm(rng, words[:len(words) - 5], order, 6 * len(words), 8 * len(words)))
        path = os.path.join(str(tmpdir), f"lm{seed}.arpa")
        write_arpa(path, lm)
        ngram = NgramLM.from_arpa(path)
    logits = rng.standard_normal((T, B, C)) * (scale * 0.5)
    for b in range(B):
        t = 0
        while t < T:
            w = int(rng.integers(len(pairs)))
            for c in list(pairs[w][1]) + [sep]:
                for _ in range(int(rng.integers(1, 3))):
                    if t < T:
                        logits[t, b, c] += scale
                        t += 1
                if t < T and rng.random() < 0.5:
                    logits[t, b, blank] += scale
                    t += 1
    lens = rng.integers(T // 2, T + 1, B)
    lens[0] = T
    if ragged and B >= 3:
        lens[1], lens[2] = 0, 1
    return logits.astype(np.float32), lens.astype(np.int64), pairs, lex, lm, ngram


def oracle_batch(logits, lens, W, pairs, sep, lm, alpha, beta, nbest, blank=0, batch=None):
    lp = O.log_softmax(logits.astype(np.float64), axis=-1)
    words = Words(pairs, sep, lm, alpha, beta)
    beams, fins, gap = [], [], np.inf
    for b in (range(lp.shape[1]) if batch is None else batch):
        beam, g = word_beam_search(lp[:, b], int(lens[b]), W, words, blank)
        fin = finalize(beam, words)
        for lst in (beam, fin):
            tot = [e[2] for e in lst[:nbest + 1] if e[2] > NEG_INF]
            g = min([g] + [x - y for x, y in zip(tot, tot[1:])])
        beams.append(beam)
        fins.append(fin)
        gap = min(gap, g)
    return beams, fins, gap


def check(out, expected, nbest, tol, rows=None):
    h, hl, w, wl = out.hyps.cpu().numpy(), out.hyp_len.cpu().numpy(), out.words.cpu().numpy(), out.word_len.cpu().numpy()
    sc, ac = out.score.cpu().numpy(), out.acoustic.cpu().numpy()
    for b, lst in zip(rows if rows is not None else range(len(expected)), expected):
        for k in range(nbest):
            if k < len(lst) and lst[k][2] > NEG_INF:
                labels, words, total, acoustic = lst[k]
                assert tuple(h[b, k, :hl[b, k]].tolist()) == labels, (b, k)
                assert tuple(w[b, k, :wl[b, k]].tolist()) == tuple(words), (b, k)
                assert abs(sc[b, k] - total) <= tol and abs(ac[b, k] - acoustic) <= tol, (b, k, sc[b, k], total)
            else:
                assert hl[b, k] == 0 and wl[b, k] == 0 and sc[b, k] == -np.inf and ac[b, k] == -np.inf, (b, k)
            assert (h[b, k, hl[b, k]:] == -1).all() and (w[b, k, wl[b, k]:] == -1).all()


def check_spelling(out, lex, final):
    """Every word hypothesis spelled through the lexicon, with sep after each completed word, is its phoneme hypothesis.  The
    phonemes after the last sep are a word only in the final read-out (the pending word); before it they have no word yet."""
    h, hl, w, wl = out.hyps.cpu().numpy(), out.hyp_len.cpu().numpy(), out.words.cpu().numpy(), out.word_len.cpu().numpy()
    for b in range(h.shape[0]):
        for k in range(h.shape[1]):
            labels = h[b, k, :hl[b, k]].tolist()
            segs, cur = [], []
            for c in labels:
                if c == lex.sep:
                    segs.append(cur)
                    cur = []
                else:
                    cur.append(c)
            if cur and final:
                segs.append(cur)
            words = w[b, k, :wl[b, k]].tolist()
            assert len(words) == len(segs), (b, k)
            for seg, wid in zip(segs, words):
                assert seg in lex.prons[wid], (b, k)


# (W, nbest, T, B, C, sep, LM order, lm_weight, word_bonus, seed): every seed's oracle gap is above GAP (asserted below)
PARITY = [
    (1, 1, 118, 6, 41, 40, 0, 0.0, 0.5, 1),
    (8, 4, 118, 6, 41, 40, 3, 0.8, 1.0, 18),
    (16, 8, 80, 4, 41, 40, 2, 0.5, -0.5, 5),
    (16, 16, 60, 3, 41, 40, 1, 1.2, 0.3, 2),
    (64, 8, 40, 3, 41, 40, 3, 0.6, 0.0, 12),
    (128, 16, 20, 3, 41, 40, 3, 0.5, 0.7, 8),
    (16, 4, 60, 4, 7, 3, 3, 0.7, 0.8, 2),
    (8, 8, 60, 4, 7, 3, 0, 0.0, -0.3, 3),
]


@pytest.mark.parametrize("W,nbest,T,B,C,sep,order,alpha,beta,seed", PARITY)
def test_parity_with_oracle(W, nbest, T, B, C, sep, order, alpha, beta, seed, tmp_path, poisoned):
    logits, lens, pairs, lex, lm, ngram = make_case(seed, T, B, C, sep, order, tmp_path)
    beams, fins, gap = oracle_batch(logits, lens, W, pairs, sep, lm, alpha, beta, nbest)
    assert gap > GAP, gap
    bs = WordBeamSearch(B, lex, ngram, W, T, alpha, beta, device=DEV)
    bs.advance(torch.from_numpy(logits).to(DEV), torch.from_numpy(lens), is_logits=True)
    raw = bs.nbest(nbest, final=False)
    fin = bs.nbest(nbest, final=True)
    check(raw, beams, nbest, TOL_REAL)
    check(fin, fins, nbest, TOL_REAL)
    check_spelling(raw, lex, False)
    check_spelling(fin, lex, True)
    assert raw.hyps.shape == (B, nbest, T) and raw.words.shape == (B, nbest, T // 2 + 1)


def test_kernels_launched(tmp_path):
    logits, lens, pairs, lex, lm, ngram = make_case(5, 30, 3, 41, 40, 3, tmp_path)
    act = torch.from_numpy(logits).to(DEV)
    names = kernels_launched(lambda: nsd.word_beam_search(act, torch.from_numpy(lens), lex, ngram, 16, 4, 0.5, 0.2, is_logits=True))
    assert "ctc_word_beam_advance_kernel" in names and "ctc_word_beam_nbest_kernel" in names and "ctc_word_beam_init_kernel" in names
    assert "ctc_beam_advance_kernel" not in names


# ------------------------------------------------------------------------------------------------ bit identity
def _bits(out):
    return [t.cpu().view(torch.int32) if t.dtype == torch.float32 else t.cpu() for t in out]


def _same(a, b):
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("W,order", [(16, 3), (128, 2), (3, 0)])
def test_chunked_alone_and_again(W, order, tmp_path):
    T, B, C = 97, 5, 41
    logits, lens, pairs, lex, lm, ngram = make_case(20 + W, T, B, C, 40, order, tmp_path)
    act = torch.from_numpy(logits).to(DEV)
    kw = dict(lm=ngram, beam_width=W, max_frames=T, lm_weight=0.6, word_bonus=-0.2, device=DEV)
    one = WordBeamSearch(B, lex, **kw)
    one.advance(act, torch.from_numpy(lens), True)
    ref = [_bits(one.nbest(W, final=f)) for f in (False, True)]
    lens_t = torch.from_numpy(lens)
    cuts = sorted(set(np.random.default_rng(W).integers(1, T, 6).tolist()))
    for splits in (list(range(1, T)), cuts):
        bs = WordBeamSearch(B, lex, **kw)
        for t0, t1 in zip([0] + splits, splits + [T]):
            bs.advance(act[t0:t1], (lens_t - t0).clamp(0, t1 - t0), True)
        for f, r in zip((False, True), ref):
            _same(_bits(bs.nbest(W, final=f)), r)
    again = WordBeamSearch(B, lex, **kw)
    again.advance(act, lens_t, True)
    _same(_bits(again.nbest(W, final=True)), ref[1])
    for b in (0, 3):
        alone = WordBeamSearch(1, lex, **kw)
        alone.advance(act[:, b:b + 1], lens_t[b:b + 1], True)
        for f, r in zip((False, True), ref):
            _same([g[0] for g in _bits(alone.nbest(W, final=f))], [x[b] for x in r])


def test_reset_utterances(tmp_path):
    T, B, C, W = 60, 4, 41, 16
    logits, lens, pairs, lex, lm, ngram = make_case(7, T, B, C, 40, 3, tmp_path, ragged=False)
    act = torch.from_numpy(logits).to(DEV)
    kw = dict(lm=ngram, beam_width=W, max_frames=T, lm_weight=0.5, word_bonus=0.1, device=DEV)
    bs = WordBeamSearch(B, lex, **kw)
    bs.advance(act[:30], is_logits=True)
    before = bs.state.clone().view(B, -1)
    mask = torch.tensor([1, 0, 1, 0], dtype=torch.int32, device=DEV)
    bs.reset_utterances(mask)
    after = bs.state.view(B, -1)
    assert torch.equal(after[1], before[1]) and torch.equal(after[3], before[3])
    bs.advance(act[30:], is_logits=True)
    got = _bits(bs.nbest(W))
    fresh = WordBeamSearch(B, lex, **kw)
    fresh.advance(act[30:], is_logits=True)
    cont = WordBeamSearch(B, lex, **kw)
    cont.advance(act, is_logits=True)
    ref_fresh, ref_cont = _bits(fresh.nbest(W)), _bits(cont.nbest(W))
    for b in range(B):
        _same([g[b] for g in got], [r[b] for r in (ref_fresh if b in (0, 2) else ref_cont)])


def test_graph_replay_equals_eager(tmp_path):
    T, B, C, W, chunk = 60, 3, 41, 16, 10
    logits, lens, pairs, lex, lm, ngram = make_case(9, T, B, C, 40, 3, tmp_path)
    act = torch.from_numpy(logits).to(DEV)
    lens_t = torch.from_numpy(lens).to(DEV).to(torch.int32)
    kw = dict(lm=ngram, beam_width=W, max_frames=T, lm_weight=0.5, word_bonus=0.3, device=DEV)
    eager = WordBeamSearch(B, lex, **kw)
    graphed = WordBeamSearch(B, lex, **kw)
    buf = torch.zeros(chunk, B, C, device=DEV)
    lbuf = torch.zeros(B, dtype=torch.int32, device=DEV)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graphed.enqueue(buf, lbuf, True)
    graphed.reset()
    for t0 in range(0, T, chunk):
        piece = act[t0:t0 + chunk]
        ln = (lens_t - t0).clamp(0, chunk)
        eager.advance(piece, ln, True)
        buf.copy_(piece)
        lbuf.copy_(ln)
        g.replay()
    for f in (False, True):
        _same(_bits(graphed.nbest(W, final=f)), _bits(eager.nbest(W, final=f)))


# ------------------------------------------------------------------------------------------------ guards
def test_guards(tmp_path):
    logits, lens, pairs, lex, lm, ngram = make_case(11, 12, 2, 41, 40, 3, tmp_path, ragged=False)
    act = torch.from_numpy(logits).to(DEV)
    with pytest.raises(nsd.NsdError):
        WordBeamSearch(2, lex, ngram, beam_width=129, device=DEV)
    with pytest.raises(nsd.NsdError):
        WordBeamSearch(2, lex, ngram, beam_width=4, device=DEV).nbest(5)
    with pytest.raises(nsd.NsdError):
        WordBeamSearch(2, lex, torch.zeros(41, 41), device=DEV)                 # K5b's bigram prior with a lexicon
    with pytest.raises(nsd.NsdError):
        nsd.word_beam_search(act, None, lex, torch.zeros(41, 41, device=DEV))
    with pytest.raises(nsd.NsdError):
        WordBeamSearch(2, lex, ngram, device=DEV).advance(torch.zeros(4, 2, 40, device=DEV))   # classes differ from the lexicon's
    with pytest.raises(ValueError):
        Lexicon.from_pronunciations([("X", [41])], 41)                          # a phone >= C
    with pytest.raises(nsd.NsdError):
        nsd.word_beam_search(act.cpu(), None, lex)
    # the raw entry point: sep == blank, sep outside [0, C), a bad lexicon size
    bs = WordBeamSearch(2, lex, ngram, beam_width=8, max_frames=10, device=DEV)
    st, sb, sc = act.stride()
    s = torch.cuda.current_stream().cuda_stream
    args = bs._model_args()

    def raw(sep, model_args=args, T=2, a=act):
        return _lib.lib().nsd_ctc_word_beam_advance(a.data_ptr(), st, sb, sc, 1, None, T, 2, 41, 0, sep, *model_args, 0.5, 0.0, 8, 10,
                                                    bs.state.data_ptr(), bs.state_bytes, bs.err_flag.data_ptr(), s)
    assert raw(0) == -1 and raw(41) == -1 and raw(-1) == -1
    assert raw(40, (args[0], 0) + args[2:]) == -1
    assert raw(40, args[:6] + (0, 0, 0)) == -1                                  # an LM without a vocabulary
    # max_frames: refused on the host; past capacity on the device the flag is set and the state is untouched
    bs.advance(act[:6], is_logits=True)
    with pytest.raises(nsd.NsdError):
        bs.advance(act[6:11], is_logits=True)
    bs.advance(act[6:10], is_logits=True)
    ref = _bits(bs.nbest(8))
    state = bs.state.clone()
    assert raw(40, T=2, a=act[10:12]) == 0
    torch.cuda.synchronize()
    assert int(bs.err_flag.item()) == 1
    assert torch.equal(bs.state, state)
    _same(_bits(bs.nbest(8)), ref)


def test_poisoned_outputs_and_zero_lengths(tmp_path, poisoned):
    logits, lens, pairs, lex, lm, ngram = make_case(13, 8, 3, 41, 40, 3, tmp_path)
    lens[:] = [8, 0, 1]
    out = nsd.word_beam_search(torch.from_numpy(logits).to(DEV), torch.from_numpy(lens), lex, ngram, 64, 64, 0.5, 0.5, is_logits=True,
                               final=False)
    for t in out:
        if t.is_floating_point():
            assert not torch.isnan(t).any()
    s = out.score.cpu().numpy()
    assert s[1, 0] == 0.0 and (s[1, 1:] == -np.inf).all() and out.hyp_len[1, 0] == 0 and out.word_len[1, 0] == 0
    n2 = int((s[2] > -np.inf).sum())
    assert n2 == 1 + int((lex.nodes[0, :4].view(np.uint32)[None, :] >> np.arange(32, dtype=np.uint32)[:, None] & 1).sum())
    assert (out.hyps[:, :, :] >= -1).all() and (out.words >= -1).all()


# ------------------------------------------------------------------------------------------------ word error rate
def levenshtein(a, b):
    d = list(range(len(b) + 1))
    for i, x in enumerate(a, 1):
        prev, d[0] = d[0], i
        for j, y in enumerate(b, 1):
            prev, d[j] = d[j], min(d[j] + 1, d[j - 1] + 1, prev + (x != y))
    return d[len(b)]


def test_word_error_rate(tmp_path):
    T, B, C, W = 100, 8, 41, 8
    logits, lens, pairs, lex, lm, ngram = make_case(17, T, B, C, 40, 3, tmp_path)
    rng = np.random.default_rng(17)
    transcripts = []
    for b in range(B):
        ws = [lex.words[i] for i in rng.integers(len(lex.words), size=int(rng.integers(0, 9)))]
        if ws and b % 2:
            ws[0] = "OUT-OF-VOCABULARY"
        transcripts.append(ws)
    ids, ilens = nsd.words_to_ids(transcripts, lex)
    assert (ids == -1).any()
    act = torch.from_numpy(logits).to(DEV)
    dec = WordBeamSearch(B, lex, ngram, W, T, 0.5, 0.5, device=DEV)
    got = nsd.word_error_rate(act, torch.from_numpy(lens), ids.to(DEV), ilens.to(DEV), dec, is_logits=True)
    top = dec.nbest(1)
    words = [top.words[b, 0, :top.word_len[b, 0]].tolist() for b in range(B)]
    want = sum(levenshtein(ids[b, :ilens[b]].tolist(), words[b]) for b in range(B))
    assert got == (want, int(ilens.sum()))
    # targets equal to the decode: no errors
    same = torch.full((B, max(1, max(len(w) for w in words))), -1, dtype=torch.int32)
    for b, w in enumerate(words):
        same[b, :len(w)] = torch.tensor(w, dtype=torch.int32)
    wl = torch.tensor([len(w) for w in words], dtype=torch.int32)
    assert nsd.word_error_rate(act, torch.from_numpy(lens), same.to(DEV), wl.to(DEV), dec, is_logits=True) == (0, int(wl.sum()))


def test_eval_batch_words_gru(tmp_path):
    from neural_speech_decoder_b200.synthetic import make_batch
    kw = dict(neural_dim=16, n_classes=6, hidden_dim=32, layer_dim=2, nDays=3, dropout=0.0, strideLen=4, kernelLen=14,
              gaussianSmoothWidth=2.0, bidirectional=True)
    torch.manual_seed(0)
    m = nsd.GRUDecoder(device="cuda", **kw).to(DEV).eval()
    X, _, X_len, _, day = make_batch(4, 80, n_feat=16, n_days=3, n_classes=6, seed=3, ragged=True, min_tgt=2, max_tgt=6, kernel_len=14,
                                     stride_len=4)
    lex = Lexicon.from_pronunciations(random_lexicon(np.random.default_rng(2), 12, [1, 2, 4, 5, 6], 1, 3, homophones=2), 7, 0, 3)
    ids, ilens = nsd.words_to_ids([lex.words[:3], lex.words[2:4], [], ["NOPE"]], lex)
    X, X_len, day = X.to(DEV), X_len.to(DEV), day.to(DEV)
    for packed in (False, True):
        dec = WordBeamSearch(4, lex, None, 8, 80, word_bonus=0.5, device=DEV)
        got = nsd.eval_batch_words(m, X, X_len, day, ids.to(DEV), ilens.to(DEV), dec, packed=packed)
        with torch.no_grad():
            logits = m.forward(X, day, X_len) if packed else m.forward(X, day)
        lens = nsd.out_lens(X_len, 14, 4)
        dec2 = WordBeamSearch(4, lex, None, 8, 80, word_bonus=0.5, device=DEV)
        want = nsd.word_error_rate(nsd.ctc.log_softmax_tbc(logits), lens, ids.to(DEV), ilens.to(DEV), dec2)
        assert got == want and got[1] == int(ilens.sum())


def test_word_error_rate_conformer_log_probs():
    kw = dict(n_channels=32, n_classes=11, n_days=3, frontend_dim=64, latent_dim=64, autoencoder_hidden_dim=32, transformer_layers=2,
              transformer_heads=4, transformer_ff_dim=128, transformer_dropout=0.0, temporal_kernel=16, temporal_stride=4)
    torch.manual_seed(0)
    m = nsd.NeuralTransformerCTCModel(device="cuda", **kw).to(DEV).eval()
    g = torch.Generator().manual_seed(4)
    X = torch.randn(3, 96, 32, generator=g).to(DEV)
    X_len = torch.tensor([96, 70, 40], dtype=torch.int32, device=DEV)
    with torch.no_grad():
        lp, olen, _ = m(X, torch.zeros(3, dtype=torch.int64, device=DEV), X_len)
    lex = Lexicon.from_pronunciations(random_lexicon(np.random.default_rng(5), 20, list(range(1, 10)), 1, 3), lp.shape[2], 0, 10)
    ids, ilens = nsd.words_to_ids([lex.words[:4], lex.words[4:6], ["NOPE"]], lex)
    dec = WordBeamSearch(3, lex, None, 16, lp.shape[0], word_bonus=1.0, device=DEV)
    got = nsd.word_error_rate(lp, olen, ids.to(DEV), ilens.to(DEV), dec)
    top = dec.nbest(1)
    want = sum(levenshtein(ids[b, :ilens[b]].tolist(), top.words[b, 0, :top.word_len[b, 0]].tolist()) for b in range(3))
    assert got == (want, int(ilens.sum()))


# ------------------------------------------------------------------------------------------------ realistic size
def big_lm(rng, words, n2, n3):
    """A seeded 3-gram of about n2 + n3 entries over ``words``, built vectorised (log10 values, as random_lm)."""
    vocab = ["<s>", "</s>", "<unk>"] + list(words)
    V = len(vocab)
    lm = {(w,): (float(-rng.uniform(1.0, 5.0)) if w != "<s>" else -99.0, float(-rng.uniform(0.0, 1.0))) for w in vocab}
    pairs = np.unique(np.stack([np.where(rng.random(n2) < 0.05, 0, rng.integers(2, V, n2)), rng.integers(1, V, n2)], 1), axis=0)
    pairs = pairs[pairs[:, 0] != 1]
    p2, b2 = -rng.uniform(0.1, 3.0, len(pairs)), -rng.uniform(0.0, 1.0, len(pairs))
    for (a, w), p, bo in zip(pairs.tolist(), p2.tolist(), b2.tolist()):
        lm[(vocab[a], vocab[w])] = (round(p, 6), round(bo, 6))
    hist = pairs[pairs[:, 1] != 1]
    pick = hist[rng.integers(len(hist), size=n3)]
    tri = np.unique(np.concatenate([pick, rng.integers(1, V, (n3, 1))], 1), axis=0)
    for (a, b, w), p in zip(tri.tolist(), (-rng.uniform(0.05, 2.5, len(tri))).tolist()):
        lm[(vocab[a], vocab[b], vocab[w])] = (round(p, 6), 0.0)
    return {k: (round(v[0], 6), round(v[1], 6)) for k, v in lm.items()}


def test_realistic_size(tmp_path):
    """20 k words, a 3-gram of about 500 k entries, B=64, T'=118, W=16: the top hypotheses match the oracle where the gap allows."""
    rng = np.random.default_rng(2024)
    T, B, C, W = 118, 64, 41, 16
    pairs = random_lexicon(rng, 20000, list(range(1, 40)), 2, 8, homophones=500, prefixes=500)
    lex = Lexicon.from_pronunciations(pairs, C)
    lm = big_lm(rng, lex.words[:19000], 250000, 250000)
    assert 450000 < len(lm) < 550000
    path = str(tmp_path / "big.arpa")
    write_arpa(path, lm)
    ngram = NgramLM.from_arpa(path)
    logits = rng.standard_normal((T, B, C)) * 2.5
    for b in range(B):
        t = 0
        while t < T:
            for c in list(pairs[int(rng.integers(len(pairs)))][1]) + [40]:
                for _ in range(int(rng.integers(1, 3))):
                    if t < T:
                        logits[t, b, c] += 5.0
                        t += 1
    logits = logits.astype(np.float32)
    lens = rng.integers(100, T + 1, B)
    lens[0] = T
    out = nsd.word_beam_search(torch.from_numpy(logits).to(DEV), torch.from_numpy(lens), lex, ngram, W, 4, 0.8, 0.5, is_logits=True)
    check_spelling(out, lex, True)
    rows = list(range(16))
    words = Words(pairs, 40, lm, 0.8, 0.5)
    lp = O.log_softmax(logits.astype(np.float64), axis=-1)
    checked = 0
    for b in rows:
        beam, gap = word_beam_search(lp[:, b], int(lens[b]), W, words)
        fin = finalize(beam, words)
        tot = [e[2] for e in fin[:2] if e[2] > NEG_INF]
        if gap > GAP and (len(tot) < 2 or tot[0] - tot[1] > GAP):
            check(out, [fin], 1, TOL_REAL, rows=[b])
            checked += 1
    assert checked >= 4, checked
