"""K5b CTC prefix beam search (``nsd_ctc_beam_*``, ``CtcBeamSearch``, ``ctc_beam_search``) against the float64 oracle
(tests/ctc_beam_oracle.py), the exact CTC probability and itself: resumability, batch independence, guards, the PER path
and streaming.

Parity cases are drawn only where the oracle's smallest keep/drop score gap exceeds 1e-3 (asserted), so that fp32
rounding cannot legitimately change which hypotheses survive.  The ``poisoned`` fixture fills fresh CUDA allocations with
NaN / all-ones bits, so output rows the kernels fail to write show up."""
import numpy as np
import pytest
import torch

from ctc_beam_oracle import ctc_prefix_beam_search, prior_of
from oracle import nsd_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200 import _lib
    from neural_speech_decoder_b200.ctc import CtcBeamSearch, ctc_beam_search

DEV = "cuda"
GAP = 1e-3
# |kernel - oracle| of total / acoustic, ≈3x the worst measured on a B200: 4.6e-5 over the realistic cases (scores up to
# |190|, where 1 ulp is 1.5e-5) and 1.9e-6 over the exhaustive ones (scores below |12|)
TOL_REAL = 1.5e-4
TOL_SMALL = 6e-6


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


def make_case(seed, T, B, C, blank, ragged=True, scale=6.0):
    """Logits [T,B,C] f32 shaped like a trained decoder's (blank-heavy, peaky), ragged lengths including 0 and 1, and a
    bigram table [C,C] of log-probs."""
    rng = np.random.default_rng(seed)
    logits = rng.standard_normal((T, B, C)) * scale
    logits[:, :, blank] += 2.0
    lens = rng.integers(T // 2, T + 1, B)
    lens[0] = T
    if ragged and B >= 3:
        lens[1], lens[2] = 0, 1
    lm = O.log_softmax(rng.standard_normal((C, C)) * 1.5)
    return logits.astype(np.float32), lens.astype(np.int64), lm.astype(np.float32)


def oracle_batch(lp, lens, W, blank, lm, alpha, beta, nbest=1):
    """lp: float64 [T,B,C] -> (per-utterance beams, smallest gap over the batch that decides the first ``nbest``: keep/drop
    at every frame and adjacent totals among the first nbest + 1 final entries)."""
    res = [ctc_prefix_beam_search(lp[:, b], int(lens[b]), W, blank, lm if alpha != 0.0 else None, alpha, beta) for b in range(lp.shape[1])]
    gap = min(r[1] for r in res)
    for beam, _ in res:
        tot = [t for _, t, _ in beam[:nbest + 1]]
        gap = min([gap] + [a - b for a, b in zip(tot, tot[1:])])
    return [r[0] for r in res], gap


def as_lists(hyps, hyp_len):
    h, l = hyps.cpu().numpy(), hyp_len.cpu().numpy()
    return [[tuple(h[b, k, :l[b, k]].tolist()) for k in range(h.shape[1])] for b in range(h.shape[0])]


def check_against_oracle(out, beams, nbest, tol):
    hyps, hyp_len, score, acoustic = out
    got = as_lists(hyps, hyp_len)
    score, acoustic = score.cpu().numpy(), acoustic.cpu().numpy()
    h = hyps.cpu().numpy()
    for b, beam in enumerate(beams):
        for k in range(nbest):
            if k < len(beam):
                labels, total, ac = beam[k]
                assert got[b][k] == labels, (b, k)
                assert abs(score[b, k] - total) <= tol and abs(acoustic[b, k] - ac) <= tol, (b, k, score[b, k], total)
                assert (h[b, k, len(labels):] == -1).all()
            else:
                assert got[b][k] == () and score[b, k] == -np.inf and acoustic[b, k] == -np.inf


# ---------------------------------------------------------------------------------------------------- exhaustive cases
@pytest.mark.parametrize("C,T", [(4, T) for T in range(1, 5)] + [(3, T) for T in range(1, 7)])
def test_exhaustive(C, T, poisoned):
    rng = np.random.default_rng(10 * C + T)
    B = 3
    lp = np.stack([O.log_softmax(rng.standard_normal((T, C)) * 2.0) for _ in range(B)], axis=1).astype(np.float32)
    lm = O.log_softmax(rng.standard_normal((C, C))).astype(np.float32)
    alpha, beta = 0.6, 0.3
    lp_d = torch.from_numpy(lp).to(DEV)
    lens = torch.full((B,), T, dtype=torch.int32, device=DEV)
    out = ctc_beam_search(lp_d, lens, 128, 128, 0, torch.from_numpy(lm), alpha, beta)
    beams, _ = oracle_batch(lp.astype(np.float64), [T] * B, 128, 0, lm.astype(np.float64), alpha, beta)
    check_against_oracle(out, beams, 128, TOL_SMALL)
    # acoustic = the exact CTC log-probability of the labels, as torch computes it
    hyps, hyp_len, score, acoustic = out
    lists = as_lists(hyps, hyp_len)
    for b in range(B):
        seqs = lists[b][:len(beams[b])]
        tgt = torch.zeros((len(seqs), max(1, T)), dtype=torch.int64)
        for i, s in enumerate(seqs):
            tgt[i, :len(s)] = torch.tensor(s, dtype=torch.int64)
        nll = torch.nn.CTCLoss(blank=0, reduction="none", zero_infinity=False)(
            torch.from_numpy(lp[:, b:b + 1].astype(np.float64)).expand(T, len(seqs), C).contiguous(), tgt,
            torch.full((len(seqs),), T, dtype=torch.int64), torch.tensor([len(s) for s in seqs]))
        ac = acoustic[b, :len(seqs)].cpu().double()
        assert torch.allclose(ac, -nll, atol=TOL_SMALL, rtol=0)
        for i, s in enumerate(seqs):
            assert abs(score[b, i].item() - (ac[i].item() + prior_of(s, 0, lm, alpha, beta))) <= TOL_SMALL


# ---------------------------------------------------------------------------------------------------- realistic parity
# (W, nbest, T, B, prior, blank, input form, seed).  Near-ties get denser with the width and the number of frames, so the
# widest beams run shorter inputs; every seed gives an oracle gap above 2e-3 (asserted > GAP below).  "_btc": a permuted
# view of a [B,T,C] buffer.  B >= 3 carries lengths 0 and 1.
PARITY = [
    (1, 1, 118, 8, False, 0, "lp", 1),
    (4, 4, 118, 8, True, 0, "logits_btc", 1),
    (16, 1, 60, 4, True, 0, "lp", 1),
    (16, 16, 40, 3, False, 7, "logits", 2),
    (16, 1, 118, 1, True, 0, "logits", 6),
    (64, 4, 24, 3, True, 0, "lp_btc", 5),
    (64, 64, 16, 3, False, 0, "logits", 59),
    (128, 4, 16, 3, True, 0, "lp", 1),
    (128, 1, 16, 3, False, 0, "logits_btc", 24),
    (128, 128, 6, 3, True, 0, "logits", 1406),
]


def parity_inputs(W, T, B, prior, blank, form, seed, C=41):
    logits, lens, lm = make_case(seed, T, B, C, blank)
    lp = np.asarray(O.log_softmax(logits.astype(np.float64), axis=-1), dtype=np.float32)
    alpha, beta = (0.5, 0.8) if prior else (0.0, 0.0)
    src = lp if form.startswith("lp") else logits
    if form.endswith("btc"):
        act = torch.from_numpy(np.ascontiguousarray(src.transpose(1, 0, 2))).to(DEV).permute(1, 0, 2)   # a [B,T,C] buffer
    else:
        act = torch.from_numpy(src).to(DEV)
    lp64 = O.log_softmax(logits.astype(np.float64), axis=-1) if not form.startswith("lp") else lp.astype(np.float64)
    return act, lens, lm, alpha, beta, lp64, not form.startswith("lp")


@pytest.mark.parametrize("W,nbest,T,B,prior,blank,form,seed", PARITY)
def test_parity_with_oracle(W, nbest, T, B, prior, blank, form, seed, poisoned):
    C = 41
    act, lens, lm, alpha, beta, lp64, is_logits = parity_inputs(W, T, B, prior, blank, form, seed, C)
    beams, gap = oracle_batch(lp64, lens, W, blank, lm.astype(np.float64), alpha, beta, nbest)
    assert gap > GAP, gap
    out = ctc_beam_search(act, torch.from_numpy(lens).to(DEV), W, nbest, blank, torch.from_numpy(lm) if prior else None, alpha, beta,
                          is_logits=is_logits)
    check_against_oracle(out, beams, nbest, TOL_REAL)
    assert out[0].shape == (B, nbest, T)


def test_advance_kernel_runs():
    act, lens, lm, alpha, beta, _, _ = parity_inputs(16, 20, 2, True, 0, "lp", 11)
    names = kernels_launched(lambda: ctc_beam_search(act, torch.from_numpy(lens).to(DEV), 16, 4, 0, torch.from_numpy(lm), alpha, beta))
    assert "ctc_beam_advance_kernel" in names and "ctc_beam_nbest_kernel" in names and "ctc_beam_init_kernel" in names


# ---------------------------------------------------------------------------------------------------- bit identity
def _bits(out):
    return [t.cpu() for t in out]


def _same(a, b):
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x, y.view(torch.int32) if y.dtype == torch.float32 else y)


@pytest.mark.parametrize("W,is_logits", [(16, False), (128, True), (3, True)])
def test_chunked_equals_one_call(W, is_logits):
    T, B, C = 97, 5, 41
    logits, lens, lm = make_case(20 + W, T, B, C, 0)
    act = torch.from_numpy(logits).to(DEV)
    if not is_logits:
        act = act.log_softmax(-1)
    lm_d = torch.from_numpy(lm).to(DEV)
    kw = dict(blank=0, lm=lm_d, lm_weight=0.4, insertion_bonus=-0.2, device=DEV)
    one = CtcBeamSearch(B, C, W, T, **kw)
    one.advance(act, torch.from_numpy(lens), is_logits)
    ref = _bits(one.nbest(W))
    lens_t = torch.from_numpy(lens)
    rng = np.random.default_rng(W)
    cuts = sorted(set(rng.integers(1, T, 6).tolist()))
    for splits in (list(range(1, T)), cuts):
        bs = CtcBeamSearch(B, C, W, T, **kw)
        for t0, t1 in zip([0] + splits, splits + [T]):
            bs.advance(act[t0:t1], (lens_t - t0).clamp(0, t1 - t0), is_logits)
        _same(_bits(bs.nbest(W)), ref)
    # and again: a second run of the same call gives the same bits
    again = CtcBeamSearch(B, C, W, T, **kw)
    again.advance(act, lens_t, is_logits)
    _same(_bits(again.nbest(W)), ref)
    # an utterance of the ragged batch equals the same utterance decoded alone
    for b in (0, 3):
        alone = CtcBeamSearch(1, C, W, T, **kw)
        alone.advance(act[:, b:b + 1], lens_t[b:b + 1], is_logits)
        got = _bits(alone.nbest(W))
        _same([g[0] for g in got], [r[b] for r in ref])


def test_zero_weight_table_equals_no_table():
    T, B, C = 50, 4, 41
    logits, lens, lm = make_case(31, T, B, C, 0)
    act = torch.from_numpy(logits).to(DEV)
    a = ctc_beam_search(act, torch.from_numpy(lens).to(DEV), 16, 16, is_logits=True)
    b = ctc_beam_search(act, torch.from_numpy(lens).to(DEV), 16, 16, lm=torch.from_numpy(lm), lm_weight=0.0, insertion_bonus=0.0, is_logits=True)
    _same(_bits(a), _bits(b))


# ---------------------------------------------------------------------------------------------------- order, padding, guards
def test_order_and_padding(poisoned):
    T, B, C = 6, 3, 5
    logits, lens, _ = make_case(41, T, B, C, 0)
    lens[:] = [6, 0, 1]
    hyps, hyp_len, score, acoustic = ctc_beam_search(torch.from_numpy(logits).to(DEV), torch.from_numpy(lens).to(DEV), 64, 64, is_logits=True)
    lists = as_lists(hyps, hyp_len)
    s = score.cpu().numpy()
    for b in range(B):
        n = int((s[b] > -np.inf).sum())
        assert (np.diff(s[b, :n]) <= 0).all()
        assert len(set(lists[b][:n])) == n
        assert (s[b, n:] == -np.inf).all() and (hyp_len[b, n:] == 0).all() and (acoustic[b, n:] == -np.inf).all()
        assert (hyps[b, n:] == -1).all()
    assert lists[1][0] == () and s[1, 0] == 0.0 and int((s[1] > -np.inf).sum()) == 1      # len 0: the empty hypothesis
    assert int((s[2] > -np.inf).sum()) == C                                                # len 1: empty + every label


def test_bounds():
    act = torch.zeros(4, 2, 41, device=DEV)
    lens = torch.full((2,), 4, device=DEV)
    with pytest.raises(nsd.NsdError):
        ctc_beam_search(act, lens, beam_width=129)
    with pytest.raises(nsd.NsdError):
        ctc_beam_search(torch.zeros(4, 2, 129, device=DEV), lens)
    with pytest.raises(nsd.NsdError):
        ctc_beam_search(act, lens, beam_width=4, nbest=5)
    with pytest.raises(nsd.NsdError):
        ctc_beam_search(act.cpu(), lens.cpu())
    with pytest.raises(nsd.NsdError):
        CtcBeamSearch(2, 41, 4, 10, device=DEV).nbest(5)
    with pytest.raises(nsd.NsdError):
        CtcBeamSearch(2, 41, 4, 10, device="cpu")


def test_max_frames_overflow():
    T, B, C = 12, 2, 41
    logits, _, _ = make_case(51, T, B, C, 0)
    act = torch.from_numpy(logits).to(DEV)
    bs = CtcBeamSearch(B, C, 8, 10, device=DEV)
    bs.advance(act[:6], is_logits=True)
    with pytest.raises(nsd.NsdError):
        bs.advance(act[6:11], is_logits=True)      # 6 + 5 > 10: refused on the host, nothing launched
    bs.advance(act[6:10], is_logits=True)
    ref = _bits(bs.nbest(8))
    state = bs.state.clone()
    # the raw entry point past capacity: the flag is set and the state (beam and trie) is untouched
    a = act[10:12]
    st, sb, sc = a.stride()
    _lib.call("nsd_ctc_beam_advance", a.data_ptr(), st, sb, sc, 1, None, 2, B, C, 0, None, 0.0, 0.0, 8, 10, bs.state.data_ptr(),
              bs.state_bytes, bs.err_flag.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert int(bs.err_flag.item()) == 1
    assert torch.equal(bs.state, state)
    _same(_bits(bs.nbest(8)), ref)


# ---------------------------------------------------------------------------------------------------- PER path
@pytest.mark.parametrize("W,prior,seed", [(8, False, 13), (4, True, 1)])
def test_phoneme_error_rate_with_beam(W, prior, seed):
    T, B, C = 100, 8, 41
    logits, lens, lm = make_case(seed, T, B, C, 0)
    lp = torch.from_numpy(logits).to(DEV).log_softmax(-1)
    rng = np.random.default_rng(seed)
    y = rng.integers(1, C, (B, 30)).astype(np.int32)
    y_len = rng.integers(5, 30, B).astype(np.int32)
    args = (lp, torch.from_numpy(lens).to(DEV), torch.from_numpy(y).to(DEV), torch.from_numpy(y_len).to(DEV))
    greedy = nsd.phoneme_error_rate(*args)
    dec, dec_len = nsd.greedy_decode(*args[:2])
    assert greedy == nsd.phoneme_error_rate(*args, beam_width=None)
    assert greedy == O.phoneme_error_rate(nsd.decoded_to_lists(dec, dec_len), y, y_len)
    a, b = (0.5, 0.8) if prior else (0.0, 0.0)
    got = nsd.phoneme_error_rate(*args, beam_width=W, lm=torch.from_numpy(lm) if prior else None, lm_weight=a, insertion_bonus=b)
    beams, gap = oracle_batch(lp.double().cpu().numpy(), lens, W, 0, lm.astype(np.float64), a, b)
    assert gap > GAP, gap
    assert got == O.phoneme_error_rate([list(bm[0][0]) for bm in beams], y, y_len)


# ---------------------------------------------------------------------------------------------------- streaming
SMALL = dict(neural_dim=64, n_classes=40, hidden_dim=512, layer_dim=2, nDays=4, strideLen=4, kernelLen=32, gaussianSmoothWidth=2.0)


def _stream_model():
    from test_gpu_streaming import build
    return build(**SMALL)


def _stream_run(sd, X, chunks):
    outs, pos = [], 0
    for n in chunks:
        o = sd.push(X[:, pos:pos + n])
        pos += n
        if o is not None:
            outs.append(o)
    o = sd.finish()
    if o is not None:
        outs.append(o)
    return torch.cat(outs, dim=1)


@pytest.mark.parametrize("B,fast,use_graph", [(1, False, False), (5, False, False), (1, True, False), (1, True, True), (5, True, True)])
def test_streaming_hypotheses(B, fast, use_graph):
    m = _stream_model()
    C = SMALL["n_classes"] + 1
    lm = torch.from_numpy(O.log_softmax(np.random.default_rng(B).standard_normal((C, C))).astype(np.float32))
    g = torch.Generator().manual_seed(B)
    day = torch.randint(0, SMALL["nDays"], (B,), generator=g).to(DEV)
    kw = dict(beam_width=16, nbest=4, lm=lm, lm_weight=0.3, insertion_bonus=0.5, max_frames=512)
    sd = nsd.StreamingDecoder(m, B, day, fast=fast, use_graph=use_graph, **kw)
    for T in (200, 230):                          # a second utterance after reset()
        X = torch.randn(B, T, SMALL["neural_dim"], generator=g).to(DEV)
        # steady one-stride pushes, one irregular push in the middle (leaves and re-enters the fast form), steady again
        chunks = [44] + [4] * 20 + [7] + [4] * 12
        chunks.append(T - sum(chunks))
        logits = _stream_run(sd, X, chunks)
        if fast:
            assert sd._graph is not None or not use_graph
        ref = ctc_beam_search(logits.permute(1, 0, 2), None, 16, 4, 0, lm, 0.3, 0.5, is_logits=True)
        got = sd.hypotheses()
        assert got[0].shape == (B, 4, 512)
        _same([r.cpu() for r in ref[1:]], [x.cpu() for x in got[1:]])
        _same([ref[0].cpu()], [got[0][:, :, :logits.shape[1]].cpu()])
        assert (got[0][:, :, logits.shape[1]:] == -1).all()
        sd.reset()


def test_streaming_fast_form_launches_the_beam():
    m = _stream_model()
    sd = nsd.StreamingDecoder(m, 1, torch.zeros(1, dtype=torch.int64, device=DEV), fast=True, use_graph=False, beam_width=16)
    X = torch.randn(1, 64, SMALL["neural_dim"], device=DEV)
    for pos in range(0, 60, 4):
        sd.push(X[:, pos:pos + 4])
    assert sd._steady
    names = kernels_launched(lambda: sd.push_decode(X[:, 60:64].cpu()))
    assert "ctc_beam_advance_kernel" in names and "stream_push_kernel" in names


def test_streaming_max_frames():
    m = _stream_model()
    sd = nsd.StreamingDecoder(m, 1, torch.zeros(1, dtype=torch.int64, device=DEV), beam_width=4, max_frames=3)
    X = torch.randn(1, 64, SMALL["neural_dim"], device=DEV)
    sd.push(X[:, :48])                             # frames 0..1
    with pytest.raises(nsd.NsdError):
        sd.push(X[:, 48:64])                       # 4 more frames: refused before anything runs
    assert sd.next_frame == 2


def test_streaming_without_beam_is_unchanged():
    m = _stream_model()
    sd = nsd.StreamingDecoder(m, 1, torch.zeros(1, dtype=torch.int64, device=DEV))
    assert sd._beam is None
    with pytest.raises(nsd.NsdError):
        sd.hypotheses()
    X = torch.randn(1, 64, SMALL["neural_dim"], device=DEV)
    for pos in range(0, 64, 4):
        sd.push(X[:, pos:pos + 4])
    assert sd._steady
    names = kernels_launched(lambda: sd.push(torch.randn(1, 4, SMALL["neural_dim"], device=DEV)))
    assert "ctc_beam" not in names
