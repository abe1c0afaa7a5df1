"""Live word decoding in streaming: the word beam (K5d) inside StreamingDecoder and StreamingSessions, and its live read-out
(``nsd_ctc_word_beam_live``, ``WordBeamSearch.enqueue_live``): committed and tentative words after every push.

The streamed word N-best must be the bits of a ``WordBeamSearch`` advanced over the logits the stream returned; the committed
words after every push must be the longest common word-id prefix of the live hypotheses (computed here on the host from the
full N-best), never change once given, and prefix the final top hypothesis; the tentative words are the top hypothesis's
words after them.  The lexicon gives some words five one-phone pronunciations (and some homophones), so live hypotheses often
hold the same words on different word-trie nodes: the read-out must compare words, not nodes."""
import ctypes
import os
import random

import numpy as np
import pytest
import torch

from ctc_word_beam_oracle import random_lexicon, random_lm, read_back, write_arpa
from test_gpu_stream_sessions import ARCHS, build, make_utterances, run_schedule

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200.ctc import Lexicon, NgramLM, WordBeamSearch

DEV = "cuda"
W = 16
WORD_KW = dict(beam_width=W, nbest=W, lm_weight=0.5, word_bonus=2.0)


def sep_of(arch):
    return ARCHS[arch]["n_classes"]              # the last class: 40 = SIL for the competition's 41 classes


_MODELS, _WORDS = {}, {}


def model(arch):
    if arch not in _MODELS:
        _MODELS[arch] = build(**ARCHS[arch])
    return _MODELS[arch]


def words_for(arch, tmp_dir):
    """(lexicon, 3-gram NgramLM) over the model's classes: the non-separator phones in groups of five, each group the one-phone
    pronunciations of one word (G0, G1, ...), three homophones of those, and 30 words of two or three phones."""
    if arch not in _WORDS:
        C, sep = ARCHS[arch]["n_classes"] + 1, sep_of(arch)
        rng = np.random.default_rng(C)
        phones = [c for c in range(1, C) if c != sep]
        pairs = [(f"G{i // 5}", [c]) for i, c in enumerate(phones)]
        pairs += [(f"H{k}", [phones[5 * k]]) for k in range(3)]
        pairs += random_lexicon(rng, 30, phones, 2, 3)
        lex = Lexicon.from_pronunciations(pairs, C, 0, sep)
        path = os.path.join(str(tmp_dir), f"stream_words_{arch}.arpa")
        write_arpa(path, read_back(random_lm(rng, lex.words, 3, 300, 400)))
        _WORDS[arch] = (lex, NgramLM.from_arpa(path))
    return _WORDS[arch]


def bits(out):
    return [t.cpu().view(torch.int32) if t.dtype == torch.float32 else t.cpu() for t in out]


def same(a, b, what=""):
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), f"{what} field {i}"


def offline(lex, lm, logits_tbc, max_frames):
    """A WordBeamSearch advanced over the logits a stream returned ([T', B, C])."""
    bs = WordBeamSearch(logits_tbc.shape[1], lex, lm, W, max_frames, WORD_KW["lm_weight"], WORD_KW["word_bonus"], device=DEV)
    bs.advance(logits_tbc, None, True)
    return bs


class LiveCheck:
    """Checks one transcript against the N-best of the same beam, and keeps what the checks found."""

    def __init__(self, lex):
        self.lex, self.given, self.pushes_with_committed, self.twins = lex, {}, 0, 0

    def __call__(self, key, transcript, hyps):
        committed, tentative = transcript
        hl, wl = hyps.hyp_len.cpu().tolist(), hyps.word_len.cpu().tolist()
        h, w, sc = hyps.hyps.cpu().numpy(), hyps.words.cpu().numpy(), hyps.score.cpu().numpy()
        live = [k for k in range(len(sc)) if np.isfinite(sc[k])]
        seqs = [tuple(w[k, :wl[k]].tolist()) for k in live]
        lcp = 0
        while seqs and all(len(s) > lcp and s[lcp] == seqs[0][lcp] for s in seqs):
            lcp += 1
        names, prev = self.lex.words, self.given.get(key, [])
        assert committed == ([names[i] for i in seqs[0][:lcp]] if seqs else prev), key
        assert committed[:len(prev)] == prev, f"{key}: committed words changed"
        self.given[key] = list(committed)
        assert tentative == ([names[i] for i in seqs[0][lcp:]] if seqs else []), key
        self.pushes_with_committed += bool(committed)
        # live hypotheses with the same words spelled by different phonemes up to their last separator: different word-trie nodes
        spelled = []
        for k in live:
            p = h[k, :hl[k]].tolist()
            cut = max([i + 1 for i, c in enumerate(p) if c == self.lex.sep], default=0)
            spelled.append(tuple(p[:cut]))
        self.twins += sum(seqs[i] == seqs[j] and spelled[i] != spelled[j] for i in range(len(live)) for j in range(i))

    def final(self, key, committed, fin):
        """The committed words prefix the final top hypothesis (when it has a finite score)."""
        if np.isfinite(float(fin.score[0])):
            top = [self.lex.words[i] for i in fin.words[0, :int(fin.word_len[0])].tolist()]
            assert top[:len(committed)] == committed, key


# ------------------------------------------------------------------------------------------------ StreamingDecoder
def decode_stream(sd, X, chunks, check, B, tag):
    """Push ``chunks`` of X [B, T, N] (push, or push_decode on steady one-stride pushes), check the transcript of every row after
    each push and after finish -> the logits the stream returned, [B, T', C]."""
    outs, pos, S = [], 0, sd.S
    rng = random.Random(len(chunks))
    for n in chunks:
        bins = X[:, pos:pos + n]
        pos += n
        if sd._steady and n == S and rng.random() < 0.5:
            sd.push_decode(bins.cpu().pin_memory())
            outs.append(sd._logits_host.clone().unsqueeze(1).to(DEV))
        else:
            o = sd.push(bins)
            if o is not None:
                outs.append(o)
        hyps = sd.hypotheses()
        for r in range(B):
            check((tag, r), sd.transcript(r), type(hyps)(*(t[r] for t in hyps)))
    o = sd.finish()
    if o is not None:
        outs.append(o)
    hyps = sd.hypotheses()
    fin = sd.hypotheses(final=True)
    for r in range(B):
        t = sd.transcript(r)
        check((tag, r), t, type(hyps)(*(x[r] for x in hyps)))
        check.final((tag, r), t[0], type(fin)(*(x[r] for x in fin)))
    return torch.cat(outs, dim=1)


@pytest.mark.parametrize("arch,B,fast,use_graph", [
    ("small", 1, False, False), ("small", 3, False, False), ("small", 1, True, True), ("small", 3, True, False),
    ("comp", 3, True, True), ("comp", 1, True, False),
])
def test_decoder_equals_offline(arch, B, fast, use_graph, tmp_path):
    m = model(arch)
    lex, lm = words_for(arch, tmp_path)
    K, S, N = m.kernelLen, m.strideLen, m.neural_dim
    g = torch.Generator().manual_seed(B * 7 + int(fast))
    day = torch.randint(0, ARCHS[arch]["nDays"], (B,), generator=g).to(DEV)
    sd = nsd.StreamingDecoder(m, B, day, fast=fast, use_graph=use_graph, lexicon=lex, lm=lm, max_frames=512, **WORD_KW)
    check = LiveCheck(lex)
    for T in (260, 301):                                    # a second utterance after reset()
        X = torch.randn(B, T, N, generator=g).to(DEV)
        if fast:                                            # steady pushes, one irregular push (leaves the fast form), steady again
            chunks = [K + 4 * S] + [S] * 25 + [S + 2] + [S] * 15
        else:
            r = random.Random(T)
            chunks = [r.choice([1, 2, S, 5, 11, 17]) for _ in range(60)]
        chunks = [c for c in chunks if c > 0]
        while sum(chunks) > T:
            chunks.pop()
        chunks.append(T - sum(chunks))
        logits = decode_stream(sd, X, chunks, check, B, T)
        if fast:
            assert sd._graph is not None or not use_graph
        ref = offline(lex, lm, logits.permute(1, 0, 2), 512)
        for f in (False, True):
            same(bits(ref.nbest(W, final=f)), bits(sd.hypotheses(final=f)), f"final={f}")
        sd.reset()
        assert sd.transcript(0) == ([], [])
    assert check.pushes_with_committed > 0 and check.twins > 0, (check.pushes_with_committed, check.twins)


# ------------------------------------------------------------------------------------------------ StreamingSessions
class CheckedSessions(nsd.StreamingSessions if torch.cuda.is_available() else object):
    """StreamingSessions that checks every open slot's transcript after every push and at every finish."""

    def __init__(self, *a, check=None, **kw):
        super().__init__(*a, **kw)
        self.check, self.sessions, self.key = check, 0, {}

    def _check_open(self):
        for s in range(self.slots):
            if self._open[s]:
                self.check(self.key[s], self.transcript(s), self.hypotheses(s))

    def open(self, slot, day):
        super().open(slot, day)
        self.sessions += 1
        self.key[slot] = (id(self), self.sessions)

    def push(self, bins, active):
        out = super().push(bins, active)
        self._check_open()
        return out

    def push_decode(self, bins, active):
        ids = super().push_decode(bins, active).clone()
        self._check_open()
        return ids

    def finish(self, slot, tail):
        out = super().finish(slot, tail)
        t = self.transcript(slot)
        self.check(self.key[slot], t, self.hypotheses(slot))
        self.check.final(self.key[slot], t[0], self.hypotheses(slot, final=True))
        return out


def sessions_run(arch, slots, use_graph, utts, tmp_path, seed):
    """run_schedule with every transcript checked -> (sessions, {utterance: (transcript, raw N-best bits, final N-best bits)}
    read right after its finish, the checker)."""
    m = model(arch)
    lex, lm = words_for(arch, tmp_path)
    check = LiveCheck(lex)
    ss = CheckedSessions(m, slots, use_graph=use_graph, lexicon=lex, lm=lm, max_frames=256, check=check, **WORD_KW)
    done = {}

    def read(u, s):
        done[u] = (ss.transcript(s), bits(ss.hypotheses(s)), bits(ss.hypotheses(s, final=True)))
    run_schedule(ss, m, utts, seed=seed, decode_share=0.4, on_finish=read)
    if use_graph:
        assert ss._graph is not None, getattr(ss, "_graph_error", "no graph captured")
    assert sorted(done) == list(range(len(utts)))
    return done, check


def alone(arch, X, day, tmp_path):
    """The session streamed alone through one slot -> (transcript, raw N-best bits, final N-best bits, logits)."""
    m = model(arch)
    lex, lm = words_for(arch, tmp_path)
    ss = nsd.StreamingSessions(m, 1, lexicon=lex, lm=lm, max_frames=256, **WORD_KW)
    S = m.strideLen
    ss.open(0, day)
    outs, pos = [], 0
    while X.shape[0] - pos >= S:
        lg, em = ss.push(X[pos:pos + S].unsqueeze(0).to(DEV), [True])
        pos += S
        if bool(em[0]):
            outs.append(lg[0:1])
    outs.append(ss.finish(0, X[pos:].to(DEV)))
    return ss.transcript(0), bits(ss.hypotheses(0)), bits(ss.hypotheses(0, final=True)), torch.cat(outs)


@pytest.mark.parametrize("arch,slots,use_graph", [("comp", 4, True), ("small", 3, False), ("small", 5, True)])
def test_sessions_equal_alone(arch, slots, use_graph, tmp_path):
    utts = make_utterances(ARCHS[arch], 9, seed=11 + slots)
    done, check = sessions_run(arch, slots, use_graph, utts, tmp_path, seed=slots)
    lex, lm = words_for(arch, tmp_path)
    refs = [alone(arch, X, d, tmp_path) for X, d in utts]
    for u, (t, raw, fin) in done.items():
        assert t == refs[u][0], f"utterance {u}: transcript"
        same(raw + fin, refs[u][1] + refs[u][2], f"utterance {u}")
    for _, raw, fin, logits in refs:                         # and the alone runs equal the offline word beam on their logits
        ref = offline(lex, lm, logits.unsqueeze(1), 256)
        same([x[0] for x in bits(ref.nbest(W, final=False))], raw, "raw")
        same([x[0] for x in bits(ref.nbest(W, final=True))], fin, "final")
    assert check.pushes_with_committed > 0 and check.twins > 0, (check.pushes_with_committed, check.twins)


def _poison(monkeypatch):
    """torch.empty / torch.empty_like return CUDA tensors filled with NaN (floating) or all-ones bits (integer)."""
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


def test_poisoned_buffers(tmp_path, monkeypatch):
    """Every fresh CUDA allocation NaN / all-ones: the sessions' transcripts and N-best lists, and a decoder's, are unchanged."""
    arch = "small"
    utts = make_utterances(ARCHS[arch], 5, seed=3)
    m = model(arch)
    lex, lm = words_for(arch, tmp_path)
    X = torch.randn(2, 70 * m.strideLen, m.neural_dim, generator=torch.Generator().manual_seed(1)).to(DEV)

    def run():
        done, _ = sessions_run(arch, 3, True, utts, tmp_path, seed=4)
        sd = nsd.StreamingDecoder(m, 2, torch.tensor([0, 2], device=DEV), lexicon=lex, lm=lm, max_frames=256, **WORD_KW)
        for pos in range(0, X.shape[1], m.strideLen):
            sd.push_decode(X[:, pos:pos + m.strideLen].cpu())
        assert sd._steady
        return done, [sd.transcript(r) for r in range(2)], bits(sd.hypotheses()) + bits(sd.hypotheses(final=True))

    clean = run()
    _poison(monkeypatch)
    dirty = run()
    assert clean[1] == dirty[1]
    for u, (t, raw, fin) in clean[0].items():
        assert t == dirty[0][u][0]
        same(raw + fin, dirty[0][u][1] + dirty[0][u][2], f"utterance {u}")
    same(clean[2], dirty[2])


# ------------------------------------------------------------------------------------------------ capture, guards, no lexicon
def kept_graphs(monkeypatch):
    """From here on every torch.cuda.CUDAGraph keeps its cudaGraph_t after capture (``keep_graph=True``; it is instantiated at the
    first replay), so the graph of a captured push can be read."""
    real = torch.cuda.CUDAGraph
    monkeypatch.setattr(torch.cuda, "CUDAGraph", lambda *a, **k: real(keep_graph=True))


def graph_nodes(g, path):
    """The driver's DOT print of a kept graph (``cuGraphDebugDotPrint``, verbose): its nodes, kernel nodes with their function
    names.  The graph itself says what a replay launches, whatever a profiler in the same process records."""
    rc = ctypes.CDLL("libcuda.so.1").cuGraphDebugDotPrint(ctypes.c_void_p(g.raw_cuda_graph()), str(path).encode(), ctypes.c_uint(1))
    assert rc == 0, f"cuGraphDebugDotPrint returned {rc}"
    with open(path) as f:
        return f.read()


def count_syncs(monkeypatch):
    n = [0]
    for owner, name in ((torch.cuda.Stream, "synchronize"), (torch.cuda.Event, "synchronize"), (torch.cuda, "synchronize")):
        real = getattr(owner, name)

        def counted(*a, _real=real, **k):
            n[0] += 1
            return _real(*a, **k)
        monkeypatch.setattr(owner, name, counted)
    return n


def test_captured_push_reads_words(tmp_path, monkeypatch):
    """The captured push holds the stream kernel, the word advance and the live read-out.  A replayed push_decode makes no
    library call outside the graph and synchronises once, and the transcript after it is current without another
    synchronisation."""
    arch = "comp"
    m = model(arch)
    lex, lm = words_for(arch, tmp_path)
    S, N = m.strideLen, m.neural_dim
    g = torch.Generator().manual_seed(8)
    kept_graphs(monkeypatch)
    ss = nsd.StreamingSessions(m, 2, lexicon=lex, lm=lm, max_frames=256, **WORD_KW)
    sd = nsd.StreamingDecoder(m, 1, torch.zeros(1, dtype=torch.int64, device=DEV), fast=True, use_graph=True, lexicon=lex, lm=lm,
                              max_frames=256, **WORD_KW)
    ss.open(0, 1)
    ss.open(1, 2)
    for _ in range(40):
        ss.push_decode(torch.randn(2, S, N, generator=g).pin_memory(), [True, True])
        sd.push_decode(torch.randn(1, S, N, generator=g).pin_memory())
    assert sd._steady and ss._graph is not None and sd._graph is not None
    monkeypatch.undo()
    for obj, push in ((ss, "stream_push_slots_kernel"), (sd, "stream_push_kernel")):
        dot = graph_nodes(obj._graph, tmp_path / f"{push}.dot")
        assert push in dot and "ctc_word_beam_advance_kernel" in dot and "ctc_word_beam_live_kernel" in dot
    bins2, bins1 = torch.randn(2, S, N, generator=g).pin_memory(), torch.randn(1, S, N, generator=g).pin_memory()
    check = LiveCheck(lex)
    for obj, rows, push in ((ss, (0, 1), lambda: ss.push_decode(bins2, [True, True])), (sd, (0,), lambda: sd.push_decode(bins1))):
        for _ in range(3):
            calls = nsd._lib.launch_count
            syncs = count_syncs(monkeypatch)
            push()
            assert syncs[0] == 1 and nsd._lib.launch_count == calls
            got = [obj.transcript(r) for r in rows]
            assert syncs[0] == 1, "transcript() after push_decode synchronised"
            monkeypatch.undo()
            hyps = [obj.hypotheses(r) for r in rows] if obj is ss else [type(h)(*(t[0] for t in h)) for h in [obj.hypotheses()]]
            for r, t, h in zip(rows, got, hyps):
                check((id(obj), r), t, h)


def test_guards(tmp_path):
    """Misuse raises on the host before anything is launched."""
    arch = "small"
    m = model(arch)
    lex, lm = words_for(arch, tmp_path)
    C = ARCHS[arch]["n_classes"] + 1
    other = Lexicon.from_pronunciations([("A", [1]), ("B", [2, 3])], C + 1, 0, C)
    day = torch.zeros(1, dtype=torch.int64, device=DEV)
    bad = [
        dict(beam_width=W, lexicon=lex, lm=torch.zeros(C, C, device=DEV)),          # a phoneme-bigram tensor with a lexicon
        dict(beam_width=W, lexicon=lex, lm=lm, insertion_bonus=0.5),                  # the phoneme beam's bonus with a lexicon
        dict(beam_width=W, lexicon=other, lm=None),                                   # other class count
        dict(lexicon=lex, lm=lm),                                                     # no beam width
        dict(beam_width=W, lm=lm),                                                    # a word LM without a lexicon
        dict(beam_width=W, word_bonus=1.0),                                           # a word bonus without a lexicon
        dict(beam_width=W, lexicon="not a lexicon"),
        dict(beam_width=4, nbest=5, lexicon=lex),
    ]
    for kw in bad:
        before = nsd.lib().nsd_launch_count()
        with pytest.raises(nsd.NsdError):
            nsd.StreamingDecoder(m, 1, day, **kw)
        with pytest.raises(nsd.NsdError):
            nsd.StreamingSessions(m, 2, **kw)
        assert nsd.lib().nsd_launch_count() == before, kw
    phon = nsd.StreamingDecoder(m, 1, day, beam_width=4)
    ss = nsd.StreamingSessions(m, 2, beam_width=4)
    plain = nsd.StreamingSessions(m, 2)
    before = nsd.lib().nsd_launch_count()
    for fn in (lambda: phon.transcript(), lambda: phon.hypotheses(final=True), lambda: ss.transcript(0), lambda: ss.hypotheses(0, final=True),
               lambda: plain.transcript(0)):
        with pytest.raises(nsd.NsdError):
            fn()
    assert nsd.lib().nsd_launch_count() == before
    bs = WordBeamSearch(2, lex, lm, 4, 16, device=DEV)
    with pytest.raises(nsd.NsdError):
        bs.enqueue_live(torch.zeros(2, 4, dtype=torch.int32, device=DEV))             # no room for a word
    with pytest.raises(nsd.NsdError):
        bs.enqueue_live(torch.zeros(3, 8, dtype=torch.int32, device=DEV))
    with pytest.raises(nsd.NsdError):
        bs.reset_reported(torch.ones(2, dtype=torch.int64, device=DEV))


def test_without_lexicon_unchanged(tmp_path, monkeypatch):
    """Without a lexicon the captured push holds what it held before: the stream kernel, K5b's advance with a phoneme beam,
    no word kernel and no live read-out."""
    arch = "comp"
    m = model(arch)
    S, N = m.strideLen, m.neural_dim
    g = torch.Generator().manual_seed(2)
    kept_graphs(monkeypatch)
    for beam in (None, 8):
        ss = nsd.StreamingSessions(m, 2, beam_width=beam)
        sd = nsd.StreamingDecoder(m, 1, torch.zeros(1, dtype=torch.int64, device=DEV), fast=True, beam_width=beam)
        ss.open(0, 0)
        for _ in range(30):
            ss.push_decode(torch.randn(2, S, N, generator=g).pin_memory(), [True, False])
            sd.push_decode(torch.randn(1, S, N, generator=g).pin_memory())
        assert ss._live is None and sd._live is None and sd._steady and ss._graph is not None and sd._graph is not None
        for obj, push in ((ss, "stream_push_slots_kernel"), (sd, "stream_push_kernel")):
            dot = graph_nodes(obj._graph, tmp_path / f"{push}_{beam}.dot")
            assert push in dot and "word_beam" not in dot
            assert ("ctc_beam_advance_kernel" in dot) == (beam is not None)


def test_live_kernel_against_host(tmp_path):
    """WordBeamSearch.enqueue_live alone, over a batch of random logits advanced frame by frame, with a narrow buffer: the
    committed words arrive in order, none lost, even when more of them than the buffer holds become final at once."""
    arch = "comp"
    lex, lm = words_for(arch, tmp_path)
    C, T, B = lex.num_classes, 120, 4
    rng = np.random.default_rng(0)
    logits = rng.standard_normal((T, B, C)) * 1.5              # random words of the lexicon, spelled with separators, plus noise
    for b in range(B):
        t = 0
        while t < T:
            for c in list(lex.prons[int(rng.integers(len(lex.words)))][0]) + [lex.sep]:
                for _ in range(int(rng.integers(1, 3))):
                    if t < T:
                        logits[t, b, c] += 6.0
                        t += 1
    logits = torch.from_numpy(logits.astype(np.float32)).to(DEV)
    bs = WordBeamSearch(B, lex, lm, W, T, 0.5, 2.0, device=DEV)
    buf = bs.live_buffer(2)
    got, overflowed = [[] for _ in range(B)], False
    for t in range(T):
        bs.advance(logits[t:t + 1], None, True)
        if t % 11 == 10 or t == T - 1:                       # read now and then: more words than the buffer holds commit between reads
            while True:
                bs.enqueue_live(buf)
                rows = nsd.read_live(buf.cpu().numpy())
                for b, (new, _, _) in enumerate(rows):
                    got[b].extend(new)
                if not any(more for _, _, more in rows):
                    break
                overflowed = True
    raw = bs.nbest(W, final=False)
    for b in range(B):
        sc, wl, w = raw.score[b].cpu().numpy(), raw.word_len[b].cpu().tolist(), raw.words[b].cpu().numpy()
        seqs = [tuple(w[k, :wl[k]].tolist()) for k in range(W) if np.isfinite(sc[k])]
        lcp = 0
        while all(len(s) > lcp and s[lcp] == seqs[0][lcp] for s in seqs):
            lcp += 1
        assert got[b] == list(seqs[0][:lcp]), b
    assert overflowed and sum(len(x) for x in got) > 4 * B
