"""StreamingSessions: independent per-slot streaming sessions on the single-launch push (nsd_stream_push_slots).

A seeded schedule opens, pushes, pauses and finishes utterances of random lengths in random slots; each utterance's logits
must be the bits of the same utterance streamed alone through ``StreamingSessions(model, 1)``, and close to the offline
forward and to the reference operators with carried state.  Idle slots keep every byte, a fresh or reused slot reads nothing
it did not write, the per-session beam equals the one-shot beam search, and misuse raises on the host before any launch."""
import random

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200.synthetic import fill_trained_like_

DEV = "cuda"
COMP = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, strideLen=4, kernelLen=32, gaussianSmoothWidth=2.0)
SMALL = dict(neural_dim=64, n_classes=20, hidden_dim=512, layer_dim=2, nDays=3, strideLen=3, kernelLen=24, gaussianSmoothWidth=1.5)
ARCHS = {"comp": COMP, "small": SMALL}
N_UTT = 22


def build(**kw):
    nsd.set_default_precision("bf16")
    try:
        torch.manual_seed(0)
        m = nsd.GRUDecoder(device=DEV, **kw)
    finally:
        nsd.set_default_precision("fp32")
    fill_trained_like_(m, seed=5)
    return m.to(DEV).eval()


def make_utterances(kw, n, seed):
    """n utterances: (bins f32 [T, N] on the CPU, day); lengths from K to ~600 bins, many not a multiple of S."""
    g = torch.Generator().manual_seed(seed)
    K = kw["kernelLen"]
    lens = [K, K + 1, K + kw["strideLen"] + 2, 600, 597] + [int(v) for v in torch.randint(K, 601, (n - 5,), generator=g)]
    return [(torch.randn(T, kw["neural_dim"], generator=g), int(torch.randint(0, kw["nDays"], (1,), generator=g))) for T in lens]


def stream_alone(m, X, day):
    """The utterance streamed alone through one slot with no gaps -> logits [T', C]."""
    ss = nsd.StreamingSessions(m, 1)
    S = m.strideLen
    ss.open(0, day)
    outs, pos = [], 0
    while X.shape[0] - pos >= S:
        lg, em = ss.push(X[pos:pos + S].unsqueeze(0).to(DEV), [True])
        pos += S
        if bool(em[0]):
            outs.append(lg[0:1])
    outs.append(ss.finish(0, X[pos:].to(DEV)))
    return torch.cat(outs)


_REF = {}


def reference(arch):
    """(model, utterances, logits of each utterance streamed alone), once per architecture."""
    if arch not in _REF:
        kw = ARCHS[arch]
        m = build(**kw)
        utts = make_utterances(kw, N_UTT, seed=2024 if arch == "comp" else 7)
        _REF[arch] = (m, utts, [stream_alone(m, X, d) for X, d in utts])
    return _REF[arch]


def run_schedule(ss, m, utts, seed, decode_share=0.0, on_finish=None):
    """Feed ``utts`` through the slots of ``ss`` on a seeded random schedule: staggered starts, open-but-inactive gaps, slot
    reuse, random tail lengths; a share of the pushes goes through push_decode.  Returns per utterance the list of its
    frames in order: logits [k, C] (push, finish) or a greedy id (push_decode).  ``on_finish(u, slot)`` runs after each
    finish."""
    rng = random.Random(seed)
    S, N, B = m.strideLen, m.neural_dim, ss.slots
    queue = list(range(len(utts)))
    slot_utt, slot_pos, slot_tail = [None] * B, [0] * B, [0] * B
    got = {u: [] for u in queue}
    while queue or any(u is not None for u in slot_utt):
        for s in range(B):                                      # free slots take the next utterance, not always at once
            if slot_utt[s] is None and queue and rng.random() < 0.6:
                u = queue.pop(0)
                slot_utt[s], slot_pos[s] = u, 0
                T = utts[u][0].shape[0]
                slot_tail[s] = min(T, rng.choice([0, 1, 2, S, S + 1, 3 * S + 2, 9]))   # bins left for finish()
                ss.open(s, utts[u][1])
        bins = torch.zeros(B, S, N)
        active = [False] * B
        for s in range(B):
            u = slot_utt[s]
            if u is None:
                continue
            X = utts[u][0]
            if X.shape[0] - slot_pos[s] - slot_tail[s] < S:    # only the tail is left: end the session
                got[u].append(ss.finish(s, X[slot_pos[s]:].to(DEV)).cpu())
                slot_utt[s] = None
                if on_finish is not None:
                    on_finish(u, s)
                continue
            if rng.random() < 0.8:                              # otherwise an open-but-inactive gap
                bins[s] = X[slot_pos[s]:slot_pos[s] + S]
                active[s] = True
        if not any(active):
            continue
        if rng.random() < decode_share:
            ids = ss.push_decode(bins.pin_memory(), active).clone()
            for s in range(B):
                if not active[s]:
                    assert int(ids[s]) == -1
                elif int(ids[s]) >= 0:
                    got[slot_utt[s]].append(int(ids[s]))
        else:
            lg, em = ss.push(bins.to(DEV), torch.tensor(active))
            lg, em = lg.cpu(), em.cpu()
            for s in range(B):
                assert active[s] or not bool(em[s])
                if bool(em[s]):
                    got[slot_utt[s]].append(lg[s:s + 1])
        for s in range(B):
            slot_pos[s] += S if active[s] else 0
    return got


def check_against(got, ref):
    """Each utterance's frames equal the alone run bit for bit (logits) or its argmax (push_decode ids)."""
    for u, parts in got.items():
        f = 0
        for p in parts:
            if isinstance(p, int):
                assert p == int(ref[u][f].argmax()), f"utterance {u}: push_decode id of frame {f}"
                f += 1
                continue
            assert torch.equal(p, ref[u][f:f + p.shape[0]].cpu()), f"utterance {u}: frames {f}..{f + p.shape[0] - 1} differ"
            f += p.shape[0]
        assert f == ref[u].shape[0], f"utterance {u}: {f} frames, alone {ref[u].shape[0]}"


@pytest.mark.parametrize("arch,slots,use_graph", [
    ("comp", 8, True), ("comp", 8, False), ("comp", 6, True), ("comp", 3, True), ("comp", 2, False), ("comp", 1, True),
    ("small", 5, True), ("small", 4, False), ("small", 2, True),
])
def test_schedule_invariance(arch, slots, use_graph):
    """Every utterance of a random schedule gives the bits of the same utterance streamed alone; push_decode ids == argmax."""
    m, utts, ref = reference(arch)
    ss = nsd.StreamingSessions(m, slots, use_graph=use_graph)
    got = run_schedule(ss, m, utts, seed=slots * 10 + int(use_graph), decode_share=0.3)
    if use_graph:
        assert ss._graph is not None, getattr(ss, "_graph_error", "no graph captured")
    check_against(got, ref)
    assert sum(isinstance(p, int) for parts in got.values() for p in parts) > 50


def port_streaming_oracle(port, X, day, frames_per_call):
    """The reference-operator oracle of tests/test_gpu_streaming.py: front end of the whole utterance, nn.GRU fed
    ``frames_per_call`` frames at a time with h_n carried into the next call, output layer -> logits [B, T', C]."""
    import torch.nn.functional as F
    with torch.no_grad():
        x = X.permute(0, 2, 1)
        x = F.conv1d(x, port.smooth_w, groups=port.neural_dim, padding="same").permute(0, 2, 1)
        w = torch.index_select(port.dayWeights, 0, day)
        x = F.softsign(torch.einsum("btd,bdk->btk", x, w) + torch.index_select(port.dayBias, 0, day))
        x = F.unfold(x.permute(0, 2, 1).unsqueeze(3), (port.kernelLen, 1), stride=port.strideLen).permute(0, 2, 1)
        h = torch.zeros(port.layer_dim, x.size(0), port.hidden_dim, dtype=x.dtype)
        outs = []
        for j in range(0, x.size(1), frames_per_call):
            hid, h = port.gru(x[:, j:j + frames_per_call], h)
            outs.append(port.fc(hid))
        return torch.cat(outs, dim=1)


@pytest.mark.parametrize("arch", ["comp", "small"])
def test_accuracy(arch):
    """Each session against the offline forward of the utterance alone (same bf16 arithmetic, other fp32 summation order)
    and against the reference operators with carried state in fp64: the bounds of the fast-form test of StreamingDecoder."""
    from oracle import torch_port as P
    m, utts, ref = reference(arch)
    kw = ARCHS[arch]
    port = P.PortGRUDecoder(bidirectional=False, dropout=0.0, **kw)
    port.load_reference_state({k: v.detach().cpu() for k, v in m.state_dict().items()})
    port = port.double().eval()
    e_off = e_ref = 0.0
    agree = []
    for (X, day), got in zip(utts, ref):
        got = got.cpu().numpy().astype(np.float64)
        with torch.no_grad():
            off = m.forward(X.unsqueeze(0).to(DEV), torch.tensor([day], device=DEV))[0].cpu().numpy().astype(np.float64)
        orc = port_streaming_oracle(port, X.unsqueeze(0).double(), torch.tensor([day]), frames_per_call=1 << 30)[0].numpy()
        assert got.shape == off.shape == orc.shape
        e_off, e_u = max(e_off, np.abs(got - off).max()), np.abs(got - orc).max()
        e_ref = max(e_ref, e_u)
        agree.append(got.argmax(-1) == orc.argmax(-1))
        top2 = np.sort(orc, axis=-1)[..., -2:]
        flips = got.argmax(-1) != orc.argmax(-1)
        assert not (flips & ((top2[..., 1] - top2[..., 0]) > 2 * e_u)).any()
    agree = np.concatenate(agree).mean()
    print(f"sessions {arch}: vs offline forward {e_off:.3e}, vs reference operators {e_ref:.3e}, argmax agreement {agree:.4f}")
    assert e_off < 0.06 and e_ref < 0.12 and agree >= 0.95


def slot_state(ss, s):
    """The bytes of every per-slot state tensor of slot s (bytes, so that never-written NaN patterns compare too)."""
    st = [ss._rawring[s], ss._x0buf[:, s], ss._h[:, s], ss._hbf[:, s], ss._n_bins[s], ss._last[s], ss._day[s]]
    if ss._beam is not None:
        per = ss._beam.state_bytes // ss.slots
        st.append(ss._beam.state[s * per:(s + 1) * per])
    return [t.reshape(-1).clone().view(torch.uint8) for t in st]


def test_idle_slots_untouched():
    """Pushes with a slot inactive, and open / finish of other slots, leave every byte of that slot's state (ring, patch
    rows, h, h_bf16, counter, last frame, day, beam) as it was -- mid-utterance and after its finish."""
    m, utts, _ = reference("comp")
    S = m.strideLen
    ss = nsd.StreamingSessions(m, 4, beam_width=8, nbest=2)
    X0, X1, X2 = utts[3][0], utts[4][0], utts[3][0].flip(0)          # 600 and 597 bins
    ss.open(0, 1)
    ss.open(1, 2)
    ss.open(3, 3)
    for i in range(15):                                       # slot 0 mid-utterance (past its warm-up), slot 3 before its first frame
        b = torch.zeros(4, S, m.neural_dim)
        b[0], b[1] = X0[i * S:(i + 1) * S], X1[i * S:(i + 1) * S]
        b[3] = X2[i * S:(i + 1) * S]
        ss.push(b.to(DEV), [True, True, False, i < 3])
    ss.finish(1, X1[15 * S:15 * S + 5].to(DEV))              # slot 1 closed: its state must stay readable and unchanged too
    snaps = {s: slot_state(ss, s) for s in (0, 1, 3)}
    for i in range(14):                                       # slot 2: an utterance of 10 pushes + 7 tail bins, then a new one
        b = torch.randn(4, S, m.neural_dim)
        if i == 0:
            ss.open(2, 0)
        if i == 10:
            ss.finish(2, torch.randn(7, m.neural_dim, device=DEV))
            ss.open(2, 4)
        ss.push(b.to(DEV), [False, False, True, False])
    torch.cuda.synchronize()
    for s, snap in snaps.items():
        for i, (a, b) in enumerate(zip(snap, slot_state(ss, s))):
            assert torch.equal(a, b), f"slot {s}, state tensor {i}"


@pytest.fixture
def poisoned(monkeypatch):
    """torch.empty / torch.empty_like return CUDA tensors filled with NaN (floating) or all-ones bits (integer), as in
    tests/test_gpu_dispatch_variants.py."""
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


def test_fresh_state_fully_written(poisoned):
    """Every buffer of a new StreamingSessions starts as NaN / all-ones: a newly opened slot and a slot reopened after an
    earlier utterance give the bits of the schedule test."""
    m, utts, ref = reference("comp")
    sub = [0, 4, 7, 2, 9]
    ss = nsd.StreamingSessions(m, 3)
    got = run_schedule(ss, m, [utts[u] for u in sub], seed=99, decode_share=0.3)
    check_against(got, [ref[u] for u in sub])


def test_beam_per_session():
    """With beam_width=16, nbest=4 and a bigram prior, each session's N-best is bit-identical to the one-shot beam search
    over that utterance's logits."""
    m, utts, ref = reference("comp")
    C = m.fc_decoder_out.weight.shape[0]
    g = torch.Generator().manual_seed(3)
    lm = torch.log_softmax(torch.randn(C, C, generator=g), dim=-1).to(DEV)
    ss = nsd.StreamingSessions(m, 4, beam_width=16, nbest=4, lm=lm, lm_weight=0.6, insertion_bonus=0.3)
    sub = list(range(8))
    nbest = {}

    def read(u, slot):                                        # the session's N-best, read right after its finish
        nbest[u] = [t.clone() for t in ss.hypotheses(slot)]

    got = run_schedule(ss, m, [utts[u] for u in sub], seed=5, decode_share=0.3, on_finish=read)
    check_against(got, [ref[u] for u in sub])
    assert sorted(nbest) == list(range(len(sub)))
    for u, (hyps, hyp_len, score, acoustic) in nbest.items():
        lg = ref[sub[u]]
        T = lg.shape[0]
        want = nsd.ctc_beam_search(lg.unsqueeze(1), None, 16, 4, 0, lm, 0.6, 0.3, is_logits=True)
        assert torch.equal(hyp_len, want[1][0]) and torch.equal(score, want[2][0]) and torch.equal(acoustic, want[3][0]), f"utterance {u}"
        assert torch.equal(hyps[:, :T], want[0][0]) and bool((hyps[:, T:] == -1).all()), f"utterance {u}"


def test_errors():
    """Misuse raises on the host before any launch; unsupported models and slot counts are refused."""
    kw = dict(SMALL)
    m = build(**kw)
    S, N, K = kw["strideLen"], kw["neural_dim"], kw["kernelLen"]
    ss = nsd.StreamingSessions(m, 2, max_frames=3)
    ok = torch.zeros(2, S, N, device=DEV)
    with pytest.raises(nsd.NsdError):                          # closed slot
        ss.push(ok, [True, False])
    ss.open(0, 1)
    with pytest.raises(nsd.NsdError):                          # the other slot is still closed
        ss.push(ok, [True, True])
    with pytest.raises(nsd.NsdError):
        ss.push(torch.zeros(2, S + 1, N, device=DEV), [True, False])
    with pytest.raises(nsd.NsdError):
        ss.push(torch.zeros(3, S, N, device=DEV), [True, False, False])
    with pytest.raises(nsd.NsdError):
        ss.push(ok, [True, False, False])
    with pytest.raises(nsd.NsdError):
        ss.push(ok, torch.ones(2, 1))
    with pytest.raises(nsd.NsdError):
        ss.push_decode(torch.zeros(2, S, N).pin_memory(), [False, True])
    with pytest.raises(nsd.NsdError):
        ss.finish(1, torch.zeros(4, N, device=DEV))
    with pytest.raises(nsd.NsdError):
        ss.finish(0, torch.zeros(4, N + 1, device=DEV))
    with pytest.raises(nsd.NsdError):
        ss.open(2, 0)
    with pytest.raises(nsd.NsdError):
        ss.hypotheses(0)
    # max_frames: the fourth frame of a session is refused by push() and by finish(), and nothing moves
    emitted = 0
    while emitted < 3:
        _, em = ss.push(torch.randn(2, S, N, device=DEV), [True, False])
        emitted += int(em[0])
    n_before = ss._n_bins.clone()
    with pytest.raises(nsd.NsdError):
        ss.push(torch.randn(2, S, N, device=DEV), [True, False])
    with pytest.raises(nsd.NsdError):
        ss.finish(0, torch.zeros(0, N, device=DEV))
    assert torch.equal(ss._n_bins, n_before)
    # an utterance shorter than kernelLen raises as the reference does (nn.Unfold), and closes the slot
    ss.open(1, 0)
    with pytest.raises(RuntimeError):
        ss.finish(1, torch.zeros(K - 1, N, device=DEV))
    with pytest.raises(nsd.NsdError):
        ss.push(ok, [False, True])
    # a day out of range sets the model's error flag, as the offline front end does
    m._err_flag.zero_()
    ss.open(1, kw["nDays"])
    ss.push(ok, [False, True])
    torch.cuda.synchronize()
    assert int(m._err_flag.item()) == 1
    m._err_flag.zero_()
    # unsupported models and sizes
    with pytest.raises(nsd.NsdError):
        nsd.StreamingSessions(m, 9)
    with pytest.raises(nsd.NsdError):
        nsd.StreamingSessions(m, 0)
    with pytest.raises(nsd.NsdError):
        nsd.StreamingSessions(build(bidirectional=True, **kw), 2)
    with pytest.raises(nsd.NsdError):
        nsd.StreamingSessions(build(**dict(kw, hidden_dim=256)), 2)
    torch.manual_seed(0)
    fp32 = nsd.GRUDecoder(device=DEV, **kw).eval()
    with pytest.raises(nsd.NsdError):
        nsd.StreamingSessions(fp32, 2)
