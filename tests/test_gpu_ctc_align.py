"""K5c CTC forced alignment (``nsd_ctc_align``, ``ctc_forced_align``, ``align_batch``) against the float64 oracle
(tests/ctc_align_oracle.py), torchaudio's ``forced_align`` and itself: exact relations between the outputs, bit identity across
input forms, batches and graph replay, guards, and the model paths.

Paths are compared with the oracle only on utterances whose smallest decision margin exceeds 1e-3, so that fp32 rounding cannot
legitimately pick another path.  The ``poisoned`` fixture fills fresh CUDA allocations with NaN / all-ones bits, so output
elements the kernel fails to write show up."""
import numpy as np
import pytest
import torch

from ctc_align_oracle import align_batch as oracle_align, min_frames
from oracle import nsd_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200.ctc import ctc_forced_align, frames_to_bins, log_softmax_tbc

DEV = "cuda"
GAP = 1e-3
# |kernel - oracle| / max(1, |oracle|) of the score (both sum the same fp32 log-probs along the same path, the kernel in fp32),
# ≈3x the worst measured on a B200: 3.9e-7 / 3.0e-7 at T'=118, 7.1e-7 at T'=493, 1.7e-6 at T'=4096
TOL_REL = 5e-6


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


def make_case(seed, T, B, C, Smax, Lmax, blank=0):
    """Peaky blank-heavy logits [T,B,C] f32 (as test_gpu_ctc_beam.make_case), ragged input lengths and padded targets [B,Smax].
    Rows: 0 full length; 1 il = 0, L = 0; 2 il = 1, L = 1; 3 L = 0; 4 il exactly at the feasibility minimum; 5 one frame short of
    it; 6 il = 0 with L > 0; 7 one label repeated, at the minimum; the rest random, about 15 % of them adjacent repeats."""
    rng = np.random.default_rng(seed)
    logits = rng.standard_normal((T, B, C)) * 6.0
    logits[:, :, blank] += 2.0
    labels = np.array([c for c in range(C) if c != blank])
    lens = rng.integers(T // 2, T + 1, B)
    lens[0] = T
    tgt = rng.choice(labels, (B, Smax)).astype(np.int32)
    rep = rng.random((B, Smax)) < 0.15
    for k in range(1, Smax):
        tgt[rep[:, k], k] = tgt[rep[:, k], k - 1]
    tl = np.array([min(Lmax, int(rng.integers(0, lens[b] // 3 + 1))) for b in range(B)])
    if B >= 8:
        lens[1], tl[1] = 0, 0
        lens[2], tl[2] = 1, 1
        tl[3] = 0
        tl[4] = min(Lmax, T // 3)
        lens[4] = min_frames(tgt[4], tl[4])
        tl[5] = min(Lmax, T // 3)
        lens[5] = min_frames(tgt[5], tl[5]) - 1
        lens[6], tl[6] = 0, 2
        tl[7] = min(Lmax, T // 3)
        tgt[7, :] = tgt[7, 0]
        lens[7] = min_frames(tgt[7], tl[7])
    assert (lens <= T).all()
    return logits.astype(np.float32), lens.astype(np.int64), tgt, tl.astype(np.int64)


def to_dev(*xs):
    return [torch.from_numpy(np.ascontiguousarray(x)).to(DEV) for x in xs]


def host(ali):
    return {k: v.cpu().numpy() for k, v in ali._asdict().items()}


def fp32_sum(x):
    """fp32 sum from left to right (the kernel's order)."""
    return np.add.accumulate(np.asarray(x, dtype=np.float32), dtype=np.float32)[-1] if len(x) else np.float32(0)


def check_valid(out, y, tgt, lens, tl, blank=0):
    """Relations that hold on every input, ties included.  y: [T,B,C] f32 log-probs the kernel aligned."""
    T, B, C = y.shape
    Smax = tgt.shape[1]
    for b in range(B):
        il, L = int(min(max(lens[b], 0), T)), int(min(max(tl[b], 0), Smax))
        lab, fl = out["labels"][b], out["frame_logp"][b]
        feasible = il >= min_frames(tgt[b], L) and not (il == 0 and L > 0)
        if not feasible or il == 0:
            assert (lab == -1).all() and (fl == 0).all() and (out["spans"][b] == -1).all() and (out["token_logp"][b] == 0).all(), b
            assert out["score"][b] == (0.0 if feasible else -np.inf), b
            continue
        assert (lab[il:] == -1).all() and (fl[il:] == 0).all()
        lab = lab[:il]
        assert ((lab == blank) | np.isin(lab, tgt[b, :L])).all()
        # frame_logp is y_t[label] bit for bit, the score and every token score its fp32 sum in frame order
        assert np.array_equal(fl[:il].view(np.int32), y[np.arange(il), b, lab].view(np.int32)), b
        assert np.float32(out["score"][b]).view(np.int32) == fp32_sum(fl[:il]).view(np.int32), b
        # the path collapses to the target; the spans are its token runs
        start = [t for t in range(il) if lab[t] != blank and (t == 0 or lab[t - 1] != lab[t])]
        assert [int(lab[t]) for t in start] == tgt[b, :L].tolist(), b
        for k, t0 in enumerate(start):
            t1 = t0
            while t1 + 1 < il and lab[t1 + 1] == lab[t0]:
                t1 += 1
            assert tuple(out["spans"][b, k]) == (t0, t1), (b, k)
            assert np.float32(out["token_logp"][b, k]).view(np.int32) == fp32_sum(fl[t0:t1 + 1]).view(np.int32), (b, k)
        assert (out["spans"][b, L:] == -1).all() and (out["token_logp"][b, L:] == 0).all()


def check_oracle(out, ref, gap=GAP):
    """Score within TOL_REL everywhere; labels, spans and token scores identical where the oracle's margin exceeds ``gap``.
    -> the worst relative score error."""
    fin = np.isfinite(ref["score"])
    assert np.array_equal(np.isfinite(out["score"]), fin)
    err = float((np.abs(out["score"][fin] - ref["score"][fin]) / np.maximum(1.0, np.abs(ref["score"][fin]))).max()) if fin.any() else 0.0
    assert err <= TOL_REL, err
    sure = ref["margin"] > gap
    assert np.array_equal(out["labels"][sure], ref["labels"][sure])
    assert np.array_equal(out["spans"][sure], ref["spans"][sure])
    tok = np.abs(out["token_logp"][sure] - ref["token_logp"][sure]) / np.maximum(1.0, np.abs(ref["token_logp"][sure]))
    assert (tok <= TOL_REL).all()
    return err


# ---------------------------------------------------------------------------------------------------- against the oracle
# (T, B, Smax, Lmax, form, seed): competition shape at two paddings, the long batch padded to 500 with targets up to ~200, and a
# StreamingDecoder-length input with targets up to 500.  Path equality is checked on the utterances whose smallest margin is above
# 1e-3: all of them at B <= 64, and at least 98 % of them (asserted) in the long batch.
PARITY = [
    (118, 64, 60, 60, "logits", 0),
    (118, 64, 500, 60, "lp_btc", 0),
    (493, 256, 500, 200, "logits_btc", 0),
    (4096, 4, 500, 500, "lp", 0),
]


@pytest.mark.parametrize("T,B,Smax,Lmax,form,seed", PARITY)
def test_matches_oracle(T, B, Smax, Lmax, form, seed, poisoned, record_property):
    C = 41
    logits, lens, tgt, tl = make_case(seed, T, B, C, Smax, Lmax)
    lg = torch.from_numpy(logits).to(DEV)
    y = log_softmax_tbc(lg.permute(1, 0, 2).contiguous()).contiguous()       # the log-probs the kernel aligns, [T,B,C]
    src = lg if form.startswith("logits") else y
    if form.endswith("btc"):
        src = src.permute(1, 0, 2).contiguous().permute(1, 0, 2)             # a [B,T,C] buffer seen as [T,B,C]
    tgt_d, lens_d, tl_d = to_dev(tgt, lens, tl)
    out = host(ctc_forced_align(src, tgt_d, lens_d, tl_d, is_logits=form.startswith("logits")))
    y_h = y.cpu().numpy()
    ref = oracle_align(y_h.astype(np.float64), tgt, lens, tl)
    fin = np.isfinite(ref["score"])
    sure = ref["margin"][fin] > GAP
    assert sure.all() if B <= 64 else sure.mean() >= 0.98, ref["margin"][fin].min()
    assert (~fin).sum() == (2 if B >= 8 else 0)                                # rows 5 and 6
    err = check_oracle(out, ref)
    record_property("score_err", err)
    print(f"T={T} B={B} Smax={Smax}: worst |score - oracle| / max(1, |oracle|) = {err:.3e}")
    check_valid(out, y_h, tgt, lens, tl)


@pytest.mark.parametrize("seed", range(4))
def test_ties_are_valid(seed, poisoned):
    """Coarse log-probs (multiples of 0.25) make exact ties between paths: whatever the kernel picks must still be a valid path
    whose outputs follow from it exactly, and its score must be the maximum."""
    T, B, C = 60, 16, 6
    logits, lens, tgt, tl = make_case(100 + seed, T, B, C, 20, 20)
    lp = np.round(np.asarray(O.log_softmax(logits.astype(np.float64)), dtype=np.float32) * 4) / 4
    lp = lp.astype(np.float32)
    tgt_d, lens_d, tl_d = to_dev(tgt, lens, tl)
    out = host(ctc_forced_align(torch.from_numpy(lp).to(DEV), tgt_d, lens_d, tl_d))
    check_valid(out, lp, tgt, lens, tl)
    ref = oracle_align(lp.astype(np.float64), tgt, lens, tl)
    fin = np.isfinite(ref["score"])
    assert np.array_equal(out["score"][fin], ref["score"][fin].astype(np.float32))   # quarter steps: every sum is exact
    assert (ref["margin"][fin] == 0).any()                                          # the case does contain ties


def test_against_torchaudio():
    F = pytest.importorskip("torchaudio.functional")
    T, B, C = 118, 64, 41
    logits, lens, tgt, tl = make_case(0, T, B, C, 60, 60)
    lg = torch.from_numpy(logits).to(DEV)
    tgt_d, lens_d, tl_d = to_dev(tgt, lens, tl)
    out = host(ctc_forced_align(lg, tgt_d, lens_d, tl_d, is_logits=True))
    y = log_softmax_tbc(lg.permute(1, 0, 2).contiguous()).contiguous().cpu()
    ref = oracle_align(y.numpy().astype(np.float64), tgt, lens, tl)
    n = 0
    for b in range(B):
        il, L = int(lens[b]), int(tl[b])
        if L == 0 or not np.isfinite(ref["score"][b]):
            continue
        lab, sc = F.forced_align(y[:il, b][None].contiguous(), torch.from_numpy(tgt[b:b + 1, :L]).int(), torch.tensor([il]), torch.tensor([L]), blank=0)
        assert abs(sc.double().sum().item() - out["score"][b]) <= TOL_REL * max(1.0, abs(out["score"][b])), b
        if ref["margin"][b] > GAP:
            assert lab[0].numpy().tolist() == out["labels"][b, :il].tolist(), b
            n += 1
    assert n >= 40


# ---------------------------------------------------------------------------------------------------- bit identity
def _same(a, b):
    for k in a:
        assert np.array_equal(a[k].view(np.int32) if a[k].dtype == np.float32 else a[k],
                              b[k].view(np.int32) if b[k].dtype == np.float32 else b[k]), k


def test_logits_equal_log_softmaxed(poisoned):
    logits, lens, tgt, tl = make_case(3, 118, 64, 41, 60, 60)
    lg = torch.from_numpy(logits).to(DEV)
    args = to_dev(tgt, lens, tl)
    a = host(ctc_forced_align(lg, *args, is_logits=True))
    b = host(ctc_forced_align(log_softmax_tbc(lg.permute(1, 0, 2)), *args))
    _same(a, b)


def test_permuted_view_equals_contiguous(poisoned):
    logits, lens, tgt, tl = make_case(4, 118, 64, 41, 60, 60)
    btc = torch.from_numpy(np.ascontiguousarray(logits.transpose(1, 0, 2))).to(DEV)
    args = to_dev(tgt, lens, tl)
    for is_logits in (True, False):
        v = btc.permute(1, 0, 2)
        _same(host(ctc_forced_align(v, *args, is_logits=is_logits)), host(ctc_forced_align(v.contiguous(), *args, is_logits=is_logits)))


def test_alone_equals_in_batch(poisoned):
    logits, lens, tgt, tl = make_case(5, 118, 64, 41, 60, 60)
    lg = torch.from_numpy(logits).to(DEV)
    tgt_d, lens_d, tl_d = to_dev(tgt, lens, tl)
    full = host(ctc_forced_align(lg, tgt_d, lens_d, tl_d, is_logits=True))
    for b in (0, 2, 4, 7, 9, 63):
        one = host(ctc_forced_align(lg[:, b:b + 1], tgt_d[b:b + 1], lens_d[b:b + 1], tl_d[b:b + 1], is_logits=True))
        _same(one, {k: v[b:b + 1] for k, v in full.items()})


def test_graph_replay_equals_eager():
    T, B, C = 118, 64, 41
    first = make_case(6, T, B, C, 60, 60)
    second = make_case(7, T, B, C, 60, 60)
    static = [torch.from_numpy(first[0]).to(DEV)] + to_dev(first[2], first[1], first[3])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ctc_forced_align(*static, is_logits=True, check=False)                # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ctc_forced_align(*static, is_logits=True, check=False)
    new = [torch.from_numpy(second[0]).to(DEV)] + to_dev(second[2], second[1], second[3])
    for dst, src in zip(static, new):
        dst.copy_(src)
    g.replay()
    torch.cuda.synchronize()
    _same(host(out), host(ctc_forced_align(*new, is_logits=True)))


# ---------------------------------------------------------------------------------------------------- guards
@pytest.mark.parametrize("bad", [0, 41, 77, -3])
def test_bad_target_sets_flag(bad, poisoned):
    T, B, C = 118, 16, 41
    logits, lens, tgt, tl = make_case(8, T, B, C, 30, 30)
    tl[9] = max(tl[9], 3)
    good = host(ctc_forced_align(torch.from_numpy(logits).to(DEV), *to_dev(tgt, lens, tl), is_logits=True))
    tgt[9, 1] = bad
    tgt[10, tl[10]:] = bad                                                   # padding past the target length is never read
    args = [torch.from_numpy(logits).to(DEV)] + to_dev(tgt, lens, tl)
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(*args, is_logits=True)
    out = host(ctc_forced_align(*args, is_logits=True, check=False))
    others = np.arange(B) != 9
    _same({k: v[others] for k, v in out.items()}, {k: v[others] for k, v in good.items()})
    assert out["score"][9] == -np.inf and (out["labels"][9] == -1).all() and (out["spans"][9] == -1).all()
    assert (out["frame_logp"][9] == 0).all() and (out["token_logp"][9] == 0).all()


def test_bounds():
    act = torch.zeros(4, 2, 41, device=DEV)
    tgt = torch.ones(2, 3, dtype=torch.int32, device=DEV)
    lens = torch.full((2,), 4, device=DEV)
    tl = torch.full((2,), 2, device=DEV)
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(act.cpu(), tgt.cpu(), lens.cpu(), tl.cpu())
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(act[0], tgt, lens, tl)
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(act, tgt[0], lens, tl)
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(act, tgt[:1], lens, tl)
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(torch.zeros(4, 2, 129, device=DEV), tgt, lens, tl)
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(act, tgt, lens, tl, blank=41)
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(torch.zeros(8193, 1, 5, device=DEV), tgt[:1], lens[:1], tl[:1])
    with pytest.raises(nsd.NsdError):
        ctc_forced_align(act, torch.ones(2, 1025, dtype=torch.int32, device=DEV), lens, tl)


def test_empty_target_width(poisoned):
    act = torch.randn(10, 3, 5, device=DEV).log_softmax(-1)
    out = host(ctc_forced_align(act, torch.zeros(3, 0, dtype=torch.int32, device=DEV), torch.tensor([10, 0, 4], device=DEV),
                                torch.zeros(3, dtype=torch.int32, device=DEV)))
    assert out["spans"].shape == (3, 0, 2) and out["token_logp"].shape == (3, 0)
    assert (out["labels"][0] == 0).all() and (out["labels"][2, :4] == 0).all() and (out["labels"][2, 4:] == -1).all()
    assert out["score"][1] == 0.0 and (out["labels"][1] == -1).all()


# ---------------------------------------------------------------------------------------------------- dispatch
def test_dispatch_reaches():
    """The host has one kernel form; the smallest call launches it by name."""
    act = torch.zeros(1, 1, 2, device=DEV)
    one = torch.ones(1, dtype=torch.int32, device=DEV)
    names = kernels_launched(lambda: ctc_forced_align(act, torch.ones(1, 1, dtype=torch.int32, device=DEV), one, one, check=False))
    assert "ctc_align_kernel" in names


# ---------------------------------------------------------------------------------------------------- models
def test_align_batch_gru(poisoned):
    from neural_speech_decoder_b200.synthetic import fill_trained_like_, make_batch
    kw = dict(neural_dim=32, n_classes=10, hidden_dim=64, layer_dim=2, nDays=4, dropout=0.0, strideLen=4, kernelLen=16,
              gaussianSmoothWidth=2.0, bidirectional=True)
    torch.manual_seed(0)
    m = nsd.GRUDecoder(device="cuda", **kw)
    fill_trained_like_(m, seed=3)
    m = m.to(DEV).eval()
    X, y, X_len, y_len, day = make_batch(8, 200, n_feat=32, n_days=4, n_classes=10, seed=5, ragged=True, min_tgt=2, max_tgt=12,
                                         kernel_len=16, stride_len=4)
    X, y, X_len, y_len, day = [t.to(DEV) for t in (X, y, X_len, y_len, day)]
    ali, bins = nsd.align_batch(m, X, y, X_len, y_len, day)
    with torch.no_grad():
        lp = log_softmax_tbc(m.forward(X, day))
    lens = nsd.out_lens(X_len, 16, 4)
    _same(host(ali), host(ctc_forced_align(lp, y, lens, y_len)))
    out, sp, bn = host(ali), ali.spans.cpu().numpy(), bins.cpu().numpy()
    check_valid(out, lp.contiguous().cpu().numpy(), y.cpu().numpy(), lens.cpu().numpy(), y_len.cpu().numpy())
    assert np.isfinite(out["score"]).all()
    has = sp[..., 0] >= 0
    assert np.array_equal(has, np.arange(sp.shape[1])[None, :] < y_len.cpu().numpy()[:, None])
    assert np.array_equal(bn[..., 0][has], sp[..., 0][has] * 4) and np.array_equal(bn[..., 1][has], sp[..., 1][has] * 4 + 16)
    assert (bn[~has] == -1).all()
    # the last frame's window ends inside the utterance: (out_len - 1) * S + K <= X_len
    assert (bn[..., 1].max(axis=1) <= X_len.cpu().numpy()).all()
    last = (lens.cpu().numpy() - 1) * 4 + 16
    assert (last <= X_len.cpu().numpy()).all()
    assert torch.equal(frames_to_bins(torch.tensor([[[0, 0], [3, 5], [-1, -1]]]), 32, 4),
                       torch.tensor([[[0, 32], [12, 52], [-1, -1]]]))


def test_conformer_log_probs():
    kw = dict(n_channels=32, n_classes=11, n_days=3, frontend_dim=64, latent_dim=64, autoencoder_hidden_dim=32, transformer_layers=2,
              transformer_heads=4, transformer_ff_dim=128, transformer_dropout=0.0, temporal_kernel=16, temporal_stride=4,
              gaussian_smooth_width=2.0, conformer_conv_kernel=7, use_spec_augment=False, drop_path_prob=0.0)
    g = torch.Generator().manual_seed(9)
    B, T = 4, 120
    X = torch.randn(B, T, 32, generator=g)
    day = torch.randint(0, 3, (B,), generator=g)
    X_len = torch.tensor([120, 84, 100, 64], dtype=torch.int32)
    y_len = torch.tensor([5, 3, 4, 6], dtype=torch.int32)
    y = torch.zeros(B, 6, dtype=torch.int32)
    for b in range(B):
        y[b, :y_len[b]] = torch.randint(1, 11, (int(y_len[b]),), generator=g).to(torch.int32)
    torch.manual_seed(0)
    m = nsd.NeuralTransformerCTCModel(device="cuda", **kw).to(DEV).eval()
    with torch.no_grad():
        lp, olen, _ = m(X.to(DEV), day.to(DEV), X_len.to(DEV))
    ali = ctc_forced_align(lp, y.to(DEV), olen, y_len.to(DEV))
    out = host(ali)
    check_valid(out, lp.contiguous().cpu().numpy(), y.numpy(), olen.cpu().numpy(), y_len.numpy())
    assert np.isfinite(out["score"]).all()
