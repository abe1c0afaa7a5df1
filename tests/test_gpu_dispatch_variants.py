"""Every kernel instance the host dispatch can select, against a plain high-precision reference.

The C-ABI entry points pick a kernel instance from the shape of each call: the fast K1 forward per kernelLen, the K3
recurrence per chain count, the streaming push per batch form.  ``test_dispatch_reaches`` pins that shape -> instance
mapping (by kernel name, under torch.profiler), so the sweeps below keep covering what they claim to.

Outputs and workspaces are allocated with ``torch.empty`` by the ops layer; in training they hold whatever the caching
allocator last had there.  The ``poisoned`` fixture fills every fresh CUDA allocation with NaN (floating types) or 0xFF bytes
(integer types), so a kernel that reads a row it never wrote shows up as a non-finite result."""
import numpy as np
import pytest
import torch

from oracle import nsd_oracle as O
from test_gpu_streaming import build as build_streaming_model, port_streaming_oracle

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from neural_speech_decoder_b200 import ops
    import neural_speech_decoder_b200 as nsd

DEV = "cuda"
COMP = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, strideLen=4, kernelLen=32, gaussianSmoothWidth=2.0)


@pytest.fixture
def poisoned(monkeypatch):
    """torch.empty / torch.empty_like return CUDA tensors filled with NaN (floating) or all-ones bits (integer); host and
    pinned tensors are left alone."""
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


def _reach_frontend(K, S, ntaps=20, bwd=False):
    x, day, W, bias = frontend_inputs(1, K + S, 0)
    taps = O.gaussian_taps(2.0) if ntaps == 20 else np.concatenate([[0.0], O.gaussian_taps(2.0)]).astype(np.float32)
    if not bwd:
        return lambda: fast_frontend(x, day, W, bias, K, S, taps=taps)
    _, ys, z = fast_frontend(x, day, W, bias, K, S)
    dp = torch.randn(O.n_frames(K + S, K, S), N1 * K, device=DEV).to(torch.bfloat16)
    return lambda: ops.frontend_bwd(dp, ys, z, day, ND1, K, S)


def _reach_gru(B, bwd):
    H, Tp = 128, 2
    gi = torch.randn(Tp * B, 3 * H, device=DEV)
    w = (torch.randn(3 * H, H, device=DEV) / H ** 0.5).to(torch.bfloat16)
    b = torch.zeros(3 * H, device=DEV)
    if not bwd:
        return lambda: ops.gru_fwd_bf16(gi, w, b, Tp, B, H, 1, False, False)
    hseq, _, sv = ops.gru_fwd_bf16(gi, w, b, Tp, B, H, 1, False, True)
    dh = torch.randn(Tp * B, H, device=DEV)
    return lambda: ops.gru_bwd_bf16(dh, hseq, sv, w.T.contiguous(), Tp, B, H, 1, False)


def _reach_stream(B):
    m = build_streaming_model(**SMALL_C)
    sd = nsd.StreamingDecoder(m, B, torch.zeros(B, dtype=torch.int64, device=DEV), use_graph=False)
    assert sd.fast
    X = torch.randn(B, 64, SMALL_C["neural_dim"], device=DEV)
    for pos in range(0, 56, 8):
        sd.push(X[:, pos:pos + 8])
    assert sd._steady
    return lambda: sd.push(X[:, 56:64])


def _reach_ctc():
    logits, y, il, yl = (torch.from_numpy(a).to(DEV) for a in _ctc_inputs())
    return lambda: nsd.ctc_loss_from_logits(logits, y, il, yl)


def _ctc_inputs():
    rng = np.random.default_rng(0)
    y = np.zeros((2, 420), np.int32)                          # max_tgt 420: the kernel needs more than 48 KB of shared memory
    y[:, :3] = [[1, 2, 3], [4, 5, 6]]
    return rng.standard_normal((2, 12, 41)).astype(np.float32), y, np.full(2, 12, np.int32), np.full(2, 3, np.int32)


REACH = {
    **{f"frontend_fwd_fast_kernel<{K // 8}>": (lambda K=K: _reach_frontend(K, 4)) for K in (8, 16, 32, 64)},
    "frontend_fwd_kernel<__nv_bfloat16,2,16>": lambda: _reach_frontend(32, 4, ntaps=21),
    "frontend_bwd_tc_kernel<2>": lambda: _reach_frontend(16, 8, bwd=True),
    "frontend_bwd_tc2_kernel": lambda: _reach_frontend(32, 4, bwd=True),
    "rts::gru_fwd_ts_kernel<2>": lambda: _reach_gru(1, False),
    "rts::gru_fwd_ts_kernel<4>": lambda: _reach_gru(65, False),
    "rts::gru_bwd_ts_kernel<2>": lambda: _reach_gru(1, True),
    "rts::gru_bwd_ts_kernel<4>": lambda: _reach_gru(65, True),
    **{f"stream_push_kernel<{bm}>": (lambda B=B: _reach_stream(B)) for B, bm in ((1, 1), (2, 2), (3, 4), (5, 8))},
    "ctc_kernel": _reach_ctc,
}


@pytest.mark.parametrize("kernel", list(REACH))
def test_dispatch_reaches(kernel):
    """The smallest call of each dispatch form launches the kernel instance the sweeps below rely on."""
    run = REACH[kernel]()
    names = kernels_launched(run)
    assert f"nsd::{kernel}(" in names, names


# ------------------------------------------------------------------ K1 fast forward
N1, ND1 = 256, 24


def frontend_inputs(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, N1, generator=g)
    W = torch.eye(N1)[None] + 0.05 * torch.randn(ND1, N1, N1, generator=g)
    bias = 0.1 * torch.randn(ND1, 1, N1, generator=g)
    day = torch.randint(0, ND1, (B,), generator=g)
    day[-1] = day[0]                                            # a repeated day exercises the segment reduce
    return x.to(DEV), day.to(DEV), W.to(DEV), bias.to(DEV)


def fast_frontend(x, day, W, bias, K, S, noise=None, taps=None, flag=None):
    taps = O.gaussian_taps(2.0) if taps is None else taps
    return ops.frontend_fwd(x, day, W, bias, torch.from_numpy(taps).float().to(DEV), K, S, torch.bfloat16, flag, noise)


# (B, T, K, S): T - K = 9 S + 3 everywhere in the grid -> ten frames, a ragged tail and a partial last 32-row block
K1_CASES = [(3, K + 9 * S + 3, K, S) for K in (8, 16, 32, 64) for S in (4, 8)] + [
    (3, 8 + 9 * 12 + 3, 8, 12),        # stride longer than the window: rows between frames belong to no frame
    (2, 8, 8, 4), (2, 64, 64, 8),      # T == K: one frame
    (3, 32 + 4 - 1, 32, 4), (3, 16 + 8 - 1, 16, 8),        # T = K + S - 1: one frame and S - 1 unused rows
    (2, 64 + 33 * 4, 64, 4),           # 33 frames, 196 rows: one row into the seventh 32-row block
    (1, 2000, 32, 4), (1, 2000, 8, 12),                     # 16 segments of one utterance
    (256, 500, 32, 4),                                     # one segment per utterance
]


@pytest.mark.parametrize("noisy", [False, True], ids=["clean", "noise"])
@pytest.mark.parametrize("B,T,K,S", K1_CASES)
def test_frontend_fast_forward_sweep(B, T, K, S, noisy, poisoned):
    """The fast K1 forward (frontend_fwd_fast_kernel<K/8>) and the bf16 K1 backward at its kernelLen / stride: ys within 1e-5
    of the fp64 oracle, z within 1e-2 (bf16 day affine), patches == bf16(unfold(z)) bit for bit, fused noise == the kernel on
    ops.input_noise(x) bit for bit, the generic form (reached with a zero tap in front: 21 taps, same alignment) bit-identical,
    dW / db against the oracle evaluated on the kernel's own forward state, an out-of-range day flagged."""
    x, day, W, bias = frontend_inputs(B, T, B * 7919 + T + K + S)
    Tp = O.n_frames(T, K, S)
    used = (Tp - 1) * S + K
    noise = (0.8, 0.2, 31) if noisy else None
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    patches, ys, z = fast_frontend(x, day, W, bias, K, S, noise, flag=flag)
    assert int(flag.item()) == 0
    # every row a frame or the backward reads is written: [0, (Tp-1)*S+K)
    assert bool(torch.isfinite(patches).all()) and bool(torch.isfinite(ys[:, :used]).all()) and bool(torch.isfinite(z[:, :used]).all())
    xin = ops.input_noise(x, *noise) if noisy else x
    if noisy:
        plain = fast_frontend(xin, day, W, bias, K, S)
        assert torch.equal(patches, plain[0])
        assert torch.equal(ys[:, :used], plain[1][:, :used]) and torch.equal(z[:, :used], plain[2][:, :used])
    # the generic bf16 form: same FIR summation order (the zero tap adds +0 first), same mma day affine, same rounding
    generic = fast_frontend(x, day, W, bias, K, S, noise, taps=np.concatenate([[0.0], O.gaussian_taps(2.0)]).astype(np.float32))
    assert torch.equal(patches, generic[0])
    assert torch.equal(ys[:, :used], generic[1][:, :used]) and torch.equal(z[:, :used], generic[2][:, :used])

    # fp64 oracle on a few utterances (all of them when B is small); with B = 256 the sampled ones own three days alone
    ii = np.arange(B) if B <= 8 else np.array([0, B // 2, B - 1])
    idx = torch.from_numpy(ii).to(DEV)
    day_np = day.cpu().numpy()
    if B > 8:
        day_np = day_np % (ND1 - 3)
        day_np[ii] = [ND1 - 3, ND1 - 2, ND1 - 1]
        day = torch.from_numpy(day_np).to(DEV)
        patches, ys, z = fast_frontend(x, day, W, bias, K, S, noise)
    Wd, bd = W.double().cpu().numpy(), bias.double().cpu().numpy()
    taps64 = O.gaussian_taps(2.0).astype(np.float64)
    _, saved = O.frontend_fwd(xin[idx].double().cpu().numpy(), taps64, Wd, bd, day_np[ii], K, S)
    ys_k, z_k = ys[idx].double().cpu().numpy(), z[idx].double().cpu().numpy()
    np.testing.assert_allclose(ys_k[:, :used], saved["ys"][:, :used], rtol=1e-5, atol=2e-6)
    zerr = np.abs(z_k[:, :used] - saved["z"][:, :used]).max()
    assert zerr < 1e-2, zerr
    got = patches.view(Tp, B, N1 * K)[:, idx].permute(1, 0, 2).cpu()
    assert torch.equal(got, torch.from_numpy(O.unfold(z_k.astype(np.float32), K, S)).to(torch.bfloat16))

    g = torch.Generator(device=DEV).manual_seed(T + K)
    dp_bf = torch.randn(Tp * B, N1 * K, device=DEV, generator=g).to(torch.bfloat16)
    dW, db = ops.frontend_bwd(dp_bf, ys, z, day, ND1, K, S)
    assert bool(torch.isfinite(dW).all()) and bool(torch.isfinite(db).all())
    dp_r = dp_bf.view(Tp, B, N1 * K)[:, idx].permute(1, 0, 2).double().cpu().numpy()
    ys_k[:, used:] = 0.0                                      # never written by the forward, never read by the backward
    z_k[:, used:] = 0.0
    saved_k = {"ys": ys_k, "z": z_k, "pre": z_k / (1.0 - np.abs(z_k))}   # the backward is checked against the kernel's own forward state
    dW_ref, db_ref = O.frontend_bwd(dp_r, saved_k, Wd, day_np[ii], T, K, S)
    days = np.unique(day_np[ii])
    dW_k, db_k, dW_ref, db_ref = dW.cpu().numpy()[days], db.cpu().numpy()[days], dW_ref[days], db_ref[days]
    e_w = np.abs(dW_k - dW_ref).max() / np.abs(dW_ref).max()
    e_b = np.abs(db_k - db_ref).max() / max(np.abs(db_ref).max(), 1e-9)
    print(f"K1 B={B} T={T} K={K} S={S} noise={noisy}: max |z - oracle| {zerr:.2e}, dW err / max|dW| {e_w:.2e}, db {e_b:.2e}")
    assert e_w < 2e-2 and e_b < 2e-3

    bad = day.clone()
    bad[-1] = ND1
    fast_frontend(x, bad, W, bias, K, S, noise, flag=flag)
    assert int(flag.item()) == 1                               # reference: IndexError from index_select (model.py:89)


# ------------------------------------------------------------------ K3
def gru_recurrence_from(gi, w_hh, b_hh, h0):
    """fp64 GRU (nn.GRU gate order r|z|n, model.py:50-57) started from h0 instead of zeros.  gi [Tp,B,3H] includes b_ih."""
    H = h0.shape[1]
    sig = lambda v: 1.0 / (1.0 + np.exp(-v))
    h, out = h0, []
    for x in gi:
        gh = h @ w_hh.T + b_hh
        r, zg = sig(x[:, :H] + gh[:, :H]), sig(x[:, H:2 * H] + gh[:, H:2 * H])
        n = np.tanh(x[:, 2 * H:] + r * gh[:, 2 * H:])
        h = (1.0 - zg) * n + zg * h
        out.append(h)
    return np.stack(out)


@pytest.mark.parametrize("H", [128, 1024])
@pytest.mark.parametrize("B", [3, 70, 257])
def test_gru_tc_initial_state(B, H, poisoned):
    """K3 forward from a carried state h0 != 0 (the streaming exact form) against the fp64 recurrence started from h0;
    bf16 tolerance of test_gru_tc_fwd_bwd (h in [-1, 1]; bf16 state exchange + tanh.approx)."""
    Tp = 4
    rng = np.random.default_rng(B + H)
    w_hh = torch.from_numpy(rng.standard_normal((3 * H, H)) / np.sqrt(H)).to(torch.bfloat16)
    b_hh = rng.standard_normal(3 * H) * 0.1
    gi = rng.standard_normal((Tp, B, 3 * H)) * 0.8
    h0 = np.tanh(rng.standard_normal((B, H)))
    ref = gru_recurrence_from(gi, w_hh.double().numpy(), b_hh, torch.from_numpy(h0).float().double().numpy())
    hseq, hseq_bf, _ = ops.gru_fwd_bf16(torch.from_numpy(gi.reshape(Tp * B, 3 * H)).float().to(DEV), w_hh.to(DEV),
                                        torch.from_numpy(b_hh).float().to(DEV), Tp, B, H, 1, False, False,
                                        h0=torch.from_numpy(h0).float().to(DEV))
    got = hseq.view(Tp, B, H).double().cpu().numpy()
    err = np.abs(got - ref).max()
    print(f"gru_tc from h0 B={B} H={H}: max abs err {err:.2e}")
    assert np.isfinite(got).all() and err < 2.5e-2
    assert torch.equal(hseq_bf, hseq.to(torch.bfloat16))


@pytest.mark.parametrize("B,Tp,H,D", [(3, 5, 128, 1), (70, 4, 320, 2), (40, 3, 1024, 2)])
def test_gru_tc_strided_gi(B, Tp, H, D):
    """gi read through a row stride ldgi > D*3H (a column slice of a wider buffer) == the contiguous copy, bit for bit."""
    torch.manual_seed(B + H)
    wide = torch.randn(Tp * B, D * 3 * H + 96, device=DEV)
    gi = wide[:, 32:32 + D * 3 * H]
    w = (torch.randn(D * 3 * H, H, device=DEV) / H ** 0.5).to(torch.bfloat16)
    b = torch.randn(D * 3 * H, device=DEV) * 0.1
    strided = ops.gru_fwd_bf16(gi, w, b, Tp, B, H, D, False, True)
    contiguous = ops.gru_fwd_bf16(gi.contiguous(), w, b, Tp, B, H, D, False, True)
    assert torch.equal(strided[0], contiguous[0]) and torch.equal(strided[1], contiguous[1])
    for a, c in zip(strided[2], contiguous[2]):
        assert torch.equal(a, c)


# ------------------------------------------------------------------ streaming push
SMALL_A = dict(neural_dim=128, n_classes=10, hidden_dim=512, layer_dim=1, nDays=4, strideLen=2, kernelLen=16, gaussianSmoothWidth=2.0)
SMALL_B = dict(neural_dim=64, n_classes=40, hidden_dim=512, layer_dim=8, nDays=4, strideLen=1, kernelLen=8, gaussianSmoothWidth=2.0)
SMALL_C = dict(neural_dim=64, n_classes=12, hidden_dim=512, layer_dim=2, nDays=4, strideLen=8, kernelLen=16, gaussianSmoothWidth=2.0)


def stream_oracle(m, kw, X, day):
    from oracle import torch_port as P
    port = P.PortGRUDecoder(bidirectional=False, dropout=0.0, **kw)
    port.load_reference_state({k: v.detach().cpu() for k, v in m.state_dict().items()})
    return port_streaming_oracle(port.double().eval(), X.double(), day, frames_per_call=1).numpy()


def check_stream(sd, X, sizes, ref, off):
    """Push ``X`` in ``sizes`` bins at a time through ``sd``; the fast form's logits against the chunked fp64 oracle and the
    module's offline forward with the bounds of test_gpu_streaming.test_streaming_fast_form, greedy ids == argmax."""
    outs, fast_frames, pos = [], 0, 0
    for n in filter(None, sizes):
        o = sd.push(X[:, pos:pos + n].to(DEV))
        pos += n
        if o is not None:
            outs.append(o)
            if sd._steady:
                fast_frames += o.shape[1]
                assert torch.equal(sd.last_ids.long(), o[:, -1].argmax(-1))
    assert pos == X.shape[1]
    o = sd.finish()
    if o is not None:
        outs.append(o)
    got = torch.cat(outs, dim=1).cpu().numpy().astype(np.float64)
    assert got.shape == ref.shape and np.isfinite(got).all() and fast_frames >= 20
    e_ref, e_off = np.abs(got - ref).max(), np.abs(got - off).max()
    agree = (got.argmax(-1) == ref.argmax(-1)).mean()
    top2 = np.sort(ref, axis=-1)[..., -2:]
    flips = got.argmax(-1) != ref.argmax(-1)
    print(f"   {fast_frames} frames through the step kernel; vs oracle {e_ref:.3e}, vs offline forward {e_off:.3e}, argmax agreement {agree:.4f}")
    assert not (flips & ((top2[..., 1] - top2[..., 0]) > 2 * e_ref)).any()
    assert e_ref < 0.12 and agree >= 0.95 and e_off < 0.06


@pytest.mark.parametrize("kw,B,T", [(COMP, 2, 232), (COMP, 5, 232), (COMP, 7, 232), (SMALL_A, 3, 120), (SMALL_B, 2, 60)],
                         ids=["comp-B2", "comp-B5", "comp-B7", "H512-L1-N128-K16-S2", "H512-L8-N64-K8-S1"])
def test_streaming_fast_form_variants(kw, B, T, poisoned):
    """nsd_stream_push at every batch form and at architectures other than the competition one, with and without graph replay."""
    m = build_streaming_model(**kw)
    g = torch.Generator().manual_seed(B * 100 + T)
    X = torch.randn(B, T, kw["neural_dim"], generator=g)
    day = torch.randint(0, kw["nDays"], (B,), generator=g)
    ref = stream_oracle(m, kw, X, day)
    with torch.no_grad():
        off = m.forward(X.to(DEV), day.to(DEV)).cpu().numpy().astype(np.float64)
    S = kw["strideLen"]
    for use_graph in (False, True):
        sd = nsd.StreamingDecoder(m, B, day.to(DEV), use_graph=use_graph)
        assert sd.fast
        print(f"streaming B={B} graph={use_graph}")
        check_stream(sd, X, [S] * (T // S) + ([T % S] if T % S else []), ref, off)
        if use_graph:
            assert sd._graph is not None, getattr(sd, "_graph_error", "no graph captured")


def test_streaming_every_extra(poisoned):
    """extra = bins received beyond the newest frame's look-ahead is a kernel argument, fixed by the length of the push that
    engages the fast form.  A first push of K + right + 16 + e bins makes it e: every value in [0, S), each re-capturing the graph
    of the same decoder, each stream equal to the oracle."""
    kw, B, T = SMALL_C, 3, 240
    S = kw["strideLen"]
    m = build_streaming_model(**kw)
    g = torch.Generator().manual_seed(9)
    X = torch.randn(B, T, kw["neural_dim"], generator=g)
    day = torch.randint(0, kw["nDays"], (B,), generator=g)
    ref = stream_oracle(m, kw, X, day)
    with torch.no_grad():
        off = m.forward(X.to(DEV), day.to(DEV)).cpu().numpy().astype(np.float64)
    sd = nsd.StreamingDecoder(m, B, day.to(DEV))
    assert sd.fast
    for e in range(S):
        sd.reset()
        first = kw["kernelLen"] + sd.right + 16 + e
        n_steady = (T - first) // S
        sizes = [first] + [S] * n_steady + [T - first - S * n_steady]
        print(f"streaming extra={e}")
        check_stream(sd, X, sizes, ref, off)
        assert sd._extra == e and sd._graph is not None, getattr(sd, "_graph_error", "no graph captured")
