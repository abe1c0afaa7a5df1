"""Packed-sequence semantics of GRUDecoder: ``forward(X, dayIdx, X_len)`` and the ``packed=`` keyword of the trainer entry points.

Each utterance behaves as if it ran alone on X[b, :X_len[b]]: K1 reads bins past X_len as 0, the recurrence runs n_b frames per row
in both directions (nn.GRU on a pack_padded_sequence), the outputs past n_b are 0 and no gradient flows through them.  Checked
against the fp64 packed restatement (tests/packed_oracle.py), against the utterances run alone, against today's path, at the
kernel level against oracle/nsd_oracle.py per utterance, and through the trainer.
"""
from __future__ import annotations

import json
import os
import tempfile

import numpy as np
import pytest
import torch

from packed_oracle import frame_counts as oracle_frame_counts, packed_forward

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200 import ops, trainer
    from neural_speech_decoder_b200.model import gaussian_kernel_1d
    from neural_speech_decoder_b200.synthetic import fill_trained_like_, make_batch
    from oracle import nsd_oracle as O
    from oracle import torch_port as P

DEV = "cuda"
SMALL = dict(neural_dim=32, n_classes=10, hidden_dim=64, layer_dim=2, nDays=4, dropout=0.0, strideLen=4, kernelLen=16,
             gaussianSmoothWidth=2.0)
COMP = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, dropout=0.0, strideLen=4, kernelLen=32,
            gaussianSmoothWidth=2.0)
# bf16 bounds (rel L2 against the fp64 packed oracle; loss: relative error): about 3x the B200 measurements (1000 W power limit) in
# profiles/parity_packed.json -- small uni / bi: logits 3.9e-3, loss 5.4e-4, gradients 5.3e-3, X.grad 5.1e-3; comp bi: 6.4e-3,
# 2.0e-4, 1.6e-2, 1.6e-2
BF16_TOL = {"small": dict(logits=0.012, loss=1.6e-3, grad=0.016, xgrad=0.016), "comp": dict(logits=0.02, loss=6e-4, grad=0.05, xgrad=0.05)}
# fp32: rtol 1e-3 with atol a fraction of the largest entry (entries cross zero), as the full-shape parity tests use
FP32_ATOL = {"small": 1e-5, "comp": 1e-4}


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


def record(key, val):
    path = os.path.join(os.environ.get("NSD_PARITY_OUT") or tempfile.gettempdir(), "parity_packed.json")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    try:
        cur = json.load(open(path))
    except Exception:
        cur = {}
    cur[key] = val
    json.dump(cur, open(path, "w"), indent=1, sort_keys=True)


def _rel_l2(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _model(kw, precision, seed=3):
    torch.manual_seed(0)
    m = nsd.GRUDecoder(device=DEV, **kw)
    fill_trained_like_(m, seed=seed)
    m.precision = precision
    return m.to(DEV).eval()


def _port_of(m, kw):
    port = P.PortGRUDecoder(**dict(kw, dropout=0.0, bidirectional=m.bidirectional))
    port.load_reference_state({k: v.detach().cpu() for k, v in m.state_dict().items()})
    return port.double().eval()


def _batch(kw, B, T, seed):
    X, y, X_len, y_len, day = make_batch(B, T, n_feat=kw["neural_dim"], n_days=kw["nDays"], n_classes=kw["n_classes"], seed=seed,
                                         ragged=True, kernel_len=kw["kernelLen"], stride_len=kw["strideLen"], min_tgt=2,
                                         max_tgt=min(12, (kw["kernelLen"] + T) // 8))
    X_len[1] = kw["kernelLen"]                            # one frame
    y_len[1] = 0
    y[1] = 0
    X[1, kw["kernelLen"]:] = 0.0
    assert int(X_len[0]) == T                             # the whole batch length
    return X, y, X_len, y_len, day


def _run(m, X, y, X_len, y_len, day, packed=True, x_grad=True):
    """-> (logits, loss, {param: grad}, X.grad) with X_len passed to the forward when ``packed``."""
    m.zero_grad(set_to_none=True)
    Xd = X.to(DEV).requires_grad_(x_grad)
    logits = m(Xd, day.to(DEV), X_len.to(DEV)) if packed else m(Xd, day.to(DEV))
    lens = nsd.out_lens(X_len.to(DEV), m.kernelLen, m.strideLen)
    loss = nsd.ctc_loss_from_logits(logits, y.to(DEV), lens, y_len.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    grads = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
    return logits.detach(), loss.detach(), grads, (Xd.grad.detach() if x_grad else None)


def _oracle(port, X, y, X_len, y_len, day, kernel_len, stride_len):
    Xd = X.double().requires_grad_(True)
    logits = packed_forward(port, Xd, day, X_len)
    lens = ((X_len - kernel_len) / stride_len).to(torch.int32)
    lp = logits.log_softmax(2).permute(1, 0, 2)
    loss = torch.nn.CTCLoss(blank=0, reduction="mean", zero_infinity=True)(lp, y.long(), lens, y_len)
    port.zero_grad(set_to_none=True)
    loss.backward()
    grads = {}
    for k, p in port.named_parameters():
        if p.grad is None:
            continue
        if k.startswith("gru."):
            k = "gru_decoder." + k[4:]
        elif k.startswith("fc."):
            k = "fc_decoder_out." + k[3:]
        grads[k] = p.grad.detach()
    return logits.detach(), loss.detach(), grads, Xd.grad.detach()


# ------------------------------------------------------------------------------------------------- 1. parity with packed nn.GRU
PARITY = [("small", "uni", 6, 90), ("small", "bi", 6, 90), ("comp", "bi", 64, 500)]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("arch,direction,B,T", PARITY, ids=[f"{a}_{d}" for a, d, _, _ in PARITY])
def test_parity_with_packed_gru(arch, direction, B, T, precision):
    kw = dict(SMALL if arch == "small" else COMP, bidirectional=direction == "bi")
    m = _model(kw, precision)
    X, y, X_len, y_len, day = _batch(kw, B, T, seed=11)
    X[2, int(X_len[2]):] = 1e30                           # the padding is not read
    logits, loss, grads, xg = _run(m, X, y, X_len, y_len, day)
    ref_logits, ref_loss, ref_grads, ref_xg = _oracle(_port_of(m, kw), X, y, X_len, y_len, day, kw["kernelLen"], kw["strideLen"])
    n = oracle_frame_counts(X_len, kw["kernelLen"], kw["strideLen"], T)
    got = logits.cpu().double()
    valid = torch.arange(got.shape[1]).view(1, -1) < n.view(-1, 1)
    # past its frames every utterance's logits are exactly the output bias, in both precisions
    bias = m.fc_decoder_out.bias.detach().cpu().double()
    assert torch.equal(got[~valid], bias.expand(int((~valid).sum()), -1))
    errs = dict(logits=_rel_l2(got[valid], ref_logits[valid]), loss=abs(float(loss) - float(ref_loss)) / abs(float(ref_loss)),
                xgrad=_rel_l2(xg.cpu(), ref_xg))
    errs["grad"] = max(_rel_l2(grads[k].cpu(), ref_grads[k]) for k in ref_grads)
    Xs = X_len.view(-1, 1)
    assert torch.all(xg.cpu()[torch.arange(T).view(1, -1) >= Xs] == 0)          # no gradient at padded bins
    print(f"{arch}_{direction}_{precision}: {errs}")
    record(f"{arch}_{direction}_{precision}", errs)
    if precision == "fp32":
        np.testing.assert_allclose(got[valid].numpy(), ref_logits[valid].numpy(), rtol=1e-3, atol=2e-5)
        np.testing.assert_allclose(float(loss), float(ref_loss), rtol=1e-3)
        a = FP32_ATOL[arch]
        for k, r in ref_grads.items():
            np.testing.assert_allclose(grads[k].cpu().double().numpy(), r.numpy(), rtol=1e-3, atol=a * max(1.0, r.abs().max().item()), err_msg=k)
        np.testing.assert_allclose(xg.cpu().double().numpy(), ref_xg.numpy(), rtol=1e-3, atol=a * max(1.0, ref_xg.abs().max().item()))
    else:
        for k, bound in BF16_TOL[arch].items():
            assert errs[k] < bound, (k, errs[k], bound)


# ------------------------------------------------------------------------------------------------- 2. batch invariance
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_batch_invariance(precision):
    kw = dict(SMALL, bidirectional=True)
    m = _model(kw, precision)
    B, T = 6, 90
    X, y, X_len, y_len, day = _batch(kw, B, T, seed=21)
    b = 3
    nb = int(oracle_frame_counts(X_len, 16, 4, T)[b])
    L = int(X_len[b])

    def fwd(X_, day_, X_len_):
        with torch.no_grad():
            return m(X_.to(DEV), day_.to(DEV), X_len_.to(DEV))[b, :nb].cpu()

    base = fwd(X, day, X_len)
    # the other utterances replaced (data, day and length)
    X2, _, X_len2, _, day2 = _batch(kw, B, T, seed=22)
    X2[b], X_len2[b], day2[b] = X[b], X_len[b], day[b]
    assert torch.equal(fwd(X2, day2, X_len2), base)
    # its own padding refilled with large values and NaN: the mask selects
    X3 = X.clone()
    X3[b, L:] = 1e30
    X3[b, L + 1::2] = float("nan")
    assert torch.equal(fwd(X3, day, X_len), base)
    # more padding for everyone
    X4 = torch.cat([X, torch.full((B, 37, X.shape[2]), 5.0)], dim=1)
    grown = fwd(X4, day, X_len)
    # against the utterance run alone (B = 1, T = X_len)
    with torch.no_grad():
        alone = m(X[b:b + 1, :L].to(DEV), day[b:b + 1].to(DEV), X_len[b:b + 1].to(DEV))[0].cpu()
    print(f"{precision}: longer T bit-exact={torch.equal(grown, base)}, alone bit-exact={torch.equal(alone, base)}, "
          f"alone max|diff|={float((alone - base).abs().max()):.3g}")
    record(f"invariance_{precision}", dict(longer_T_bits_equal=bool(torch.equal(grown, base)), alone_bits_equal=bool(torch.equal(alone, base)),
                                           alone_max_abs_diff=float((alone - base).abs().max())))
    assert torch.equal(grown, base)
    tol = dict(rtol=1e-3, atol=2e-5) if precision == "fp32" else dict(rtol=2e-2, atol=2e-2)
    np.testing.assert_allclose(alone.numpy(), base.numpy(), **tol)


# ------------------------------------------------------------------------------------------------- 3. consistency with today's path
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("direction", ["uni", "bi"])
def test_full_lengths_equal_unpacked(precision, direction):
    kw = dict(SMALL, bidirectional=direction == "bi")
    m = _model(kw, precision)
    X, y, _, y_len, day = _batch(kw, 5, 80, seed=31)
    X_len = torch.full((5,), 80, dtype=torch.int32)
    y_len = y_len.clamp(max=8)
    a = _run(m, X, y, X_len, y_len, day, packed=False)
    b = _run(m, X, y, X_len, y_len, day, packed=True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[3], b[3])
    for k in a[2]:
        assert torch.equal(a[2][k], b[2][k]), k


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_unidirectional_zero_padded_matches_unpacked(precision):
    kw = dict(SMALL, bidirectional=False)
    m = _model(kw, precision)
    X, y, X_len, y_len, day = _batch(kw, 6, 90, seed=41)               # make_batch zero-pads past X_len
    n = oracle_frame_counts(X_len, 16, 4, 90)
    with torch.no_grad():
        a = m(X.to(DEV), day.to(DEV)).cpu()
        b = m(X.to(DEV), day.to(DEV), X_len.to(DEV)).cpu()
    for u in range(6):
        assert torch.equal(a[u, :int(n[u])], b[u, :int(n[u])]), u


# ------------------------------------------------------------------------------------------------- 4. kernel level
def _oracle_dirs(gi, w_hh, b_hh, n, D, H, dh=None):
    """Per utterance on its own frames: hseq [B,Tp,D*H] (0 past n_b) and, with ``dh``, dgi [B,Tp,D*3H]."""
    B, Tp, _ = gi.shape
    hseq = np.zeros((B, Tp, D * H))
    dgi = np.zeros((B, Tp, D * 3 * H))
    for b in range(B):
        nb = int(n[b])
        if nb == 0:
            continue
        for d in range(D):
            g = gi[b:b + 1, :nb, d * 3 * H:(d + 1) * 3 * H]
            h, saved = O.gru_dir_fwd(g, None, w_hh[d], None, b_hh[d], reverse=d == 1)
            hseq[b, :nb, d * H:(d + 1) * H] = h[0]
            if dh is not None:
                dg, _, _, _, _ = O.gru_dir_bwd(dh[b:b + 1, :nb, d * H:(d + 1) * H], saved, None, w_hh[d], reverse=d == 1)
                dgi[b, :nb, d * 3 * H:(d + 1) * 3 * H] = dg[0]
    return hseq, dgi


KERNEL_CASES = [(3, 7, 128, 2), (40, 6, 1024, 2), (70, 5, 320, 1), (257, 4, 128, 2)]      # the dispatch's chain forms (B <= 64, B > 64)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("B,Tp,H,D", KERNEL_CASES)
def test_recurrence_kernels_with_frame_counts(B, Tp, H, D, precision, poisoned):
    rng = np.random.default_rng([B, Tp, H, D])
    n = rng.integers(1, Tp + 1, size=B)
    n[0], n[-1] = Tp, 1
    if B > 2:
        n[1] = 0
    gi = rng.standard_normal((Tp, B, D * 3 * H)) * 0.5
    w_hh = rng.standard_normal((D, 3 * H, H)) / np.sqrt(H)
    b_hh = rng.standard_normal((D, 3 * H)) * 0.1
    dh = rng.standard_normal((Tp, B, D * H))
    nf = torch.from_numpy(n.astype(np.int32)).to(DEV)
    gi_t = torch.from_numpy(gi.reshape(Tp * B, -1).astype(np.float32)).to(DEV)
    dh_t = torch.from_numpy(dh.reshape(Tp * B, -1).astype(np.float32)).to(DEV)
    if precision == "bf16":
        w_bf = torch.from_numpy(w_hh.reshape(D * 3 * H, H).astype(np.float32)).to(DEV).bfloat16()
        w_used = w_bf.float().cpu().numpy().astype(np.float64).reshape(D, 3 * H, H)
        hseq, hseq_bf, saves, hdrop = ops.gru_fwd_bf16(gi_t, w_bf, torch.from_numpy(b_hh.reshape(-1).astype(np.float32)).to(DEV),
                                                       Tp, B, H, D, False, True, 0.3, 99, n_frames=nf)
        wT = torch.stack([w_bf[d * 3 * H:(d + 1) * 3 * H].t() for d in range(D)]).reshape(D * H, 3 * H).contiguous()
        db_ih = torch.empty(D * 3 * H, device=DEV)
        db_hh = torch.empty(D * 3 * H, device=DEV)
        dgi, dgh = ops.gru_bwd_bf16(dh_t, hseq, saves, wT, Tp, B, H, D, False, 0.0, 0, db_ih, db_hh, n_frames=nf)
        tol_h, tol_g = 3e-2, 6e-2
    else:
        w_used = w_hh
        hseq = torch.empty((Tp * B, D * H), device=DEV)
        saves = [tuple(torch.empty((Tp * B, H), device=DEV) for _ in range(4)) for _ in range(D)]
        dgi = torch.empty((Tp * B, D * 3 * H), device=DEV)
        dghn = [torch.empty((Tp * B, H), device=DEV) for _ in range(D)]
        for d in range(D):
            ops.gru_fwd_f32(gi_t, D * 3 * H, d * 3 * H, torch.from_numpy(w_hh[d].astype(np.float32)).to(DEV),
                            torch.from_numpy(b_hh[d].astype(np.float32)).to(DEV), Tp, B, H, d == 1, hseq, D * H, d * H, saves[d], n_frames=nf)
        for d in range(D):
            ops.gru_bwd_f32(dh_t, D * H, d * H, hseq, D * H, d * H, saves[d], torch.from_numpy(w_hh[d].astype(np.float32)).to(DEV),
                            Tp, B, H, d == 1, dgi, D * 3 * H, d * 3 * H, dghn[d], n_frames=nf)
        tol_h, tol_g = 1e-4, 1e-3
    torch.cuda.synchronize()
    ref_h, ref_g = _oracle_dirs(gi.transpose(1, 0, 2), w_used, b_hh, n, D, H, dh.transpose(1, 0, 2))
    got_h = hseq.cpu().double().numpy().reshape(Tp, B, D * H).transpose(1, 0, 2)
    got_g = dgi.float().cpu().double().numpy().reshape(Tp, B, D * 3 * H).transpose(1, 0, 2)
    pad = np.arange(Tp)[None, :] >= n[:, None]
    assert np.all(got_h[pad] == 0) and np.all(got_g[pad] == 0)
    assert np.isfinite(got_h).all() and np.isfinite(got_g).all()
    eh, eg = _rel_l2(got_h, ref_h), _rel_l2(got_g, ref_g)
    print(f"B={B} Tp={Tp} H={H} D={D} {precision}: hseq {eh:.3g} dgi {eg:.3g}")
    assert eh < tol_h and eg < tol_g, (eh, eg)
    if precision == "bf16":
        assert torch.all(hdrop.float().cpu().reshape(Tp, B, -1).permute(1, 0, 2)[torch.from_numpy(pad)] == 0)
        dgh_np = dgh.float().cpu().double().numpy().reshape(Tp, B, D * 3 * H).transpose(1, 0, 2)
        assert np.all(dgh_np[pad] == 0)
        # the bias sums cover the valid steps only
        ref_bih = ref_g.reshape(-1, D * 3 * H).sum(0)
        assert _rel_l2(db_ih.cpu(), ref_bih) < tol_g


FRONT_CASES = [("fast", 4, 232, 256, 32, 4), ("generic_bf16", 3, 120, 64, 16, 4)]


@pytest.mark.parametrize("noisy", [False, True], ids=["clean", "noise"])
@pytest.mark.parametrize("name,B,T,N,K,S", FRONT_CASES, ids=[c[0] for c in FRONT_CASES])
def test_frontend_with_lengths(name, B, T, N, K, S, noisy, poisoned):
    rng = np.random.default_rng([B, T, N])
    X = torch.from_numpy(rng.standard_normal((B, T, N)).astype(np.float32))
    x_len = torch.tensor([T, K] + [int(v) for v in rng.integers(K, T, size=B - 2)], dtype=torch.int64)
    garbage = X.clone()
    for b in range(B):
        garbage[b, int(x_len[b]):] = float("nan") if b % 2 else 1e30
    day = torch.from_numpy(rng.integers(0, 3, size=B)).to(DEV)
    dw = torch.eye(N).repeat(3, 1, 1).to(DEV) + 0.01 * torch.randn(3, N, N, device=DEV)
    db = 0.1 * torch.randn(3, 1, N, device=DEV)
    taps = gaussian_kernel_1d(20, 2.0).to(DEV)
    noise = (0.8, 0.2, 1234) if noisy else None
    xl = x_len.to(DEV)
    outs = []
    for Xi in (X, garbage):
        p, _, z = ops.frontend_fwd(Xi.to(DEV), day, dw, db, taps, K, S, torch.bfloat16, None, noise, x_len=xl)
        outs.append((p.float().cpu(), z))
    Tp = (T - K) // S + 1
    n = oracle_frame_counts(x_len, K, S, T)
    pa = outs[0][0].view(Tp, B, -1)
    pb = outs[1][0].view(Tp, B, -1)
    for b in range(B):
        assert torch.equal(pa[:int(n[b]), b], pb[:int(n[b]), b]), b           # padded bins contribute nothing, noise or not
    # dx is exactly 0 at padded bins
    dp = torch.randn(Tp * B, N * K, device=DEV).bfloat16()
    dx = ops.frontend_bwd_input(dp, outs[1][1], day, dw, taps, K, S, x_len=xl).cpu()
    assert torch.isfinite(dx).all()
    for b in range(B):
        assert torch.all(dx[b, int(x_len[b]):] == 0), b
        assert torch.any(dx[b, :int(x_len[b])] != 0), b
    nf = ops.frame_counts(xl, T, K, S)
    assert torch.equal(nf.cpu().long(), n)


# ------------------------------------------------------------------------------------------------- 5. trainer level
def test_eval_batch_packed_is_sum_of_utterances():
    kw = dict(SMALL, bidirectional=True)
    m = _model(kw, "bf16")
    X, y, X_len, y_len, day = make_batch(6, 90, n_feat=32, n_days=4, n_classes=10, seed=51, ragged=True, kernel_len=16, stride_len=4,
                                         min_tgt=2, max_tgt=6)
    dev = lambda *ts: [t.to(DEV) for t in ts]
    _, dist, tot = trainer.eval_batch(m, *dev(X, y, X_len, y_len, day), packed=True)
    ds = ts = 0
    for b in range(6):
        L = int(X_len[b])
        _, d1, t1 = trainer.eval_batch(m, *dev(X[b:b + 1, :L], y[b:b + 1, :int(y_len[b])], X_len[b:b + 1], y_len[b:b + 1], day[b:b + 1]),
                                       packed=True)
        ds, ts = ds + int(d1), ts + int(t1)
    assert (int(dist), int(tot)) == (ds, ts)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_input_attribution_packed_zero_at_padding(precision):
    kw = dict(SMALL, bidirectional=True)
    m = _model(kw, precision)
    X, y, X_len, y_len, day = make_batch(5, 90, n_feat=32, n_days=4, n_classes=10, seed=52, ragged=True, kernel_len=16, stride_len=4,
                                         min_tgt=2, max_tgt=6)
    att, nll = trainer.input_attribution(m, X.to(DEV), y.to(DEV), X_len.to(DEV), y_len.to(DEV), day.to(DEV), packed=True)
    att = att.cpu()
    for b in range(5):
        assert torch.all(att[b, int(X_len[b]):] == 0), b
        assert torch.any(att[b, :int(X_len[b])] != 0), b
    assert torch.isfinite(nll).all()


def test_train_step_packed_matches_oracle_adam():
    kw = dict(SMALL, bidirectional=True)
    m = _model(kw, "fp32").train()
    port = _port_of(m, kw)
    X, y, X_len, y_len, day = _batch(kw, 6, 90, seed=61)
    args = dict(lrStart=0.02, lrEnd=0.02, nBatch=10, l2_decay=1e-5)
    opt, _ = trainer.make_optimizer(m, args)
    p0 = {k: p.detach().cpu().double().clone() for k, p in m.named_parameters()}
    loss = trainer.train_step(m, opt, X.to(DEV), y.to(DEV), X_len.to(DEV), y_len.to(DEV), day.to(DEV), packed=True)
    ref_opt = P.make_adam(port, lr=0.02, l2=1e-5)
    ref_opt.zero_grad()
    _, ref_loss, _, _ = _oracle(port, X, y, X_len, y_len, day, 16, 4)
    ref_opt.step()
    np.testing.assert_allclose(float(loss), float(ref_loss), rtol=1e-4)
    ref_params = {}
    for k, p in port.named_parameters():
        name = "gru_decoder." + k[4:] if k.startswith("gru.") else "fc_decoder_out." + k[3:] if k.startswith("fc.") else k
        ref_params[name] = p.detach()
    for k, p in m.named_parameters():
        if k not in ref_params:
            continue
        d_got = p.detach().cpu().double() - p0[k]
        d_ref = ref_params[k] - p0[k]
        assert _rel_l2(d_got, d_ref) < 2e-3, (k, _rel_l2(d_got, d_ref))


def test_out_of_range_lengths_raise():
    kw = dict(SMALL, bidirectional=True)
    m = _model(kw, "bf16")
    X, _, X_len, _, day = make_batch(4, 90, n_feat=32, n_days=4, n_classes=10, seed=71, ragged=True, kernel_len=16, stride_len=4)
    for bad in (15, 91):
        L = X_len.clone()
        L[2] = bad
        with pytest.raises(ValueError):
            m(X.to(DEV), day.to(DEV), L)
        out = m(X.to(DEV), day.to(DEV), L.to(DEV))
        assert torch.isfinite(out).all()
        with pytest.raises(ValueError):
            m.check_errors()
        m.check_errors()                                  # the flag was cleared
    m(X.to(DEV), day.to(DEV), X_len.to(DEV))
    m.check_errors()


def test_streaming_initial_state_and_frame_counts_do_not_combine():
    gi = torch.zeros((4 * 3, 3 * 64), device=DEV)
    w = torch.zeros((3 * 64, 64), device=DEV, dtype=torch.bfloat16)
    with pytest.raises(nsd.NsdError):
        ops.gru_fwd_bf16(gi, w, torch.zeros(3 * 64, device=DEV), 4, 3, 64, 1, False, False, h0=torch.zeros((3, 64), device=DEV),
                         n_frames=torch.full((3,), 4, dtype=torch.int32, device=DEV))
