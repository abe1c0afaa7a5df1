"""K3 tensor-core recurrence (tcgen05, persistent, both directions in one launch) and the bf16 model path,
against the numpy oracle run on bf16-rounded weights.  bf16 tolerances are stated per check."""
import numpy as np
import pytest
import torch

from conftest import golden_ctor, golden_state, load_golden
from oracle import nsd_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from neural_speech_decoder_b200 import ops
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200.synthetic import fill_trained_like_

DEV = "cuda"


def bf(a):
    return torch.from_numpy(np.asarray(a, dtype=np.float32)).to(torch.bfloat16).float().numpy().astype(np.float64)


def cu(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).to(DEV)


@pytest.mark.parametrize("B,Tp,H,D,rev0", [(3, 7, 64, 1, 0), (3, 7, 64, 1, 1), (5, 1, 64, 2, 0), (70, 5, 128, 2, 0),
                                           (64, 6, 1024, 2, 0), (64, 4, 1024, 1, 0), (16, 9, 256, 2, 0),
                                           # B > 64: four 32-row chains in flight; partial last chain, missing chains, two chain groups
                                           (100, 6, 256, 2, 0), (130, 5, 1024, 2, 0), (200, 4, 128, 1, 1),
                                           # ring stages of several boxes: 192 / 320 / 576 / 960 unaligned (boxes straddle zones,
                                           # partial last box; the BPTT at 960 fills the 96 KB ring bound), 512 / 768 chunked
                                           (5, 3, 192, 2, 0), (5, 4, 320, 2, 0), (5, 3, 512, 2, 0), (5, 5, 576, 2, 0),
                                           (5, 3, 768, 2, 0), (5, 4, 960, 2, 0),
                                           # batch edges: one row, whole chain groups, three or more chain groups (B > 256)
                                           *[(B, 3, H, 2, 0) for H in (128, 256) for B in (1, 32, 64, 128, 256, 257, 300)],
                                           (300, 3, 1024, 2, 0)])
def test_gru_tc_fwd_bwd(B, Tp, H, D, rev0):
    rng = np.random.default_rng(H + Tp + B)
    M = Tp * B
    w_hh = [bf(rng.standard_normal((3 * H, H)) / np.sqrt(H)) for _ in range(D)]
    b_hh = [rng.standard_normal(3 * H) * 0.1 for _ in range(D)]
    gi = rng.standard_normal((B, Tp, D * 3 * H)) * 0.8
    # oracle: the input projection is the identity (x = gi, W_ih = I, b_ih = 0)
    eye, zero = np.eye(3 * H), np.zeros(3 * H)
    href, saved = [], []
    for d in range(D):
        reverse = (d == 1) or bool(rev0)
        h, sv = O.gru_dir_fwd(gi[:, :, d * 3 * H:(d + 1) * 3 * H], eye, w_hh[d], zero, b_hh[d], reverse)
        href.append(h); saved.append(sv)
    href = np.concatenate(href, axis=2)                                     # [B,Tp,D*H]
    gi_tm = cu(gi.transpose(1, 0, 2).reshape(M, D * 3 * H))
    w_bf = cu(np.concatenate(w_hh, 0), torch.bfloat16)
    hseq, hseq_bf, sv = ops.gru_fwd_bf16(gi_tm, w_bf, cu(np.concatenate(b_hh)), Tp, B, H, D, rev0, True)
    got = hseq.view(Tp, B, D * H).permute(1, 0, 2).cpu().numpy()
    err = np.abs(got - href).max()
    print(f"gru_tc fwd max abs err {err:.2e}")
    assert err < 2.5e-2                                                     # h in [-1,1]; bf16 state exchange + tanh.approx
    assert torch.equal(hseq_bf, hseq.to(torch.bfloat16))
    for d in range(D):
        for name, t in zip(("r", "z", "n", "hn"), sv):
            ref = saved[d][name].transpose(1, 0, 2).reshape(M, H)
            assert np.abs(t[d].cpu().numpy() - ref).max() < 4e-2, name

    dh = rng.standard_normal((B, Tp, D * H))
    dh_tm = cu(dh.transpose(1, 0, 2).reshape(M, D * H))
    whT = torch.cat([cu(w_hh[d], torch.bfloat16).T.contiguous() for d in range(D)], 0)      # [D*H, 3H]
    dgi, dgh = ops.gru_bwd_bf16(dh_tm, hseq, sv, whT, Tp, B, H, D, rev0)
    dgi_np, dgh_np = dgi.float().cpu().numpy().astype(np.float64), dgh.float().cpu().numpy().astype(np.float64)
    for d in range(D):
        reverse = (d == 1) or bool(rev0)
        dx_ref, dwi_ref, dwh_ref, dbi_ref, dbh_ref = O.gru_dir_bwd(dh[:, :, d * H:(d + 1) * H], saved[d], eye, w_hh[d], reverse)
        dgi_ref = dx_ref.transpose(1, 0, 2).reshape(M, 3 * H)               # W_ih = I  =>  dx == dgi
        sl = slice(d * 3 * H, (d + 1) * 3 * H)
        scale = np.abs(dgi_ref).max()
        e1 = np.abs(dgi_np[:, sl] - dgi_ref).max() / scale
        print(f"gru_tc bwd dir {d} max err / max |dgi| = {e1:.2e}")
        assert e1 < 4e-2
        hprev = saved[d]["hprev"].transpose(1, 0, 2).reshape(M, H)
        dwh = dgh_np[:, sl].T @ hprev
        assert np.abs(dwh - dwh_ref).max() < 4e-2 * max(1.0, np.abs(dwh_ref).max())


@pytest.mark.parametrize("name", ["comp_uni", "comp_bi"])
def test_bf16_model_matches_reference_fixture(name):
    """bf16 mode of the whole drop-in module on the competition architecture; tolerance stated separately from fp32
    (north star): logits within 6e-2 absolute of the reference's fp32 logits (|logits| is O(1..10) with these weights),
    loss within 2 %, identical greedy decisions on every frame whose top-2 margin exceeds 0.12, gradients within 10 % in relative L2 norm."""
    g = load_golden(name + "_f32")
    kw = dict(golden_ctor(g))
    nsd.set_default_precision("bf16")
    try:
        torch.manual_seed(0)
        m = nsd.GRUDecoder(device=DEV, **kw)
    finally:
        nsd.set_default_precision("fp32")
    fill_trained_like_(m, seed=7)
    m = m.to(DEV).eval()
    X, day = torch.from_numpy(g["X"]).to(DEV), torch.from_numpy(g["dayIdx"]).to(DEV)
    y, X_len, y_len = (torch.from_numpy(g[k]).to(DEV) for k in ("y", "X_len", "y_len"))
    pred = m.forward(X, day)
    lens = nsd.out_lens(X_len, m.kernelLen, m.strideLen)
    loss = nsd.ctc_loss_from_logits(pred, y, lens, y_len)
    loss.backward()
    ref = g["logits"]
    err = np.abs(pred.detach().cpu().numpy() - ref).max()
    print(f"{name}: bf16 logits max abs err {err:.3e} (|ref| max {np.abs(ref).max():.2f}), loss {loss.item():.5f} vs {float(g['loss']):.5f}")
    assert err < 6e-2
    np.testing.assert_allclose(loss.item(), g["loss"], rtol=2e-2)
    # greedy decisions must agree wherever the reference's top-2 margin exceeds twice the logit error bound
    top2 = np.sort(ref, axis=-1)[..., -2:]
    clear = (top2[..., 1] - top2[..., 0]) > 2 * 6e-2
    same = pred.detach().argmax(-1).cpu().numpy() == ref.argmax(-1)
    assert same[clear].all() and same.mean() >= 0.9
    params = dict(m.named_parameters())
    for n in [str(n) for n in g["live_grad_names"]]:
        gr = params[n].grad.detach().reshape(-1)
        step = max(1, gr.numel() // 4096)
        rs = g["gsample." + n].astype(np.float64)
        got = gr[::step][:4096].cpu().numpy().astype(np.float64)
        rel = np.linalg.norm(got - rs) / max(np.linalg.norm(rs), 1e-12)
        print(f"   grad {n}: rel L2 err {rel:.3e}")
        assert rel < 0.1, n


@pytest.mark.parametrize("B,Tp,H,D", [(64, 5, 1024, 2), (40, 6, 128, 2), (7, 4, 64, 1)])
def test_gru_tc_fused_dropout_and_bias_sums(B, Tp, H, D):
    """The fused forms must equal the separate kernels: the dropped copy written by the forward epilogue == nsd_dropout
    of the bf16 states (bit-exact), the BPTT with the mask applied on load == BPTT of nsd_dropout(dh) (bit-exact), and
    the in-kernel bias gradients == fp32 column sums of dgi / dgh up to their bf16 rounding."""
    torch.manual_seed(B + H)
    M = Tp * B
    gi = torch.randn(M, D * 3 * H, device=DEV)
    w = (torch.randn(D * 3 * H, H, device=DEV) / np.sqrt(H)).to(torch.bfloat16)
    b = torch.randn(D * 3 * H, device=DEV) * 0.1
    p, seed = 0.4, 1234
    hseq, hbf, sv, hdrop = ops.gru_fwd_bf16(gi, w, b, Tp, B, H, D, False, True, p, seed)
    hseq2, hbf2, sv2 = ops.gru_fwd_bf16(gi, w, b, Tp, B, H, D, False, True)
    assert torch.equal(hseq, hseq2) and torch.equal(hbf, hbf2)
    assert torch.equal(hdrop, ops.dropout(hbf, p, seed))
    keep = (hdrop != 0).float().mean().item()
    assert abs(keep - 0.6) < 0.02

    wT = torch.cat([w[d * 3 * H:(d + 1) * 3 * H].T.contiguous() for d in range(D)], 0)
    dh = torch.randn(M, D * H, device=DEV)
    db_ih = torch.full((D * 3 * H,), 7.0, device=DEV)      # must be overwritten, not accumulated into
    db_hh = torch.full((D * 3 * H,), -3.0, device=DEV)
    dgi, dgh = ops.gru_bwd_bf16(dh, hseq, sv, wT, Tp, B, H, D, False, p, seed, db_ih, db_hh)
    dgi_ref, dgh_ref = ops.gru_bwd_bf16(ops.dropout(dh, p, seed), hseq, sv, wT, Tp, B, H, D, False)
    assert torch.equal(dgi, dgi_ref) and torch.equal(dgh, dgh_ref)
    for got, mat in ((db_ih, dgi), (db_hh, dgh)):
        ref = mat.double().sum(0)
        # each of the M summands carries a bf16 rounding error of at most 2^-9 relative in `mat`, none in `got`
        tol = mat.double().abs().sum(0) * 2.0 ** -8 + 1e-6
        assert bool(((got.double() - ref).abs() <= tol).all())
    # run-to-run determinism of the two-warpgroup accumulation
    db2_ih, db2_hh = torch.empty_like(db_ih), torch.empty_like(db_hh)
    ops.gru_bwd_bf16(dh, hseq, sv, wT, Tp, B, H, D, False, p, seed, db2_ih, db2_hh)
    assert torch.equal(db_ih, db2_ih) and torch.equal(db_hh, db2_hh)
