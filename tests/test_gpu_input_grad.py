"""Gradients with respect to the neural input: the K1 input-gradient kernel (nsd_frontend_bwd_input), X.grad of GRUDecoder (fp32
and bf16) and of the Conformer against fp64 restatements of the reference, the backward that skips the parameter work of frozen
weights, and input_attribution (saliency, integrated gradients).

Measured errors go to parity_input_grad.json in the directory $NSD_PARITY_OUT names (default: the system's temporary directory);
profiles/parity_input_grad.json holds the B200 measurements the bounds below are set from (each bound is at most 3x its measurement).
"""
import json
import os
import tempfile

import numpy as np
import pytest
import torch

from frontend_input_oracle import frontend_bwd_input as oracle_bwd_input

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import neural_speech_decoder_b200 as nsd
    from neural_speech_decoder_b200 import _lib, ops
    from neural_speech_decoder_b200.model import gaussian_kernel_1d
    from neural_speech_decoder_b200.synthetic import fill_trained_like_, make_batch

DEV = "cuda"
SMALL = dict(neural_dim=32, n_classes=10, hidden_dim=64, layer_dim=2, nDays=4, dropout=0.0, strideLen=4, kernelLen=16,
             gaussianSmoothWidth=2.0)
COMP = dict(neural_dim=256, n_classes=40, hidden_dim=1024, layer_dim=5, nDays=24, dropout=0.0, strideLen=4, kernelLen=32,
            gaussianSmoothWidth=2.0)

# Bounds: at most 3x the B200 measurements (1000 W power limit) in profiles/parity_input_grad.json, quoted beside each.
MODEL_BF16_TOL = {"small": 0.014, "bench": 0.055}  # rel L2 of X.grad, bf16 model path (measured 4.9e-3 / 5.8e-3 small, 2.0e-2 bench)
CONFORMER_TOL = {"fp32": 5e-5, "bf16": 0.07}       # rel L2 of X.grad (fp32: the Conformer's parameter-gradient bound; measured 1.6e-6 / 2.4e-2)


def record(key, val):
    path = os.path.join(os.environ.get("NSD_PARITY_OUT") or tempfile.gettempdir(), "parity_input_grad.json")
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


# ----------------------------------------------------------------------------------------------------------- 1. the kernel
# (name, B, T, N, K, S, ntaps, dpatches dtype, days, bound): every variant the dispatch selects -- FFMA with f32 and with bf16
# dpatches, tensor cores at N = 64, 128, 256 -- at an odd shape (T - K not a multiple of S), a stride longer than the window, and the
# benchmark shape.  bound: max |dx - ref| / max |ref| in every region, at most 3x the largest region's measurement (in the comment).
KERNEL_CASES = [
    ("odd_f32", 5, 61, 24, 16, 4, 20, "f32", [2, 0, 2, 1, 0], 6.5e-7),     # 2.2e-7
    ("odd_bf16", 5, 61, 24, 16, 4, 20, "bf16", [2, 0, 2, 1, 0], 6.5e-7),   # 2.2e-7 (FFMA: only dpatches are bf16)
    ("gap_f32", 3, 33, 20, 3, 5, 7, "f32", [1, 0, 1], 4.5e-7),             # 1.6e-7
    ("n64_bf16", 3, 77, 64, 16, 4, 20, "bf16", [1, 1, 0], 1.1e-2),         # 3.7e-3 (tensor cores: dpre and W rounded to bf16)
    ("n128_bf16", 3, 40, 128, 8, 2, 20, "bf16", [0, 2, 1], 8.5e-3),        # 2.9e-3
    ("bench_bf16", 64, 500, 256, 32, 4, 20, "bf16", None, 1.1e-2),         # 3.9e-3
    ("bench_f32", 64, 500, 256, 32, 4, 20, "f32", None, 1.9e-6),           # 6.7e-7
]


@pytest.mark.parametrize("case", KERNEL_CASES, ids=[c[0] for c in KERNEL_CASES])
def test_kernel_vs_oracle(case):
    name, B, T, N, K, S, ntaps, dt, days, bound = case
    rng = np.random.default_rng([B, T, N, K, S, ntaps])
    n_days = 24 if days is None else max(days) + 1
    day = np.asarray(days if days is not None else rng.integers(0, n_days, B), dtype=np.int64)
    Tp = (T - K) // S + 1
    Tz = (Tp - 1) * S + K
    pre = rng.standard_normal((B, T, N)) * 1.5
    z = pre / (1 + np.abs(pre))
    W = rng.standard_normal((n_days, N, N)) / np.sqrt(N) + np.eye(N)
    taps = gaussian_kernel_1d(ntaps, 2.0).numpy().astype(np.float64)
    tdt = torch.float32 if dt == "f32" else torch.bfloat16
    dp = torch.from_numpy(rng.standard_normal((Tp * B, N * K)).astype(np.float32)).to(tdt)
    z32, W32 = z.astype(np.float32), W.astype(np.float32)
    got = ops.frontend_bwd_input(dp.to(DEV), torch.from_numpy(z32).to(DEV), torch.from_numpy(day).to(DEV),
                                 torch.from_numpy(W32).to(DEV), torch.from_numpy(taps.astype(np.float32)).to(DEV), K, S)
    # the oracle sees exactly the operands the kernel got: bf16 dpatches, f32 z (pre recovered from it), f32 W and taps
    dp64 = dp.float().numpy().astype(np.float64).reshape(Tp, B, N * K).transpose(1, 0, 2)
    z64 = z32.astype(np.float64)
    ref = oracle_bwd_input(dp64, {"pre": z64 / (1 - np.abs(z64))}, W32, day, taps.astype(np.float32), T, K, S)
    g = got.cpu().numpy().astype(np.float64)
    scale = np.abs(ref).max()
    regions = {"first10": slice(0, 10), "interior": slice(10, T - 10), "last10": slice(T - 10, T), "past_last_frame": slice(Tz, T)}
    errs = {k: float(np.abs(g[:, sl] - ref[:, sl]).max() / scale) for k, sl in regions.items() if sl.start < sl.stop}
    if Tz < T:
        assert np.abs(ref[:, Tz:]).max() > 0                 # the smoother reaches bins no frame covers
    print(f"{name}: max err / max|ref| by region {errs}")
    record("kernel_" + name, errs)
    for k, e in errs.items():
        assert e < bound, (k, e)
    # deterministic: a second launch gives the same bits
    again = ops.frontend_bwd_input(dp.to(DEV), torch.from_numpy(z32).to(DEV), torch.from_numpy(day).to(DEV),
                                   torch.from_numpy(W32).to(DEV), torch.from_numpy(taps.astype(np.float32)).to(DEV), K, S)
    assert torch.equal(again, got)


def test_kernel_rejects_bad_shapes():
    z = torch.zeros((2, 10, 8), device=DEV)
    dp = torch.zeros((1, 8 * 16), device=DEV)
    with pytest.raises(nsd.NsdError):
        ops.frontend_bwd_input(dp, z, torch.zeros(2, dtype=torch.int64, device=DEV), torch.zeros((1, 8, 8), device=DEV),
                               torch.ones(20, device=DEV), 16, 4)          # T=10 shorter than kernelLen=16
    big = torch.zeros((1, 32, 3000), device=DEV)
    with pytest.raises(nsd.NsdError):
        ops.frontend_bwd_input(torch.zeros((4, 3000 * 8), device=DEV), big, torch.zeros(1, dtype=torch.int64, device=DEV),
                               torch.zeros((1, 3000, 3000), device=DEV), torch.ones(20, device=DEV), 8, 8)   # ring does not fit


# ----------------------------------------------------------------------------------------------------------- 2. GRUDecoder
_PORT = {}


def port_input_grad(kw, B, T, seed):
    """fp64 CPU run of oracle/torch_port.PortGRUDecoder with fill_trained_like_ weights: X.grad of the summed CTC NLL."""
    key = (tuple(sorted(kw.items())), B, T, seed)
    if key in _PORT:
        return _PORT[key]
    from oracle import torch_port as P
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    ours = nsd.GRUDecoder(device="cpu", **kw)
    fill_trained_like_(ours, seed=7)
    sd = {k: v.detach().clone() for k, v in ours.state_dict().items()}
    port = P.PortGRUDecoder(**kw)
    port.load_reference_state(sd)
    port = port.double().eval()
    batch = make_batch(B, T, n_feat=kw["neural_dim"], n_days=kw["nDays"], n_classes=kw["n_classes"], seed=seed, ragged=True,
                       kernel_len=kw["kernelLen"], stride_len=kw["strideLen"], min_tgt=2, max_tgt=20)
    X, y, X_len, y_len, day = batch
    Xd = X.double().requires_grad_(True)
    pred = port(Xd, day)
    lens = ((X_len - port.kernelLen) / port.strideLen).to(torch.int32)
    lp = pred.log_softmax(2).permute(1, 0, 2)
    torch.nn.CTCLoss(blank=0, reduction="sum", zero_infinity=True)(lp, y, lens, y_len).backward()
    _PORT[key] = (sd, batch, Xd.grad.numpy().copy())
    return _PORT[key]


def _model(kw, precision, sd):
    nsd.set_default_precision(precision)
    try:
        torch.manual_seed(0)
        m = nsd.GRUDecoder(device=DEV, **kw)
    finally:
        nsd.set_default_precision("fp32")
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval()


def _x_grad(m, batch, x_grad=True):
    X, y, X_len, y_len, day = (t.to(DEV) for t in batch)
    X = X.clone().requires_grad_(x_grad)
    pred = m.forward(X, day)
    loss = nsd.ctc_loss_from_logits(pred, y, nsd.out_lens(X_len, m.kernelLen, m.strideLen), y_len, reduction="sum")
    loss.backward()
    m.check_errors()
    return X.grad


def _check_against_port(tag, precision, got, ref, bf16_tol):
    g = got.cpu().numpy().astype(np.float64)
    e_l2, e_max = _rel_l2(g, ref), float(np.abs(g - ref).max() / np.abs(ref).max())
    print(f"{tag}: X.grad rel L2 {e_l2:.3e}, max err / max|ref| {e_max:.3e}")
    record(tag, dict(rel_l2=e_l2, max_rel=e_max))
    if precision == "fp32":      # north star, as for the parameter gradients
        np.testing.assert_allclose(g, ref, rtol=1e-3, atol=1e-4 * np.abs(ref).max())
    else:
        assert e_l2 < bf16_tol


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("bidirectional", [False, True])
def test_model_x_grad_small_vs_port(bidirectional, precision):
    kw = dict(SMALL, bidirectional=bidirectional)
    sd, batch, ref = port_input_grad(kw, 6, 90, seed=3)
    m = _model(kw, precision, sd)
    _check_against_port(f"model_small_{'bi' if bidirectional else 'uni'}_{precision}", precision, _x_grad(m, batch), ref,
                        MODEL_BF16_TOL["small"])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_model_x_grad_benchmark_shape_vs_port(precision):
    kw = dict(COMP, bidirectional=True)
    sd, batch, ref = port_input_grad(kw, 64, 500, seed=11)
    m = _model(kw, precision, sd)
    _check_against_port(f"model_bench_bi_{precision}", precision, _x_grad(m, batch), ref, MODEL_BF16_TOL["bench"])


def _small_setup(precision, bidirectional=True):
    kw = dict(SMALL, bidirectional=bidirectional)
    m = _model(kw, precision, _seeded_state(kw))
    batch = make_batch(6, 90, n_feat=32, n_days=4, n_classes=10, seed=5, ragged=True, kernel_len=16, stride_len=4, min_tgt=2, max_tgt=6)
    return m, batch


def _seeded_state(kw):
    torch.manual_seed(0)
    ours = nsd.GRUDecoder(device="cpu", **kw)
    fill_trained_like_(ours, seed=7)
    return ours.state_dict()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_frozen_weights_give_the_same_x_grad(precision):
    """model.requires_grad_(False) + X.requires_grad_(): the forward keeps its backward state, the backward runs (it raised an
    AttributeError before) and X.grad has the bits of the run with trainable parameters."""
    m, batch = _small_setup(precision)
    full = _x_grad(m, batch)
    m.zero_grad(set_to_none=True)
    m.requires_grad_(False)
    frozen = _x_grad(m, batch)
    assert frozen is not None and torch.equal(frozen, full)
    assert all(p.grad is None for p in m.parameters())


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_x_requires_grad_changes_no_parameter_gradient(precision):
    m, batch = _small_setup(precision)
    _x_grad(m, batch, x_grad=False)
    base = {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}
    m.zero_grad(set_to_none=True)
    _x_grad(m, batch, x_grad=True)
    now = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    assert sorted(base) == sorted(now) and len(base) > 0
    for n in base:
        assert torch.equal(base[n], now[n]), n


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_day_bias_only_gets_its_gradient(precision):
    """Only dayBias trainable: the layer-0 dgrad and the front-end backward run for it (they keyed on dayWeights alone before)."""
    m, batch = _small_setup(precision)
    _x_grad(m, batch, x_grad=False)
    want = m.dayBias.grad.clone()
    m.zero_grad(set_to_none=True)
    m.requires_grad_(False)
    m.dayBias.requires_grad_(True)
    _x_grad(m, batch, x_grad=False)
    assert torch.equal(m.dayBias.grad, want)


class _Recorder:
    """Stands in for the loaded library: forwards every entry point and records (name, first argument) in call order."""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def rec(*args):
            self.calls.append((name, args[0] if args else None, args))
            return fn(*args)
        return rec


def _recorded(fn):
    real = _lib.lib()
    rec = _Recorder(real)
    _lib._lib = rec
    try:
        fn()
    finally:
        _lib._lib = real
    torch.cuda.synchronize()
    return rec.calls


def _wgrad_calls(calls):
    """Weight-gradient work: transposed-A GEMMs (dW = dY^T X), the W_hh pair, column sums, BPTT bias sums, the day backward."""
    out = []
    for name, a0, args in calls:
        if name in ("nsd_gemm_f32", "nsd_gemm_bf16") and a0 == 1:
            out.append(name)
        elif name in ("nsd_gemm_bf16_x2", "nsd_colsum", "nsd_frontend_bwd"):
            out.append(name)
        elif name == "nsd_gru_bwd_bf16" and args[-5] is not None:          # db_ih
            out.append(name + "(bias sums)")
    return out


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_frozen_backward_issues_no_parameter_work(precision):
    m, batch = _small_setup(precision)
    m.requires_grad_(False)
    calls = _recorded(lambda: _x_grad(m, batch))
    names = [c[0] for c in calls]
    assert _wgrad_calls(calls) == [], _wgrad_calls(calls)
    assert names.count("nsd_frontend_bwd_input") == 1
    assert names.count("nsd_gru_bwd_bf16" if precision == "bf16" else "nsd_gru_bwd_f32") == SMALL["layer_dim"] * (1 if precision == "bf16" else 2)
    # with trainable parameters the same backward does all of it
    m.requires_grad_(True)
    assert len(_wgrad_calls(_recorded(lambda: _x_grad(m, batch)))) > 0


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_train_step_launches_no_input_gradient(precision):
    kw = dict(SMALL, bidirectional=True, dropout=0.3)
    nsd.set_default_precision(precision)
    try:
        torch.manual_seed(0)
        m = nsd.GRUDecoder(device=DEV, **kw)
    finally:
        nsd.set_default_precision("fp32")
    fill_trained_like_(m, seed=3)
    m = m.to(DEV).train()
    batch = [t.to(DEV) for t in make_batch(6, 90, n_feat=32, n_days=4, n_classes=10, seed=7, ragged=True, kernel_len=16, stride_len=4,
                                           min_tgt=2, max_tgt=6)]
    opt, sched = nsd.make_optimizer(m, dict(lrStart=0.02, lrEnd=0.01, nBatch=10, l2_decay=1e-5))
    nsd.train_step(m, opt, *batch, scheduler=sched, white_noise_sd=0.3)
    names = [c[0] for c in _recorded(lambda: nsd.train_step(m, opt, *batch, scheduler=sched, white_noise_sd=0.3))]
    assert "nsd_frontend_bwd_input" not in names
    assert names.count("nsd_frontend_bwd") == 1


def test_create_graph_raises():
    m, batch = _small_setup("fp32")
    X, y, X_len, y_len, day = (t.to(DEV) for t in batch)
    X = X.clone().requires_grad_(True)
    pred = m.forward(X, day)
    loss = (pred ** 2).sum()                       # a loss whose gradient itself has a graph
    (gx,) = torch.autograd.grad(loss, X, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gx.sum().backward()


# ----------------------------------------------------------------------------------------------------------- 3. Conformer
CONF = dict(n_channels=32, n_classes=11, n_days=3, frontend_dim=64, latent_dim=64, autoencoder_hidden_dim=32, transformer_layers=2,
            transformer_heads=4, transformer_ff_dim=128, transformer_dropout=0.0, temporal_kernel=16, temporal_stride=4,
            gaussian_smooth_width=2.0, conformer_conv_kernel=7, use_spec_augment=False, drop_path_prob=0.0)


def _conformer(precision):
    torch.manual_seed(0)
    m = nsd.NeuralTransformerCTCModel(device="cuda", precision=precision, **CONF)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for p in m.parameters():                                      # off the symmetric initial values
            p.add_(torch.randn(p.shape, generator=g) * (0.02 if p.dim() >= 2 else 0.05) * (p.abs().mean() + 0.1))
    m.output[3].p = 0.0
    B, T = 4, 120
    X = torch.randn(B, T, CONF["n_channels"], generator=g)
    day = torch.tensor([2, 0, 2, 1])
    X_len = torch.tensor([120, 97, 110, 64], dtype=torch.int32)
    y_len = torch.tensor([8, 5, 7, 3], dtype=torch.int32)
    y = torch.zeros(B, 8, dtype=torch.int32)
    for b in range(B):
        y[b, :y_len[b]] = torch.randint(1, CONF["n_classes"], (int(y_len[b]),), generator=g).to(torch.int32)
    return m, (X, y, X_len, y_len, day)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_conformer_x_grad_vs_port(precision):
    from oracle import conformer_port as CP
    m, (X, y, X_len, y_len, day) = _conformer(precision)
    sd = {k: (v.detach().double() if v.is_floating_point() else v.detach()) for k, v in m.state_dict().items()}
    Xd = X.double().requires_grad_(True)
    lp_r, olen_r, _ = CP.forward(sd, Xd, day, X_len, training=False, n_layers=2, n_heads=4, temporal_kernel=16, temporal_stride=4,
                                 conv_kernel=7)
    torch.nn.CTCLoss(blank=0, reduction="sum", zero_infinity=True)(lp_r, y.long(), olen_r.long(), y_len.long()).backward()
    m = m.to(DEV).eval()
    Xg = X.to(DEV).requires_grad_(True)
    lp, olen, _ = m(Xg, day.to(DEV), X_len.to(DEV))
    nsd.CTCLoss(blank=0, reduction="sum", zero_infinity=True)(lp, y.to(DEV), olen, y_len.to(DEV)).backward()
    assert olen.tolist() == olen_r.tolist()
    e = _rel_l2(Xg.grad.cpu().numpy(), Xd.grad.numpy())
    print(f"conformer [{precision}] X.grad rel L2 {e:.3e}")
    record(f"conformer_{precision}", dict(rel_l2=e))
    assert e < CONFORMER_TOL[precision]
    # frozen day parameters: same X.grad, and no day-parameter gradient is made
    m.zero_grad(set_to_none=True)
    m.day_linear.requires_grad_(False)
    Xg2 = X.to(DEV).requires_grad_(True)
    lp, olen, _ = m(Xg2, day.to(DEV), X_len.to(DEV))
    nsd.CTCLoss(blank=0, reduction="sum", zero_infinity=True)(lp, y.to(DEV), olen, y_len.to(DEV)).backward()
    assert torch.equal(Xg2.grad, Xg.grad) and m.day_linear.day_weights.grad is None


# ----------------------------------------------------------------------------------------------------------- 4. input_attribution
def _attr_setup():
    m, batch = _small_setup("fp32")
    return m, [t.to(DEV) for t in batch]


def test_saliency_equals_hand_written_backward():
    m, (X, y, X_len, y_len, day) = _attr_setup()
    att, nll = nsd.input_attribution(m, X, y, X_len, y_len, day, method="saliency")
    Xg = X.clone().requires_grad_(True)
    m.requires_grad_(False)
    lp = m(Xg, day).log_softmax(2).permute(1, 0, 2)
    loss = nsd.CTCLoss(blank=0, reduction="sum", zero_infinity=True)(lp, y, nsd.out_lens(X_len, m.kernelLen, m.strideLen), y_len)
    loss.backward()
    rel = float((att - Xg.grad).norm() / Xg.grad.norm())
    print(f"saliency vs hand-written CTCLoss(sum) backward: rel L2 {rel:.3e}; nll sum {float(nll.sum()):.6f} vs {loss.item():.6f}")
    record("saliency_vs_hand_written", rel)
    assert rel < 2.5e-6                              # the two log-softmax routes differ in fp32 rounding only (measured 9.2e-7)
    assert torch.allclose(nll.sum(), loss.detach(), rtol=1e-5)


def test_integrated_gradients_completeness_and_chunking():
    m, (X, y, X_len, y_len, day) = _attr_setup()
    _, nll_base = nsd.input_attribution(m, torch.zeros_like(X), y, X_len, y_len, day)
    gaps = {}
    for steps in (8, 64):
        ig, nll = nsd.input_attribution(m, X, y, X_len, y_len, day, method="integrated_gradients", steps=steps)
        gaps[steps] = ((ig.sum(dim=(1, 2)) - (nll - nll_base)).abs() / (nll - nll_base).abs()).cpu()
    print(f"integrated gradients completeness gap / |nll(X) - nll(0)| per utterance: 8 steps {gaps[8].tolist()}, 64 steps {gaps[64].tolist()}")
    record("ig_completeness", {str(k): v.tolist() for k, v in gaps.items()})
    assert float(gaps[64].max()) < 1e-3                  # measured 3.6e-4 (8 steps: 4.4e-2)
    assert float(gaps[64].max()) < float(gaps[8].max())
    one, _ = nsd.input_attribution(m, X, y, X_len, y_len, day, method="integrated_gradients", steps=8, max_batch=1000)
    chunked, _ = nsd.input_attribution(m, X, y, X_len, y_len, day, method="integrated_gradients", steps=8, max_batch=5)
    assert torch.allclose(chunked, one, rtol=1e-5, atol=1e-6 * float(one.abs().max()))


def test_attribution_restores_the_model_after_an_error():
    m, (X, y, X_len, y_len, day) = _attr_setup()
    m.train()
    m.gru_decoder.eval()                                                      # a submodule in the other mode than its parent
    m.fc_decoder_out.bias.requires_grad_(False)
    flags = {n: p.requires_grad for n, p in m.named_parameters()}
    modes = {n: mod.training for n, mod in m.named_modules()}
    with pytest.raises(RuntimeError):
        nsd.input_attribution(m, X[:, :, :7], y, X_len, y_len, day)          # wrong channel count: the forward raises
    assert flags == {n: p.requires_grad for n, p in m.named_parameters()}
    assert modes == {n: mod.training for n, mod in m.named_modules()}
    nsd.input_attribution(m, X, y, X_len, y_len, day, method="integrated_gradients", steps=2)
    assert flags == {n: p.requires_grad for n, p in m.named_parameters()}
    assert modes == {n: mod.training for n, mod in m.named_modules()}
    with pytest.raises(ValueError):
        nsd.input_attribution(m, X, y, X_len, y_len, day, method="gradcam")


def test_attribution_of_a_conformer():
    m, (X, y, X_len, y_len, day) = _conformer("fp32")
    m = m.to(DEV)
    batch = [t.to(DEV) for t in (X, y, X_len, y_len, day)]
    sal, nll = nsd.input_attribution(m, *batch)
    ig, nll2 = nsd.input_attribution(m, *batch, method="integrated_gradients", steps=4, max_batch=6)
    assert sal.shape == X.shape and ig.shape == X.shape and torch.isfinite(ig).all() and float(sal.abs().max()) > 0
    assert nll.shape == (X.shape[0],) and torch.allclose(nll, nll2, rtol=1e-6)
