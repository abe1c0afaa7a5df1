"""What the Conformer TRAINING step computes with its regularisers on, against the reference run in fp64 on the host.

Every mask of the Conformer path is counter-based (Philox keyed by (seed, element) or (seed, utterance)) and is regenerated in the
backward instead of being stored; under GraphedConformerStep a device-resident offset is added to every seed.  This file checks:
  A. every mask kernel at p > 0 (LayerNorm(+act)(+dropout), act(+dropout), residual + DropPath, masked softmax + dropout, SpecAugment
     bands + positional encoding) forward and backward against fp64 torch with the mask the kernel itself draws, that this mask
     extraction is valid, and that the device seed offset o with seed s gives exactly what seed s + o gives without it;
  B. (host only) the masked fp64 restatement (tests/conformer_masked_oracle.py) equals oracle/conformer_port with unit masks;
  C. one eager conformer_train_step with dropout, DropPath, SpecAugment, input noise and the head's Dropout(0.3), fp32 and bf16, at a
     small 6-block size and at the competition architecture: log-probs, InterCTC log-probs, loss and every gradient against the
     masked reference fed with the step's own draws, with coverage assertions and four negative controls;
  D. three eager steps with FusedAdamW(max_grad_norm=1) and the warm-up / cosine schedule against torch.optim.AdamW + clip_grad_norm_;
  E. GraphedConformerStep, per replay: gradients, loss and update against the masked reference and AdamW, masks rebuilt under the
     replay's seed offset and SpecAugment bands read back from the device.
The step's draws are taken from the library calls it makes (the loaded library object is wrapped, as in test_gpu_update_schedule.py),
never from a copy of the model's seed arithmetic.  Measured errors go to parity_conformer_training.json in the directory
$NSD_PARITY_OUT names (default: the system's temporary directory); profiles/parity_conformer_training.json holds the B200
measurements the bounds below are set from.
"""
import ctypes
import json
import math
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import conformer_port as CP
import conformer_masked_oracle as MO
import neural_speech_decoder_b200 as nsd

if torch.cuda.is_available():
    from neural_speech_decoder_b200 import _lib, ops
    from neural_speech_decoder_b200._lib import BF16, F32, call, ptr, stream

DEV = "cuda"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
U64 = (1 << 64) - 1
NOISE = (0.8, 0.2)                 # (white_noise_sd, constant_offset_sd)
LS, IW = 0.1, 0.3                  # label smoothing, InterCTC weight
OPT = dict(lr=2e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=1e-2)
SCHED = (2, 10)                    # warm-up steps, total steps of lr_lambda

# fp32 mode: the north star rtol 1e-3 with the absolute floors of test_gpu_training.py (log-probs / gradient entries near zero)
FP32_RTOL = 1e-3
FP32_ATOL = dict(lp=2e-5, grad=1e-5)          # grad: times max(1, max |ref|) of the tensor
# Measured on one B200 (1000 W power limit; profiles/parity_conformer_training.json).  fp32, worst over the small and the
# competition-size step: log-probs 2.9e-6 abs, loss 9.5e-8 rel, gradients 1.7e-5 rel L2 -- the north star's rtol 1e-3 holds with
# a wide margin.  bf16, one train step at the small size (about 3x: log-probs 7.7e-3, InterCTC 8.9e-3, loss 2.2e-5 rel, worst
# gradient 1.6e-2 rel L2 / 1.6e-2 max over max, frontend.temporal_conv.weight):
BF16_TOL = dict(lp_abs=0.025, inter_abs=0.03, loss_rel=1e-4, grad_rel_l2=0.05, grad_max_rel=0.05)
# three-step trajectories (eager and graphed) against torch.optim.AdamW in fp64, about 3x the worst of the eager and graphed runs.
# AdamW's first update is about lr * sign(g) per element (eps 1e-6), so entries whose gradient is near zero move by a full step
# in either direction: the parameter change is the loosest quantity (bf16: 0.25 rel L2, and single entries of opposite sign,
# 2.0 max over max; fp32: 3.2e-3 / 6.5e-3), while the loss (fp32 6.3e-8, bf16 1.6e-4 rel), the gradients of each step (3.3e-6 /
# 4.4e-2 rel L2) and both moments (1.5e-5 / 4.2e-2 rel L2) stay tight.
TRAJ_TOL = {"fp32": dict(loss_rel=2e-7, grad_rel_l2=1e-5, delta_rel_l2=1e-2, delta_max_rel=2e-2, moment_rel_l2=5e-5),
            "bf16": dict(loss_rel=5e-4, grad_rel_l2=0.13, delta_rel_l2=0.75, delta_max_rel=6.0, moment_rel_l2=0.13)}
CONTROL_MARGIN = 5.0               # a negative control must exceed its bound by this factor


def record(key, val):
    """Add a measurement to parity_conformer_training.json in $NSD_PARITY_OUT (default: the system's temporary directory)."""
    path = os.path.join(os.environ.get("NSD_PARITY_OUT") or tempfile.gettempdir(), "parity_conformer_training.json")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    try:
        cur = json.load(open(path))
    except Exception:
        cur = {}
    cur[key] = val
    json.dump(cur, open(path, "w"), indent=1, sort_keys=True)


def f64(t):
    return t.detach().double().cpu()


def keep_factor(p):
    """1/(1-p) as the kernels compute it (fp32)."""
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


# ---------------------------------------------------------------------------------------------------------------------
# the small configuration and its fixture weights
# ---------------------------------------------------------------------------------------------------------------------
SMALL = dict(n_channels=32, n_classes=11, n_days=3, frontend_dim=64, latent_dim=64, autoencoder_hidden_dim=32, transformer_layers=6,
             transformer_heads=4, transformer_ff_dim=128, temporal_kernel=16, temporal_stride=4, gaussian_smooth_width=2.0,
             conformer_conv_kernel=7)
SMALL_PORT = dict(n_layers=6, n_heads=4, temporal_kernel=16, temporal_stride=4, conv_kernel=7)
REGS = dict(transformer_dropout=0.3, drop_path_prob=0.3, use_spec_augment=True, spec_augment_freq_mask=20, spec_augment_time_mask=4)


def small_fixture():
    """conformer_small fixture: state dict (reference names) and its ragged batch (T=84 -> T'=18, out lengths 17 / 9 / 12)."""
    g = np.load(os.path.join(GOLD, "conformer_small.npz"))
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd/")}
    batch = tuple(torch.from_numpy(g[k]) for k in ("X", "y", "X_len", "y_len", "day"))
    return sd, batch


def build_small(precision, **over):
    sd, _ = small_fixture()
    m = nsd.NeuralTransformerCTCModel(device="cuda", precision=precision, **dict(SMALL, **REGS, **over))
    own = m.state_dict()
    sd = dict(sd, **{"pos_enc.pe": own["pos_enc.pe"]})            # the fixture keeps the first 256 rows of the buffer
    m.load_state_dict(sd, strict=True)
    return m.to(DEV)


# ---------------------------------------------------------------------------------------------------------------------
# recording the step's library calls and rebuilding its masks
# ---------------------------------------------------------------------------------------------------------------------
MASK_CALLS = ("nsd_layernorm_fwd", "nsd_act_fwd", "nsd_residual", "nsd_softmax_mask_fwd", "nsd_posenc_mask", "nsd_input_noise")


class _Recorder:
    """Stands in for the loaded library: forwards every entry point and records (name, args) of the mask-drawing ones."""

    def __init__(self, lib):
        self._lib = lib
        self.calls = []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name not in MASK_CALLS:
            return fn

        def rec(*args):
            a = list(args)
            if name == "nsd_posenc_mask":
                a[2] = list(a[2])                                   # the host bands (a ctypes array)
            self.calls.append((name, a))
            return fn(*args)
        return rec


class recording:
    def __enter__(self):
        self.rec = _Recorder(_lib.lib())
        _lib._lib = self.rec
        return self.rec

    def __exit__(self, *exc):
        _lib._lib = self.rec._lib
        return False


def sites_of(calls):
    """The mask sites of one step, in call order: noise, front-end LN, SpecAugment, per block (act, residual, softmax, residual,
    residual, act, residual), head LN.  Calls that draw nothing (p = 0, backward forms) are skipped."""
    out = []
    for name, a in calls:
        if name == "nsd_input_noise":
            out.append(dict(kind="noise", B=a[2], T=a[3], N=a[4], white=a[5], offset=a[6], seed=a[7]))
        elif name == "nsd_layernorm_fwd" and a[5] > 0:
            out.append(dict(kind="ln", act=a[4], p=a[5], seed=a[6], M=a[11], D=a[12]))
        elif name == "nsd_posenc_mask" and a[1] is not None:
            out.append(dict(kind="posenc", bands=a[2], bands_dev=a[3], B=a[5], T=a[6], D=a[7]))
        elif name == "nsd_act_fwd" and a[2] > 0:
            out.append(dict(kind="act", act=a[1], p=a[2], seed=a[3], n=a[6]))
        elif name == "nsd_residual" and a[0] is not None:
            out.append(dict(kind="res", scale=a[2], p=a[3], seed=a[4], p_path=a[5], path_seed=a[6], per=a[7], n=a[9]))
        elif name == "nsd_softmax_mask_fwd" and a[8] > 0:
            out.append(dict(kind="sm", B=a[4], H=a[5], T=a[6], ld=a[7], p=a[8], seed=a[9]))
    return out


def expected_kinds(n_layers, noise=True):
    return (["noise"] if noise else []) + ["ln", "posenc"] + ["act", "res", "sm", "res", "res", "act", "res"] * n_layers + ["ln"]


def seeds_of(sites):
    """Every mask seed of the step, in order (DropPath seeds only where DropPath is on)."""
    s = []
    for st in sites:
        if st["kind"] in ("ln", "act", "sm"):
            s.append(st["seed"])
        elif st["kind"] == "res":
            s.append(st["seed"])
            if st["p_path"] > 0:
                s.append(st["path_seed"])
    return s


def ln_mask(M, D, p, seed, act=0, out16=False):
    x = torch.zeros(M, D, device=DEV)
    gamma, beta = torch.zeros(D, device=DEV), torch.ones(D, device=DEV)
    y32 = None if out16 else torch.empty(M, D, device=DEV)
    y16 = torch.empty(M, D, device=DEV, dtype=torch.bfloat16) if out16 else None
    mean, rstd = torch.empty(M, device=DEV), torch.empty(M, device=DEV)
    call("nsd_layernorm_fwd", ptr(x), ptr(gamma), ptr(beta), 1e-5, act, float(p), int(seed), ptr(y32), ptr(y16), ptr(mean), ptr(rstd), M, D, stream())
    return y16.float() if out16 else y32


def act_mask(n, p, seed, act=0, out16=False):
    x = torch.ones(n, device=DEV)
    y = torch.empty(n, device=DEV, dtype=torch.bfloat16 if out16 else torch.float32)
    call("nsd_act_fwd", ptr(x), act, float(p), int(seed), None if out16 else ptr(y), ptr(y) if out16 else None, n, stream())
    return y.float()


def res_mask(n, per, p, seed, p_path, path_seed):
    y, out = torch.ones(n, device=DEV), torch.empty(n, device=DEV)
    call("nsd_residual", None, ptr(y), 1.0, float(p), int(seed), float(p_path), int(path_seed), int(per), ptr(out), n, stream())
    return out


def sm_mask(B, H, T, ld, lens, p, seed, out16=False):
    """[B,H,T,T] multiplier of the attention-weight dropout: (Pd != 0) / (1-p) on the valid keys of S = 0."""
    S = torch.zeros(B * H * T, ld, device=DEV)
    Pd = torch.empty(B * H * T, ld, device=DEV, dtype=torch.bfloat16 if out16 else torch.float32)
    call("nsd_softmax_mask_fwd", ptr(S), ptr(Pd), BF16 if out16 else F32, ptr(lens), B, H, T, ld, float(p), int(seed), stream())
    return (Pd.view(B, H, T, ld)[..., :T] != 0).double().cpu() * keep_factor(p)


def rebuild(sites, X, lens, bands=None, seed_shift=False, path=True, with_bands=True, noise=True):
    """The step's masks in the layout of conformer_masked_oracle (fp64, host), its noised input and per-site keep counts
    (p, kept, drawn), rebuilt with the kernels from the recorded (p, seed, shape).  ``sites`` follow expected_kinds().
    ``bands``: the SpecAugment bounds when the step read them from the device array.  The negative controls: ``seed_shift``
    builds each site's mask from the next site's seed, ``path`` / ``with_bands`` / ``noise`` False leave DropPath, the bands
    or the noise out."""
    seeds = seeds_of(sites)
    nxt = dict(zip(seeds, seeds[1:] + seeds[:1])) if seed_shift else {s: s for s in seeds}
    stats = []
    Xn = X.to(DEV).float().contiguous()
    if sites[0]["kind"] == "noise":
        st = sites[0]
        if noise:
            Xn = ops.input_noise(Xn, st["white"], st["offset"], st["seed"])
        sites = sites[1:]
    pe = sites[1]
    B, Tn = pe["B"], pe["T"]
    lens_h = lens.cpu().long()

    def ln(st):
        mk = ln_mask(st["M"], st["D"], st["p"], nxt[st["seed"]])
        stats.append((st["p"], int((mk != 0).sum()), mk.numel()))
        return f64(mk).view(B, Tn, -1)

    def act(st):
        mk = act_mask(st["n"], st["p"], nxt[st["seed"]])
        stats.append((st["p"], int((mk != 0).sum()), mk.numel()))
        return f64(mk).view(B, Tn, -1)

    def res(st, blk, name):
        dm = res_mask(st["n"], st["per"], st["p"], nxt[st["seed"]], 0.0, 0)
        stats.append((st["p"], int((dm != 0).sum()), dm.numel()))
        blk[name + "_drop"] = f64(dm).view(B, Tn, -1)
        if st["p_path"] > 0:
            pm = f64(res_mask(st["n"], st["per"], 0.0, 0, st["p_path"], nxt[st["path_seed"]])).view(B, -1)
            pf = pm[:, 0]                                          # DropPath: one factor per utterance, read at its first element
            stats.append((st["p_path"], int((pf != 0).sum()), B))
            blk[name + "_path"] = pf if path else None

    def sm(st):
        mk = sm_mask(st["B"], st["H"], st["T"], st["ld"], lens, st["p"], nxt[st["seed"]])
        valid = (torch.arange(Tn)[None, :] < lens_h[:, None])[:, None, None, :].expand_as(mk)
        stats.append((st["p"], int((mk[valid] != 0).sum()), int(valid.sum())))
        return mk

    masks = dict(fe=ln(sites[0]), bands=(list(bands if bands is not None else pe["bands"]) if with_bands else None), blocks=[])
    body = sites[2:-1]
    for i in range(0, len(body), 7):
        s = body[i:i + 7]
        blk = dict(ff1_act=act(s[0]))
        res(s[1], blk, "ff1")
        blk["attn_p"] = sm(s[2])
        res(s[3], blk, "attn")
        res(s[4], blk, "conv")
        blk["ff2_act"] = act(s[5])
        res(s[6], blk, "ff2")
        masks["blocks"].append(blk)
    masks["head"] = ln(sites[-1])
    return masks, f64(Xn), stats


# ---------------------------------------------------------------------------------------------------------------------
# A. the mask kernels at p > 0 against fp64, with the mask each kernel draws
# ---------------------------------------------------------------------------------------------------------------------
def _close(got, ref, tol, what=""):
    got, ref = f64(got), f64(ref)
    err = (got - ref).abs().max().item() / max(1.0, ref.abs().max().item())
    assert err < tol, f"{what}: max err / max|ref| = {err:.3e} >= {tol}"


def _act64(v, act):
    return [v, torch.nn.functional.silu(v), torch.nn.functional.gelu(v), torch.relu(v)][act]


# (M, D, act, dy dtype, skip addend): D in each instantiation (<= 512, <= 1024, <= 2048), M not a multiple of 8 and M > 256
# (several chunks of layernorm_bwd_param_kernel), each activation with f32 and bf16 dy
LN_CASES = [(300, 136, 0, "f32", True), (261, 1000, 1, "bf16", False), (517, 2048, 2, "f32", False), (45, 64, 1, "f32", True),
            (777, 520, 0, "bf16", True), (259, 1024, 2, "bf16", True)]


@pytest.mark.gpu
@pytest.mark.parametrize("M,D,act,dy_dt,skip", LN_CASES)
def test_layernorm_dropout_fwd_bwd(M, D, act, dy_dt, skip):
    p, seed = 0.3, 0x1234567 + M
    g = torch.Generator().manual_seed(M * D)
    x = torch.randn(M, D, generator=g, dtype=torch.float64) * 2 + 0.5
    gamma, beta = torch.randn(D, generator=g, dtype=torch.float64), torch.randn(D, generator=g, dtype=torch.float64)
    dy = torch.randn(M, D, generator=g, dtype=torch.float64)
    if dy_dt == "bf16":
        dy = dy.to(torch.bfloat16).double()                          # the values the kernel receives
    add = torch.randn(M, D, generator=g, dtype=torch.float64) if skip else None
    k = f64(ln_mask(M, D, p, seed))
    xr, gr, br = (t.clone().requires_grad_(True) for t in (x, gamma, beta))
    y = _act64(torch.nn.functional.layer_norm(xr, (D,), gr, br, 1e-5), act) * k
    y.backward(dy)
    xc, gc, bc = (t.float().to(DEV) for t in (x, gamma, beta))
    y32, y16 = torch.empty(M, D, device=DEV), torch.empty(M, D, device=DEV, dtype=torch.bfloat16)
    mean, rstd = torch.empty(M, device=DEV), torch.empty(M, device=DEV)
    call("nsd_layernorm_fwd", ptr(xc), ptr(gc), ptr(bc), 1e-5, act, p, seed, ptr(y32), ptr(y16), ptr(mean), ptr(rstd), M, D, stream())
    _close(y32, y, 3e-6, "y f32"); _close(y16, y, 8e-3, "y bf16")
    assert torch.equal(y32 != 0, y16 != 0) or act != 0               # the same mask in both copies
    dyc = dy.to(DEV).to(torch.bfloat16 if dy_dt == "bf16" else torch.float32)
    addc = add.float().to(DEV) if skip else None
    dx, dg, db = torch.empty(M, D, device=DEV), torch.empty(D, device=DEV), torch.empty(D, device=DEV)
    ws = torch.empty(_lib.lib().nsd_layernorm_bwd_workspace(M, D), device=DEV, dtype=torch.uint8)
    call("nsd_layernorm_bwd", ptr(dyc), BF16 if dy_dt == "bf16" else F32, ptr(xc), ptr(gc), ptr(bc), ptr(mean), ptr(rstd), act, p, seed, ptr(addc),
         ptr(dx), ptr(dg), ptr(db), M, D, ptr(ws), ws.numel(), stream())
    _close(dx, xr.grad + (add if skip else 0), 3e-5, "dx"); _close(dg, gr.grad, 3e-5, "dgamma"); _close(db, br.grad, 3e-5, "dbeta")


@pytest.mark.gpu
@pytest.mark.parametrize("act", [0, 1, 2, 3])
@pytest.mark.parametrize("out_dt", ["f32", "bf16"])
def test_activation_dropout_fwd_bwd(act, out_dt):
    p, seed, M, N = 0.3, 991 + act, 37, 100
    g = torch.Generator().manual_seed(act)
    x = torch.randn(M, N, generator=g, dtype=torch.float64) * 3
    dy = torch.randn(M, N, generator=g, dtype=torch.float64).to(torch.bfloat16).double()   # bf16 dy (as the bf16 GEMM's dgrad gives)
    k = f64(act_mask(M * N, p, seed)).view(M, N)
    xr = x.clone().requires_grad_(True)
    y = _act64(xr, act) * k
    y.backward(dy)
    xc = x.float().to(DEV)
    y_dev = torch.empty(M, N, device=DEV, dtype=torch.bfloat16 if out_dt == "bf16" else torch.float32)
    call("nsd_act_fwd", ptr(xc), act, p, seed, ptr(y_dev) if out_dt == "f32" else None, ptr(y_dev) if out_dt == "bf16" else None, M * N, stream())
    _close(y_dev, y, 3e-6 if out_dt == "f32" else 8e-3, "act")
    for dy_dt in ("f32", "bf16"):
        dyc = dy.to(DEV).to(torch.bfloat16 if dy_dt == "bf16" else torch.float32)
        dx = torch.empty(M, N, device=DEV)
        call("nsd_act_bwd", ptr(dyc), BF16 if dy_dt == "bf16" else F32, ptr(xc), act, p, seed, ptr(dx), M * N, stream())
        _close(dx, xr.grad, 3e-6, f"act grad (dy {dy_dt})")


@pytest.mark.gpu
def test_residual_dropout_droppath_fwd_bwd():
    B, T, D, scale, p, pp, seed, pseed = 16, 13, 24, 0.5, 0.3, 0.4, 4242, 777
    per, n = T * D, B * T * D
    g = torch.Generator().manual_seed(1)
    x, y, dout = (torch.randn(n, generator=g, dtype=torch.float64) for _ in range(3))
    k = f64(res_mask(n, per, p, seed, 0.0, 0))
    pm = f64(res_mask(n, per, 0.0, 0, pp, pseed)).view(B, per)
    assert torch.equal(pm, pm[:, :1].expand_as(pm))                   # whole utterances are kept or dropped
    pf = pm[:, 0]
    assert set(pf.tolist()) == {0.0, keep_factor(pp)}
    f = (scale * pf)[:, None].expand(B, per).reshape(-1) * k
    out, xd, yd, dd = torch.empty(n, device=DEV), x.float().to(DEV), y.float().to(DEV), dout.float().to(DEV)
    call("nsd_residual", ptr(xd), ptr(yd), scale, p, seed, pp, pseed, per, ptr(out), n, stream())
    _close(out, x + f * y, 3e-6, "residual")
    dy = torch.empty(n, device=DEV)
    call("nsd_residual", None, ptr(dd), scale, p, seed, pp, pseed, per, ptr(dy), n, stream())
    _close(dy, f * dout, 3e-6, "residual backward")


@pytest.mark.gpu
@pytest.mark.parametrize("pd_dt", ["f32", "bf16"])
def test_softmax_mask_dropout_fwd_bwd(pd_dt):
    B, H, T, p, seed = 4, 3, 37, 0.3, 31337
    ld = (T + 7) // 8 * 8
    g = torch.Generator().manual_seed(5)
    S0 = torch.randn(B * H * T, ld, generator=g, dtype=torch.float64) * 2
    lens = torch.tensor([T, 1, 20, 36], dtype=torch.int32)
    dPd = torch.randn(B * H * T, ld, generator=g, dtype=torch.float64)
    mk = sm_mask(B, H, T, ld, lens.to(DEV), p, seed)                  # [B,H,T,T]
    Sr = S0.view(B, H, T, ld)[..., :T].clone().requires_grad_(True)
    pad = (torch.arange(T)[None, :] >= lens[:, None].long())[:, None, None, :]
    P = torch.softmax(Sr.masked_fill(pad, float("-inf")), -1)
    Pd_ref = P * mk
    Pd_ref.backward(dPd.view(B, H, T, ld)[..., :T])
    S = S0.float().to(DEV)
    Pd = torch.empty(B * H * T, ld, device=DEV, dtype=torch.bfloat16 if pd_dt == "bf16" else torch.float32)
    call("nsd_softmax_mask_fwd", ptr(S), ptr(Pd), BF16 if pd_dt == "bf16" else F32, ptr(lens.to(DEV)), B, H, T, ld, p, seed, stream())
    _close(S.view(B, H, T, ld)[..., :T], P, 2e-6, "P")
    _close(Pd.view(B, H, T, ld)[..., :T], Pd_ref, 2e-6 if pd_dt == "f32" else 8e-3, "Pd")
    assert not S.view(B, H, T, ld)[..., T:].any() and not Pd.view(B, H, T, ld)[..., T:].float().any()     # ld padding written as 0
    d = dPd.float().to(DEV)
    d.view(B, H, T, ld)[..., T:] = float("nan")                      # the padding columns of dPd are never read
    call("nsd_softmax_mask_bwd", ptr(S), ptr(d), B, H, T, ld, p, seed, stream())
    _close(d.view(B, H, T, ld)[..., :T], Sr.grad, 3e-6, "dS")
    assert torch.isfinite(d).all()
    assert (Sr.grad[1, :, :, 1:] == 0).all() and (f64(d).view(B, H, T, ld)[1, :, :, :T] == 0).all()   # length 1: one key, P = 1, dS = 0


# (host bands, id): empty, overlapping, at 0 and at D / T', covering everything, time bands only
POSENC_BANDS = [([0] * 8, "empty"), ([2, 9, 5, 14, 1, 4, 3, 7], "overlapping"), ([0, 3, 20, 24, 0, 2, 11, 13], "edges"),
                ([0, 24, 0, 0, 0, 13, 0, 0], "everything"), ([4, 4, 0, 0, 12, 13, 6, 9], "time")]


@pytest.mark.gpu
@pytest.mark.parametrize("bands,case", POSENC_BANDS, ids=[c for _, c in POSENC_BANDS])
def test_posenc_specaugment_bands(bands, case):
    B, T, D = 3, 13, 24
    g = torch.Generator().manual_seed(2)
    z, pe, dout = torch.randn(B * T, D, generator=g), torch.randn(T, D, generator=g), torch.randn(B * T, D, generator=g)
    keep = MO.band_keep(bands, T, D).repeat(B, 1)
    bd = torch.tensor(bands, dtype=torch.int32, device=DEV)
    zd, ped, dd = z.to(DEV), pe.to(DEV), dout.to(DEV)
    outs = []
    for host in (True, False):
        arr = (ctypes.c_int * 8)(*(bands if host else [0] * 8))
        o, dz = torch.empty(B * T, D, device=DEV), torch.empty(B * T, D, device=DEV)
        call("nsd_posenc_mask", ptr(zd), ptr(ped), arr, None if host else ptr(bd), ptr(o), B, T, D, stream())
        call("nsd_posenc_mask", ptr(dd), None, arr, None if host else ptr(bd), ptr(dz), B, T, D, stream())
        outs.append((o, dz))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])     # host and device bounds: bit-identical
    keep = keep.float()                                                # the same fp32 arithmetic, so the comparison is exact
    assert torch.equal(outs[0][0].cpu(), z * keep + pe.repeat(B, 1))
    assert torch.equal(outs[0][1].cpu(), dout * keep)
    if case == "everything":
        assert not outs[0][1].any()


@pytest.mark.gpu
def test_mask_extraction_does_not_depend_on_activation_or_dtype():
    """The tests rebuild a step's masks from kernels called with ACT_NONE and f32 outputs: the mask a kernel draws must not depend
    on the activation code or the output dtype of the call that drew it."""
    M, D, p, seed = 67, 96, 0.3, 5150
    ref = ln_mask(M, D, p, seed) != 0
    for act in (0, 1, 2):
        for out16 in (False, True):
            assert torch.equal(ln_mask(M, D, p, seed, act=act, out16=out16) != 0, ref), (act, out16)
    ref = act_mask(M * D, p, seed) != 0
    for act in (0, 1, 2):                                              # (ReLU(1) = 1 as well; ReLU zeroes negatives, not used here)
        for out16 in (False, True):
            assert torch.equal(act_mask(M * D, p, seed, act=act, out16=out16) != 0, ref), (act, out16)
    lens = torch.tensor([30, 7], dtype=torch.int32, device=DEV)
    assert torch.equal(sm_mask(2, 3, 30, 32, lens, p, seed), sm_mask(2, 3, 30, 32, lens, p, seed, out16=True))


class seed_offset:
    """nsd_set_seed_offset_ptr to a device u64 holding ``o`` for the duration (cleared in any case: process-global state)."""

    def __init__(self, o):
        self.t = torch.tensor([o - (1 << 64) if o >= 1 << 63 else o], dtype=torch.int64, device=DEV)

    def __enter__(self):
        call("nsd_set_seed_offset_ptr", ptr(self.t))
        return self

    def __exit__(self, *exc):
        call("nsd_set_seed_offset_ptr", None)
        return False


def _offset_kernels(seed):
    """Every kernel that reads the seed offset, at fixed inputs, with dropout / DropPath / noise seeded by ``seed``."""
    g = torch.Generator().manual_seed(9)
    M, D, p = 300, 256, 0.3
    x, dy = torch.randn(M, D, generator=g).to(DEV), torch.randn(M, D, generator=g).to(DEV)
    gamma, beta = torch.randn(D, generator=g).to(DEV), torch.randn(D, generator=g).to(DEV)
    out = {}
    y, mean, rstd = torch.empty(M, D, device=DEV), torch.empty(M, device=DEV), torch.empty(M, device=DEV)
    call("nsd_layernorm_fwd", ptr(x), ptr(gamma), ptr(beta), 1e-5, 1, p, seed, ptr(y), None, ptr(mean), ptr(rstd), M, D, stream())
    dx, dg, db = torch.empty(M, D, device=DEV), torch.empty(D, device=DEV), torch.empty(D, device=DEV)
    ws = torch.empty(_lib.lib().nsd_layernorm_bwd_workspace(M, D), device=DEV, dtype=torch.uint8)
    call("nsd_layernorm_bwd", ptr(dy), F32, ptr(x), ptr(gamma), ptr(beta), ptr(mean), ptr(rstd), 1, p, seed, None, ptr(dx), ptr(dg), ptr(db), M, D,
         ptr(ws), ws.numel(), stream())
    out.update(ln_fwd=y, ln_dx=dx, ln_dgamma=dg, ln_dbeta=db)
    ya, dxa = torch.empty(M, D, device=DEV), torch.empty(M, D, device=DEV)
    call("nsd_act_fwd", ptr(x), 1, p, seed, ptr(ya), None, M * D, stream())
    call("nsd_act_bwd", ptr(dy), F32, ptr(x), 1, p, seed, ptr(dxa), M * D, stream())
    out.update(act_fwd=ya, act_bwd=dxa)
    r = torch.empty(M, D, device=DEV)
    call("nsd_residual", ptr(x), ptr(dy), 0.5, p, seed, 0.4, (seed + 0x5A5A) & U64, 10 * D, ptr(r), M * D, stream())   # both seeds shift by o
    out["residual"] = r
    B, H, T, ld = 2, 3, 50, 56
    S, Pd = torch.randn(B * H * T, ld, generator=g).to(DEV), torch.empty(B * H * T, ld, device=DEV)
    lens = torch.tensor([50, 33], dtype=torch.int32, device=DEV)
    call("nsd_softmax_mask_fwd", ptr(S), ptr(Pd), F32, ptr(lens), B, H, T, ld, p, seed, stream())
    dS = torch.randn(B * H * T, ld, generator=g).to(DEV)
    call("nsd_softmax_mask_bwd", ptr(S), ptr(dS), B, H, T, ld, p, seed, stream())
    out.update(softmax_fwd=Pd, softmax_bwd=dS)
    X = torch.randn(3, 40, 32, generator=g).to(DEV)
    out["input_noise"] = ops.input_noise(X, *NOISE, seed)
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("s,o", [(0x7FFFFFFFFFFFFF00, 0xC000000000000123), (12345, 1)], ids=["wraps", "plus_one"])
def test_seed_offset_is_a_seed_shift(s, o):
    """With the device offset o, seed s draws exactly what seed s + o (mod 2^64) draws without it; after the pointer is cleared,
    seed s draws its own masks again."""
    plain = _offset_kernels(s)
    shifted = _offset_kernels((s + o) & U64)
    with seed_offset(o):
        got = _offset_kernels(s)
    after = _offset_kernels(s)
    for k in plain:
        assert torch.equal(got[k], shifted[k]), k
        assert torch.equal(after[k], plain[k]), k
        assert not torch.equal(got[k], plain[k]), k                    # the offset does change the draw


# ---------------------------------------------------------------------------------------------------------------------
# B. the masked fp64 restatement equals the port with unit masks (host only)
# ---------------------------------------------------------------------------------------------------------------------
def reference_run(sd, batch, masks, cfg, dtype=torch.float64, Xn=None):
    """Log-probs, InterCTC log-probs, loss and every parameter gradient of the masked restatement (``Xn``: the noised input)."""
    X, y, X_len, y_len, day = batch
    if dtype != torch.float64:
        cast = lambda v: v.to(dtype) if torch.is_tensor(v) else v
        masks = dict({k: cast(v) for k, v in masks.items() if k != "blocks"}, blocks=[{k: cast(v) for k, v in b.items()} for b in masks["blocks"]])
    names = [k for k in sd if k not in ("pos_enc.pe", "frontend.gaussian_kernel")]
    params = {k: sd[k].to(dtype).clone().requires_grad_(True) for k in names}
    full = {**{k: v.to(dtype) for k, v in sd.items()}, **params}
    lp, olen, inter = MO.forward(full, (X if Xn is None else Xn).to(dtype), day, X_len, masks=masks, **cfg)
    loss = CP.training_loss(lp, inter, y, olen, y_len, label_smoothing=LS, interctc_weight=IW)
    loss.backward()
    return dict(lp=lp.detach(), inter=inter.detach(), loss=loss.item(), grads={k: p.grad.detach() for k, p in params.items()})


def test_masked_port_with_unit_masks_is_the_port():
    """Host only.  All-ones masks and empty bands: the masked restatement equals conformer_port.forward + training_loss in fp64
    (log-probs, InterCTC log-probs, loss, every gradient) to 1e-12, so a difference the GPU tests see comes from the masks fed
    to it.  And each kind of mask does act."""
    sd, batch = small_fixture()
    sd = {k: v.double() for k, v in sd.items()}
    X, y, X_len, y_len, day = batch
    B, Tn, D, FF, H = X.shape[0], 18, 64, 128, 4
    one = lambda *s: torch.ones(*s, dtype=torch.float64)
    blk = dict(ff1_act=one(B, Tn, FF), ff1_drop=one(B, Tn, D), ff1_path=one(B), attn_p=one(B, H, Tn, Tn), attn_drop=one(B, Tn, D),
               attn_path=one(B), conv_drop=one(B, Tn, D), ff2_act=one(B, Tn, FF), ff2_drop=one(B, Tn, D), ff2_path=one(B))
    units = dict(fe=one(B, Tn, 64), bands=[0] * 8, head=one(B, Tn, D), blocks=[dict(blk) for _ in range(6)])
    got = reference_run(sd, batch, units, SMALL_PORT)
    names = [k for k in sd if k not in ("pos_enc.pe", "frontend.gaussian_kernel")]
    params = {k: sd[k].clone().requires_grad_(True) for k in names}
    lp, olen, inter = CP.forward({**sd, **params}, X.double(), day, X_len, training=True, **SMALL_PORT)
    loss = CP.training_loss(lp, inter, y, olen, y_len, label_smoothing=LS, interctc_weight=IW)
    loss.backward()
    assert abs(got["loss"] - loss.item()) <= 1e-12 * abs(loss.item())
    torch.testing.assert_close(got["lp"], lp.detach(), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(got["inter"], inter.detach(), rtol=1e-12, atol=1e-12)
    for k, p in params.items():
        torch.testing.assert_close(got["grads"][k], p.grad, rtol=1e-12, atol=1e-12, msg=k)
    # each site kind moves the loss: a dropped element, a dropped utterance, a band, an attention weight
    for edit in ("fe", "ff1_path", "bands", "attn_p", "conv_drop", "head", "ff2_act"):
        m = dict(units, blocks=[dict(b) for b in units["blocks"]])
        if edit in ("fe", "head"):
            m[edit] = m[edit].clone(); m[edit][:, :, ::3] = 0
        elif edit == "bands":
            m["bands"] = [3, 9, 0, 0, 2, 5, 0, 0]
        else:
            t = m["blocks"][2][edit].clone()
            t.view(-1)[::3] = 0
            m["blocks"][2][edit] = t
        assert abs(reference_run(sd, batch, m, SMALL_PORT)["loss"] - got["loss"]) > 1e-6, edit


# ---------------------------------------------------------------------------------------------------------------------
# C. one eager training step against the masked reference fed with the step's own draws
# ---------------------------------------------------------------------------------------------------------------------
def rel_l2(a, b):
    return float((a - b).norm() / max(float(b.norm()), 1e-30))


def max_rel(a, b):
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def compare(got, ref, precision, tol=None):
    """Errors of one step and its score: the largest error over its bound (< 1: within the precision's tolerance).  fp32: the
    element-wise allclose(rtol 1e-3, atol floor) criterion; bf16: each error over its entry of ``tol``."""
    err = dict(lp_abs=float((got["lp"] - ref["lp"]).abs().max()), inter_abs=float((got["inter"] - ref["inter"]).abs().max()),
               loss=got["loss"], loss_ref=ref["loss"], loss_rel=abs(got["loss"] - ref["loss"]) / abs(ref["loss"]),
               grad_rel_l2={k: rel_l2(got["grads"][k], g) for k, g in ref["grads"].items()},
               grad_max_rel={k: max_rel(got["grads"][k], g) for k, g in ref["grads"].items()})
    if precision == "fp32":
        ratio = lambda a, b, atol: float(((a - b).abs() / (atol + FP32_RTOL * b.abs())).max())
        parts = dict(lp=ratio(got["lp"], ref["lp"], FP32_ATOL["lp"]), inter=ratio(got["inter"], ref["inter"], FP32_ATOL["lp"]),
                     loss=err["loss_rel"] / FP32_RTOL)
        for k, g in ref["grads"].items():
            parts[k] = ratio(got["grads"][k], g, FP32_ATOL["grad"] * max(1.0, float(g.abs().max())))
    else:
        tol = tol or BF16_TOL
        parts = dict(lp=err["lp_abs"] / tol["lp_abs"], inter=err["inter_abs"] / tol["inter_abs"], loss=err["loss_rel"] / tol["loss_rel"])
        for k in ref["grads"]:
            parts[k] = max(err["grad_rel_l2"][k] / tol["grad_rel_l2"], err["grad_max_rel"][k] / tol["grad_max_rel"])
    worst = max(parts.items(), key=lambda kv: kv[1])
    err["score"], err["worst"] = worst[1], worst[0]
    return err


def our_step(m, opt, batch, noise_seed):
    """One eager conformer_train_step with input noise; -> (log-probs, InterCTC log-probs, loss, gradients) and its mask calls."""
    out = {}
    hook = m.register_forward_hook(lambda mod, inp, o: out.update(lp=o[0], inter=o[2]))
    try:
        with recording() as rec:
            loss = nsd.conformer_train_step(m, opt, *(t.to(DEV) for t in batch), LS, IW, *NOISE, noise_seed=noise_seed)
    finally:
        hook.remove()
    torch.cuda.synchronize()
    got = dict(lp=f64(out["lp"]), inter=f64(out["inter"]), loss=loss.item(), grads={n: f64(p.grad) for n, p in m.named_parameters()})
    return got, rec.calls


def check_sites(sites, n_layers, p, p_path, p_head=0.3):
    """The recorded sites are the model's, in forward order, with its probabilities; every mask seed of the step is distinct."""
    assert [s["kind"] for s in sites] == expected_kinds(n_layers), [s["kind"] for s in sites]
    body = sites[3:-1]
    assert sites[1]["p"] == pytest.approx(p) and sites[1]["act"] == 0
    assert sites[-1]["p"] == pytest.approx(p_head) and sites[-1]["act"] == 2                 # head: LayerNorm + GELU + Dropout(0.3)
    for i in range(0, len(body), 7):
        b = body[i:i + 7]
        assert b[0]["act"] == 1 and b[5]["act"] == 1                                          # SiLU + dropout in ff1 / ff2
        assert [r["scale"] for r in (b[1], b[3], b[4], b[6])] == [0.5, 1.0, 1.0, 0.5]
        assert [r["p_path"] for r in (b[1], b[3], b[4], b[6])] == pytest.approx([p_path, p_path, 0.0, p_path])
        assert all(s["p"] == pytest.approx(p) for s in b)
    seeds = seeds_of(sites)
    assert len(set(seeds)) == len(seeds)


def check_coverage(masks, stats, lens, Tn):
    """The draws exercise what the negative controls test: a dropped and a kept utterance under DropPath, non-empty SpecAugment
    bands, padded keys; and every site keeps a fraction within five binomial standard deviations of 1-p."""
    paths = torch.cat([b[k] for b in masks["blocks"] for k in ("ff1_path", "attn_path", "ff2_path") if b.get(k) is not None])
    assert (paths == 0).any() and (paths != 0).any(), paths
    bd = masks["bands"]
    assert any(bd[i + 1] > bd[i] for i in (0, 2)) and any(bd[i + 1] > bd[i] for i in (4, 6)), bd
    assert int(lens.min()) < Tn
    for p, kept, n in stats:
        assert abs(kept / n - (1 - p)) <= 5 * math.sqrt(p * (1 - p) / n) + 1e-12, (p, kept, n)


CONTROLS = [("next_site_seed", dict(seed_shift=True)), ("no_droppath", dict(path=False)), ("no_bands", dict(with_bands=False)),
            ("no_noise", dict(noise=False))]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_train_step_small_matches_masked_reference(precision):
    """6 blocks (InterCTC on), dropout 0.3, DropPath 0.3, SpecAugment (20 / 4), noise 0.8 / 0.2, head dropout 0.3, out lengths
    17 / 9 / 12 of T'=18 (ld 24)."""
    _, batch = small_fixture()
    X, y, X_len, y_len, day = batch
    torch.manual_seed(1)                                           # the host SpecAugment draw
    m = build_small(precision).train()
    sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    opt = nsd.FusedAdamW(m.parameters(), **OPT, max_grad_norm=1.0)
    if precision == "bf16":
        opt.attach_shadows(m._shadows)
    got, calls = our_step(m, opt, batch, noise_seed=77)
    sites = sites_of(calls)
    check_sites(sites, 6, 0.3, 0.3)
    Tn = sites[2]["T"]
    lens = m.compute_output_lengths(X_len.to(DEV), Tn).to(torch.int32).contiguous()
    masks, Xn, stats = rebuild(sites, X, lens)
    check_coverage(masks, stats, lens, Tn)
    err = compare(got, reference_run(sd, batch, masks, SMALL_PORT, Xn=Xn), precision)
    ctl = {}
    for name, kw in CONTROLS:
        mk, xn, _ = rebuild(sites, X, lens, **kw)
        e = compare(got, reference_run(sd, batch, mk, SMALL_PORT, Xn=xn), precision)
        ctl[name] = dict(score=e["score"], worst=e["worst"], lp_abs=e["lp_abs"], loss_rel=e["loss_rel"], worst_grad_rel_l2=max(e["grad_rel_l2"].values()))
    print(f"train step small {precision}: lp {err['lp_abs']:.2e} inter {err['inter_abs']:.2e} loss rel {err['loss_rel']:.2e} worst grad rel-L2 "
          f"{max(err['grad_rel_l2'].values()):.2e} score {err['score']:.3f} ({err['worst']}); controls " +
          ", ".join(f"{k} {v['score']:.1f}" for k, v in ctl.items()))
    record(f"train_step_small_{precision}", dict(err, controls=ctl, bands=masks["bands"]))
    assert err["score"] < 1.0, (err["worst"], err["score"])
    for name, c in ctl.items():
        assert c["score"] > CONTROL_MARGIN, (name, c)


# bf16 at the competition architecture (B=8): about 3x the B200 measurements (log-probs 1.3e-2, InterCTC 1.2e-2, worst gradient
# 2.6e-2 rel L2 (frontend.temporal_conv.weight: 7.5k frames of bf16-rounded terms) / 3.1e-2 max over max; the loss, measured
# 1.9e-6 rel, keeps the small size's bound)
BF16_TOL_COMP = dict(lp_abs=0.04, inter_abs=0.04, loss_rel=1e-4, grad_rel_l2=0.08, grad_max_rel=0.1)


@pytest.mark.gpu
@pytest.mark.parametrize("precision,B", [("fp32", 2), ("bf16", 8)])
def test_train_step_competition_architecture_matches_masked_reference(precision, B):
    """256 channels, 24 days, d=1024, 8 layers x 8 heads, FF 2048, conv k31, k32/s4, 41 classes, T=500 -> T'=118 (ld 120), with
    dropout 0.3, DropPath 0.3, SpecAugment (100 / 40), noise and head dropout on.  The host reference runs in fp32, as the
    regularisers-off test at this size does."""
    kw = dict(n_channels=256, n_classes=41, n_days=24, transformer_dropout=0.3, use_spec_augment=True, drop_path_prob=0.3)
    torch.manual_seed(0)
    m = nsd.NeuralTransformerCTCModel(device="cuda", precision=precision, **kw)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(torch.randn(p.shape, generator=g) * (0.02 if p.dim() >= 2 else 0.05) * (p.abs().mean() + 0.1))
    T = 500
    X = torch.randn(B, T, 256, generator=g)
    day = torch.randint(0, 24, (B,), generator=g)
    X_len = torch.randint(300, T + 1, (B,), generator=g).to(torch.int32); X_len[0] = T
    y_len = torch.randint(10, 40, (B,), generator=g).to(torch.int32)
    y = torch.zeros(B, int(y_len.max()), dtype=torch.int32)
    for b in range(B):
        y[b, :y_len[b]] = torch.randint(1, 41, (int(y_len[b]),), generator=g).to(torch.int32)
    batch = (X, y, X_len, y_len, day)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.to(DEV).train()
    opt = nsd.FusedAdamW(m.parameters(), **OPT, max_grad_norm=1.0)
    if precision == "bf16":
        opt.attach_shadows(m._shadows)
    torch.manual_seed(3)
    got, calls = our_step(m, opt, batch, noise_seed=5)
    sites = sites_of(calls)
    check_sites(sites, 8, 0.3, 0.3)
    Tn = sites[2]["T"]
    assert Tn == 118 and [s for s in sites if s["kind"] == "sm"][0]["ld"] == 120
    lens = m.compute_output_lengths(X_len.to(DEV), Tn).to(torch.int32).contiguous()
    masks, Xn, stats = rebuild(sites, X, lens)
    check_coverage(masks, stats, lens, Tn)
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = dict(n_layers=8, n_heads=8, temporal_kernel=32, temporal_stride=4, conv_kernel=31)
    err = compare(got, reference_run(sd, batch, masks, cfg, dtype=torch.float32, Xn=Xn), precision, tol=BF16_TOL_COMP)
    print(f"train step competition {precision} B={B}: lp {err['lp_abs']:.2e} inter {err['inter_abs']:.2e} loss rel {err['loss_rel']:.2e} "
          f"worst grad rel-L2 {max(err['grad_rel_l2'].values()):.2e} score {err['score']:.3f} ({err['worst']})")
    record(f"train_step_competition_{precision}_B{B}", err)
    assert err["score"] < 1.0, (err["worst"], err["score"])


# ---------------------------------------------------------------------------------------------------------------------
# D / E. three optimizer steps (eager and graphed) against torch.optim.AdamW + clip_grad_norm_ in fp64
# ---------------------------------------------------------------------------------------------------------------------
def reference_trajectory(sd, batch, steps, cfg):
    """torch.optim.AdamW + clip_grad_norm_(1.0) with each step's lr (trainer:144-162, 251-260) over the masked reference;
    ``steps``: (masks, noised X, lr) per step.  -> per step (loss, gradients, parameters after), parameters, optimizer."""
    X, y, X_len, y_len, day = batch
    names = [k for k in sd if k not in ("pos_enc.pe", "frontend.gaussian_kernel")]
    params = {k: sd[k].double().clone().requires_grad_(True) for k in names}
    fixed = {k: v.double() for k, v in sd.items()}
    ropt = torch.optim.AdamW(list(params.values()), **OPT)
    out = []
    for masks, Xn, lr in steps:
        ropt.zero_grad()
        lp, olen, inter = MO.forward({**fixed, **params}, Xn, day, X_len, masks=masks, **cfg)
        loss = CP.training_loss(lp, inter, y, olen, y_len, label_smoothing=LS, interctc_weight=IW)
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in params.items()}
        torch.nn.utils.clip_grad_norm_(list(params.values()), max_norm=1.0)
        for grp in ropt.param_groups:
            grp["lr"] = lr
        ropt.step()
        out.append(dict(loss=loss.item(), grads=grads, params={k: p.detach().clone() for k, p in params.items()}))
    return out, params, ropt


def trajectory_errors(ours, ref, p0, m, opt, rparams, ropt):
    """Per step: loss (rel), worst gradient rel-L2, parameter change since the start (rel-L2, max over max); at the end: moments."""
    pm = dict(m.named_parameters())
    e = dict(loss=[o["loss"] for o in ours], loss_ref=[r["loss"] for r in ref],
             loss_rel=[abs(o["loss"] - r["loss"]) / abs(r["loss"]) for o, r in zip(ours, ref)],
             grad_rel_l2=[max(rel_l2(o["grads"][k], g) for k, g in r["grads"].items()) for o, r in zip(ours, ref)],
             delta_rel_l2=[max(rel_l2(o["params"][k] - p0[k], r["params"][k] - p0[k]) for k in rparams) for o, r in zip(ours, ref)],
             delta_max_rel=[max(max_rel(o["params"][k] - p0[k], r["params"][k] - p0[k]) for k in rparams) for o, r in zip(ours, ref)])
    e["moment_rel_l2"] = max(max(rel_l2(f64(opt.state[pm[k]]["exp_avg"]), ropt.state[q]["exp_avg"]),
                                 rel_l2(f64(opt.state[pm[k]]["exp_avg_sq"]), ropt.state[q]["exp_avg_sq"])) for k, q in rparams.items())
    return e


def assert_trajectory(e, precision):
    tol = TRAJ_TOL[precision]
    for k in ("loss_rel", "grad_rel_l2", "delta_rel_l2", "delta_max_rel"):
        assert max(e[k]) < tol[k], (k, e[k])
    assert e["moment_rel_l2"] < tol["moment_rel_l2"], e["moment_rel_l2"]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_three_adamw_steps_match_torch_adamw(precision):
    """Three eager conformer_train_steps, FusedAdamW(max_grad_norm=1) with the warm-up / cosine lr, every regulariser on."""
    _, batch = small_fixture()
    X, y, X_len, y_len, day = batch
    torch.manual_seed(2)
    m = build_small(precision).train()
    sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    p0 = {n: f64(p) for n, p in m.named_parameters()}
    opt = nsd.FusedAdamW(m.parameters(), **OPT, max_grad_norm=1.0)
    if precision == "bf16":
        opt.attach_shadows(m._shadows)
    ours, steps, seeds = [], [], []
    lens = None
    for k in range(3):
        lr = OPT["lr"] * nsd.lr_lambda(k, *SCHED)
        for grp in opt.param_groups:
            grp["lr"] = lr
        got, calls = our_step(m, opt, batch, noise_seed=500 + k)
        got["params"] = {n: f64(p) for n, p in m.named_parameters()}
        sites = sites_of(calls)
        check_sites(sites, 6, 0.3, 0.3)
        seeds += seeds_of(sites)
        if lens is None:
            lens = m.compute_output_lengths(X_len.to(DEV), sites[2]["T"]).to(torch.int32).contiguous()
        masks, Xn, _ = rebuild(sites, X, lens)
        ours.append(got)
        steps.append((masks, Xn, lr))
    assert len(set(seeds)) == len(seeds)                                # no seed repeats across the three steps
    assert not torch.equal(steps[0][0]["fe"], steps[1][0]["fe"]) and not torch.equal(steps[0][0]["blocks"][0]["attn_p"], steps[1][0]["blocks"][0]["attn_p"])
    ref, rparams, ropt = reference_trajectory(sd, batch, steps, SMALL_PORT)
    e = trajectory_errors(ours, ref, p0, m, opt, rparams, ropt)
    print(f"three AdamW steps {precision}: " + ", ".join(f"{k} {v}" for k, v in e.items()))
    record(f"trajectory_eager_{precision}", e)
    assert_trajectory(e, precision)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_graphed_step_replays_match_masked_reference_and_adamw(precision):
    """GraphedConformerStep with every regulariser on.  The first step() runs two eager warm-ups, the capture and the first
    replay; every replay uses the seeds recorded during the capture plus that replay's device offset, and the SpecAugment bands
    of that step's host draw from the device array.  For three replays: the gradients left in p.grad, the loss and the update
    against the masked reference (masks rebuilt under the replay's offset, noise with noise_seed 12345 under it) and AdamW."""
    _, batch = small_fixture()
    X, y, X_len, y_len, day = batch
    B, T = X.shape[:2]
    torch.manual_seed(2)                                           # the third host draw (the first replay's) has both kinds of band
    m = build_small(precision).train()
    sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    p0 = {n: f64(p) for n, p in m.named_parameters()}
    opt = nsd.FusedAdamW(m.parameters(), **OPT, max_grad_norm=1.0)
    if precision == "bf16":
        opt.attach_shadows(m._shadows)
    probe = lambda: act_mask(4096, 0.3, 99)
    plain = probe()
    drawn, real_draw = [], m.spec_augment.draw
    m.spec_augment.draw = lambda T_, F_: drawn.append(real_draw(T_, F_)) or drawn[-1]
    gs = nsd.GraphedConformerStep(m, opt, B, T, int(y.shape[1]), label_smoothing=LS, interctc_weight=IW, white_noise_sd=NOISE[0],
                                  constant_offset_sd=NOISE[1], base_lr=OPT["lr"], warmup_steps=SCHED[0], total_steps=SCHED[1])
    args = [t.to(DEV) for t in batch]
    ours, steps, offsets, in_graph = [], [], [], None
    try:
        with recording() as rec:
            gs.step(*args)
        noise_at = [i for i, (name, _) in enumerate(rec.calls) if name == "nsd_input_noise"]
        assert len(noise_at) == 3                                      # two eager warm-ups and the capture
        sites = sites_of(rec.calls[noise_at[-1]:])
        check_sites(sites, 6, 0.3, 0.3)
        assert sites[0]["seed"] == 12345 and sites[2]["bands"] == [0] * 8 and sites[2]["bands_dev"] == gs._bands.data_ptr()
        Tn = sites[2]["T"]
        lens = m.compute_output_lengths(X_len.to(DEV), Tn).to(torch.int32).contiguous()
        for k in range(3):
            if k:
                gs.step(*args)
            torch.cuda.synchronize()
            offsets.append(int(gs._seed.item()) & U64)
            bands = [int(v) for v in gs._bands.tolist()]
            assert bands == drawn[-1], (bands, drawn[-1])               # the device array holds this step's host draw
            masks, Xn, stats = rebuild(sites, X, lens, bands=bands)     # the kernels add the live device offset
            if k == 0:
                check_coverage(masks, stats, lens, Tn)
            ours.append(dict(loss=gs.loss.item(), grads={n: f64(p.grad) for n, p in m.named_parameters()},
                             params={n: f64(p) for n, p in m.named_parameters()}))
            steps.append((masks, Xn, OPT["lr"] * nsd.lr_lambda(k, *SCHED)))
        in_graph = probe()
        assert gs.steps_done == 3
    finally:
        gs.close()
        del m.spec_augment.draw
    assert torch.equal(probe(), plain) and not torch.equal(in_graph, plain)          # close() clears the offset
    assert len(set(offsets)) == 3
    assert not torch.equal(steps[0][0]["fe"], steps[1][0]["fe"]) and not torch.equal(steps[0][1], steps[1][1])
    ref, rparams, ropt = reference_trajectory(sd, batch, steps, SMALL_PORT)
    e = trajectory_errors(ours, ref, p0, m, opt, rparams, ropt)
    print(f"graphed replays {precision}: offsets {[hex(o) for o in offsets]}; " + ", ".join(f"{k} {v}" for k, v in e.items()))
    record(f"trajectory_graphed_{precision}", dict(e, offsets=offsets))
    assert_trajectory(e, precision)
