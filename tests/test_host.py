"""CPU-side checks: the C-ABI library loads and exports every symbol include/nsd_b200.h declares, the Python
mirror keeps the reference's module contract, and the product path refuses to run without CUDA (no fallback)."""
import hashlib
import json
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT

import neural_speech_decoder_b200 as nsd
from neural_speech_decoder_b200 import _lib

HEADER = os.path.join(ROOT, "include", "nsd_b200.h")
KW = dict(neural_dim=16, n_classes=10, hidden_dim=32, layer_dim=2, nDays=3, dropout=0.0, strideLen=4, kernelLen=14,
          gaussianSmoothWidth=2.0, bidirectional=True)
CONFORMER_KW = dict(n_channels=32, n_classes=11, n_days=3, frontend_dim=64, latent_dim=64, autoencoder_hidden_dim=32, transformer_layers=6,
                    transformer_heads=4, transformer_ff_dim=128)


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nsd_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.lib()                       # raises ImportError if the .so was not built
    syms = declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/nsd_b200.h but not exported"
        assert s in _lib.SIGNATURES, f"{s} has no ctypes signature in _lib.py"
    assert sorted(_lib.SIGNATURES) == syms
    assert lib.nsd_version() >= 100
    assert lib.nsd_ctc_workspace(10, 2, 5, 3) > 0 and lib.nsd_gru_bwd_workspace(2, 8) == 2 * 8 * 4


def test_no_cpu_fallback():
    m = nsd.GRUDecoder(device="cpu", **KW)
    with pytest.raises(nsd.NsdError):
        m.forward(torch.zeros(2, 40, 16), torch.zeros(2, dtype=torch.int64))
    with pytest.raises(nsd.NsdError):
        nsd.CTCLoss(zero_infinity=True)(torch.zeros(5, 2, 4), torch.ones(2, 2, dtype=torch.int32),
                                        torch.tensor([5, 5]), torch.tensor([2, 2]))
    with pytest.raises(nsd.NsdError):
        nsd.greedy_decode(torch.zeros(5, 2, 4), torch.tensor([5, 5]))
    # and nothing in the product package imports the oracle
    pkg = os.path.join(ROOT, "neural_speech_decoder_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            assert "oracle" not in open(os.path.join(pkg, fn)).read(), fn


def test_out_lens_matches_trainer_line():
    x_len = torch.tensor([500, 501, 503, 504, 32, 35, 36], dtype=torch.int32)
    assert nsd.out_lens(x_len, 32, 4).tolist() == [117, 117, 117, 118, 0, 0, 1]     # trainer:209 (SURVEY section 8)
    assert nsd.out_lens(x_len, 32, 4).dtype == torch.int32


def test_module_contract():
    torch.manual_seed(0)
    m = nsd.GRUDecoder(device="cpu", **KW)
    assert m.kernelLen == 14 and m.strideLen == 4
    sd = m.state_dict()
    assert sd["dayWeights"].shape == (3, 16, 16) and sd["dayBias"].shape == (3, 1, 16)
    assert torch.equal(sd["dayWeights"][1], torch.eye(16)) and sd["gaussianSmoother.weight"].shape == (16, 1, 20)
    assert sd["gru_decoder.weight_ih_l0"].shape == (96, 16 * 14) and sd["gru_decoder.weight_ih_l1_reverse"].shape == (96, 64)
    assert sd["fc_decoder_out.weight"].shape == (11, 64)
    assert "gaussianSmoother.weight" not in dict(m.named_parameters())
    w = sd["gru_decoder.weight_hh_l0"][:32]
    assert torch.allclose(w @ w.T, torch.eye(32), atol=1e-5) or torch.allclose(sd["gru_decoder.weight_hh_l0"].T @ sd["gru_decoder.weight_hh_l0"], torch.eye(32), atol=1e-5)
    with pytest.raises(ZeroDivisionError):
        nsd.GRUDecoder(16, 10, 32, 1, gaussianSmoothWidth=0)


def state_record(m):
    """Every state-dict entry of ``m`` in order as [name, shape, dtype, SHA-256 of its bytes], and the parameter names:
    the form in which tests/golden/reference_init.json keeps the reference modules' seeded initial states."""
    state = [[k, list(v.shape), str(v.dtype), hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest()]
             for k, v in m.state_dict().items()]
    return {"state": state, "parameters": [n for n, _ in m.named_parameters()]}


def reference_init(name):
    with open(os.path.join(GOLDEN, "reference_init.json")) as f:
        return json.load(f)[name]


def assert_same_state(mine, ref):
    got = state_record(mine)
    assert [e[0] for e in got["state"]] == [e[0] for e in ref["state"]]
    for g, r in zip(got["state"], ref["state"]):
        assert g == r, g[0]
    assert got["parameters"] == ref["parameters"]


@pytest.mark.parametrize("bi", [False, True])
def test_same_seed_same_weights_as_reference(bi):
    """The reference's GRUDecoder under torch seed 3 (tests/golden/reference_init.json) and ours under the same seed hold
    bit-identical state dicts: same names in the same order, same shapes, same bytes, same parameters."""
    kw = dict(KW, bidirectional=bi)
    ref = reference_init("gru_bi" if bi else "gru_uni")
    torch.manual_seed(3)
    mine = nsd.GRUDecoder(device="cpu", **kw)
    assert_same_state(mine, ref)
    other = nsd.GRUDecoder(device="cpu", **kw)                # later RNG draws: other weights until the load
    other.load_state_dict(mine.state_dict(), strict=True)     # loadModel path (trainer:409)
    assert_same_state(other, ref)


def test_fused_adam_rejects_cpu_parameters():
    p = torch.nn.Parameter(torch.zeros(4))
    p.grad = torch.ones(4)
    with pytest.raises(RuntimeError):
        nsd.adam.FusedAdam([p], lr=0.1).step()


def test_streaming_frame_arithmetic():
    """StreamingDecoder's host logic (no GPU): which frames are complete after n bins, and which window recomputes them.
    Checked against the definitions: frame j reads smoothed bins [S*j, S*j+K); smoothed bin t reads raw bins
    [t-left, t+right] (augmentations.py:91: 20 taps, padding 'same' -> left 9, right 10)."""
    from neural_speech_decoder_b200.streaming import complete_frames, window_for
    for K, S, left, right in ((32, 4, 9, 10), (14, 2, 9, 10), (16, 4, 4, 5), (7, 3, 9, 10)):
        halo = -(-left // S) * S
        for n in range(0, 120):
            brute = 0
            while S * brute + K - 1 + right <= n - 1:      # last raw bin frame `brute` needs has arrived
                brute += 1
            assert complete_frames(n, K, S, right) == brute
        for j0 in range(0, 40):
            r0, skip = window_for(j0, S, halo)
            assert r0 % S == 0 and r0 + skip * S == S * j0           # the kept frames start exactly at frame j0
            assert r0 == 0 or S * j0 - r0 >= left                    # ... with the smoothing's full left reach in the window


def test_conformer_same_seed_same_weights_as_reference():
    """Drop-in contract of the Conformer (SURVEY 8b applied to transformer_ctc.py:333-420): same constructor, same parameter /
    buffer names, same RNG consumption order -> the same seed (0) gives a bit-identical state dict to the reference's
    (tests/golden/reference_init.json), and a state dict of that form loads strictly."""
    kw = CONFORMER_KW
    ref = reference_init("conformer")
    torch.manual_seed(0)
    b = nsd.NeuralTransformerCTCModel(device="cpu", **kw)
    assert_same_state(b, ref)
    other = nsd.NeuralTransformerCTCModel(device="cpu", **kw)
    other.load_state_dict(b.state_dict(), strict=True)
    assert_same_state(other, ref)
    with pytest.raises(nsd.NsdError):
        b(torch.zeros(2, 40, 32), torch.zeros(2, dtype=torch.int64), torch.tensor([40, 40]))      # no CPU fallback
    x_len = torch.tensor([500, 501, 503, 504, 32, 35, 36], dtype=torch.int32)
    c = nsd.NeuralTransformerCTCModel(device="cpu", **{**kw, "temporal_kernel": 32})
    assert c.compute_output_lengths(x_len, 118).tolist() == [117, 117, 117, 118, 0, 0, 1]
