"""Host checks of the packed-sequence oracle (tests/packed_oracle.py) against PortGRUDecoder."""
from __future__ import annotations

import pytest
import torch

from neural_speech_decoder_b200.synthetic import make_batch
from oracle import torch_port as P
from packed_oracle import frame_counts, packed_forward

SMALL = dict(neural_dim=32, n_classes=10, hidden_dim=24, layer_dim=2, nDays=4, strideLen=4, kernelLen=16, gaussianSmoothWidth=2.0)


def _port(bidirectional):
    torch.manual_seed(7)
    return P.PortGRUDecoder(**SMALL, bidirectional=bidirectional).double().eval()


@pytest.mark.parametrize("bidirectional", [False, True], ids=["uni", "bi"])
def test_full_lengths_equal_port(bidirectional):
    """Every X_len = T: the packed restatement is PortGRUDecoder itself (to 1e-12)."""
    port = _port(bidirectional)
    X, _, _, _, day = make_batch(5, 70, n_feat=32, n_days=4, n_classes=10, seed=3, kernel_len=16, stride_len=4)
    X = X.double()
    with torch.no_grad():
        ref = port(X, day)
        got = packed_forward(port, X, day, torch.full((5,), 70))
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() <= 1e-12 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("bidirectional", [False, True], ids=["uni", "bi"])
def test_each_utterance_runs_alone(bidirectional):
    """Ragged lengths: utterance b's valid-frame logits are those of the port on X[b, :X_len[b]] alone, and past its frames
    the logits are the output bias."""
    port = _port(bidirectional)
    X, _, X_len, _, day = make_batch(4, 80, n_feat=32, n_days=4, n_classes=10, seed=4, ragged=True, kernel_len=16, stride_len=4)
    X_len[1] = 16                                          # one frame
    X = X.double()
    X[1, 16:] = float("nan")                               # padding never reaches a result
    n = frame_counts(X_len, 16, 4, 80)
    with torch.no_grad():
        got = packed_forward(port, X, day, X_len)
        for b in range(4):
            alone = port(X[b:b + 1, :int(X_len[b])], day[b:b + 1])[0]
            nb = int(n[b])
            assert alone.shape[0] == nb
            assert (got[b, :nb] - alone).abs().max().item() <= 1e-12
            assert torch.equal(got[b, nb:], port.fc.bias.expand(got.shape[1] - nb, -1))
