"""The fp64 input-gradient oracle (tests/frontend_input_oracle.py) against torch autograd through the reference's own front-end
operators (conv1d padding="same", index_select + einsum, softsign, unfold; oracle/torch_port.py), on the host."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from frontend_input_oracle import frontend_bwd_input
from oracle import nsd_oracle as O


def _torch_frontend(x, taps, W, b, day, K, S):
    N = x.shape[2]
    y = F.conv1d(x.permute(0, 2, 1), taps.view(1, 1, -1).repeat(N, 1, 1), groups=N, padding="same").permute(0, 2, 1)
    pre = torch.einsum("btd,bdk->btk", y, torch.index_select(W, 0, day)) + torch.index_select(b, 0, day)
    z = F.softsign(pre)
    return F.unfold(z.permute(0, 2, 1).unsqueeze(3), (K, 1), stride=S).permute(0, 2, 1), pre


@pytest.mark.parametrize("B,T,N,K,S,ntaps", [(3, 61, 6, 16, 4, 20), (2, 33, 5, 3, 5, 7), (2, 40, 4, 8, 2, 1), (2, 30, 3, 6, 3, 4)])
def test_input_gradient_oracle_matches_autograd(B, T, N, K, S, ntaps):
    g = torch.Generator().manual_seed(B * 1000 + T)
    n_days = 3
    x = torch.randn(B, T, N, generator=g, dtype=torch.float64, requires_grad=True)
    taps = torch.rand(ntaps, generator=g, dtype=torch.float64)
    W = torch.randn(n_days, N, N, generator=g, dtype=torch.float64)
    b = torch.randn(n_days, 1, N, generator=g, dtype=torch.float64)
    day = torch.tensor([(2 * i + 1) % n_days for i in range(B)])
    patches, pre = _torch_frontend(x, taps, W, b, day, K, S)
    dp = torch.randn(patches.shape, generator=g, dtype=torch.float64)
    patches.backward(dp)
    got = frontend_bwd_input(dp.numpy(), {"pre": pre.detach().numpy()}, W.numpy(), day.numpy(), taps.numpy(), T, K, S)
    np.testing.assert_allclose(got, x.grad.numpy(), rtol=1e-10, atol=1e-12)
    # the numpy forward of the oracle agrees with the torch operators, so the two backward restatements share a forward
    pn, _ = O.frontend_fwd(x.detach().numpy(), taps.numpy(), W.numpy(), b.numpy(), day.numpy(), K, S)
    np.testing.assert_allclose(pn, patches.detach().numpy(), rtol=1e-12, atol=1e-12)
