"""fp64 reference of the front end's gradient w.r.t. its input X (the transpose of model.py:84-101), next to
oracle/nsd_oracle.py:frontend_bwd, which gives the day parameters' gradients from the same dpatches.

  dz   = unfold_bwd(dpatches)                                   col2im
  dpre = dz / (1 + |pre|)^2                                     softsign'
  dy_b = dpre_b W[day_b]^T                                      the forward is pre = ys W + b
  dx[b,s,c] = sum_k taps[k] dy[b, s+L-k, c], 0 <= s+L-k < T     L = (ntaps-1)//2: the transpose of the "same"-padded smoother

Rows at or past (T'-1)*S + K have dz = 0 but still get dx from the smoother's reach.  The training noise is additive, so the
gradient passes through it unchanged.
"""
from __future__ import annotations

import numpy as np

from oracle import nsd_oracle as O


def frontend_bwd_input(dpatches, saved, day_w, day_idx, taps, T, kernel_len, stride_len):
    """dpatches [B,T',N*K]; saved["pre"] [B,T,N]; day_w [n_days,N,N]; taps [ntaps] -> dx [B,T,N] (float64)."""
    dp = np.asarray(dpatches, dtype=np.float64)
    dz = O.unfold_bwd(dp, T, kernel_len, stride_len)
    dpre = dz / (1.0 + np.abs(np.asarray(saved["pre"], dtype=np.float64))) ** 2
    W = np.asarray(day_w, dtype=np.float64)
    dy = np.stack([dpre[b] @ W[d].T for b, d in enumerate(np.asarray(day_idx))])
    taps = np.asarray(taps, dtype=np.float64)
    n = taps.shape[0]
    L = (n - 1) // 2
    dx = np.zeros_like(dy)
    for k in range(n):
        sh = L - k                                   # dx[s] += taps[k] dy[s + sh]
        lo, hi = max(0, -sh), min(T, T - sh)
        if lo < hi:
            dx[:, lo:hi] += taps[k] * dy[:, lo + sh:hi + sh]
    return dx
