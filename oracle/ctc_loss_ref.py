"""float64 numpy restatement of K5e, the CTC loss and gradient of ``csrc/ctc_loss.cu``, and a float64 torch reference of
the Bi-GRU head's training step.

TEST INFRASTRUCTURE (oracle).  ``loss_grad`` runs the forward (alpha) and backward (beta) recurrences over the extended
target (blank, y0, blank, ..., blank) with K5c's transitions (stay, s-1, and s-2 only between different labels) and
returns the per-clip loss and dL/dlogp = -scale * gamma, gamma_t(k) the posterior occupancy of label k at frame t, with
K5e's statuses.  ``head_reference`` is LipNet's head in float64 torch: two ``nn.GRU``s, ``Linear``, ``log_softmax``
and the same keep masks, for autograd gradients.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np

NEG_INF = -np.inf


def _shift(x: np.ndarray, k: int, fill=NEG_INF) -> np.ndarray:   # x[s - k] (k > 0) or x[s + |k|] (k < 0)
    out = np.full_like(x, fill)
    if k > 0:
        out[k:] = x[:max(len(x) - k, 0)]
    else:
        out[:len(x) + k] = x[-k:]
    return out


def loss_grad(logp: np.ndarray, y: Sequence[int], input_len: Optional[int] = None, blank: int = 0,
              scale: float = 1.0, zero_infinity: bool = False) -> Tuple[float, np.ndarray]:
    """One clip: logp [T, V]; returns (nll, grad [T, V] float64)."""
    lp = np.asarray(logp, dtype=np.float64)
    T, V = lp.shape
    y = np.asarray(y, dtype=np.int64)
    L = len(y)
    n = T if input_len is None else int(input_len)
    grad = np.zeros((T, V))
    if not 0 <= n <= T or ((y < 0) | (y >= V) | (y == blank)).any():
        return np.nan, np.full((T, V), np.nan)
    if np.isnan(lp[:n]).any():
        grad[:n] = np.nan
        return np.nan, grad
    if n == 0:
        return (0.0, grad) if L == 0 else ((0.0, grad) if zero_infinity else (np.inf, grad))
    S = 2 * L + 1
    lab = np.full(S, blank, np.int64)
    lab[1::2] = y
    skip = np.zeros(S, bool)
    skip[3::2] = y[1:] != y[:-1]
    alpha = np.full((n, S), NEG_INF)
    alpha[0, :min(S, 2)] = lp[0, lab[:2]]
    with np.errstate(invalid="ignore", divide="ignore"):
        for t in range(1, n):
            a = alpha[t - 1]
            alpha[t] = np.logaddexp(np.logaddexp(a, _shift(a, 1)), np.where(skip, _shift(a, 2), NEG_INF)) + lp[t, lab]
        ll = float(np.logaddexp(alpha[n - 1, S - 1], alpha[n - 1, S - 2]) if S > 1 else alpha[n - 1, 0])
        if ll == NEG_INF:
            grad[:n] = 0.0 if zero_infinity else np.nan
            return (0.0 if zero_infinity else np.inf), grad
        beta = np.full((n, S), NEG_INF)
        beta[n - 1, max(S - 2, 0):] = 0.0
        skip_out = _shift(skip, -2, False)          # the skip leaves s for s + 2
        for t in range(n - 2, -1, -1):
            bx = beta[t + 1] + lp[t + 1, lab]
            beta[t] = np.logaddexp(np.logaddexp(bx, _shift(bx, -1)), np.where(skip_out, _shift(bx, -2), NEG_INF))
        gamma = np.exp(alpha + beta - ll)
    for s in range(S):
        grad[:n, lab[s]] -= scale * gamma[:, s]
    return -ll, grad


def loss_grad_batch(logp: np.ndarray, targets: np.ndarray, target_lens: Sequence[int], input_lens: Sequence[int],
                    blank: int = 0, scale: Optional[Sequence[float]] = None, zero_infinity: bool = False):
    """The padded layout of ``avsync_b200.ctc_loss``: logp [B, T, V], targets [B, Lmax] -> (nll [B], grad [B, T, V])."""
    B, T, V = logp.shape
    nll, grad = np.empty(B), np.empty((B, T, V))
    for b in range(B):
        L = int(target_lens[b])
        if not 0 <= L <= targets.shape[1]:
            nll[b], grad[b] = np.nan, np.nan
            continue
        nll[b], grad[b] = loss_grad(logp[b], targets[b, :L], int(input_lens[b]), blank,
                                    1.0 if scale is None else float(scale[b]), zero_infinity)
    return nll, grad


def head_reference(state: dict, emb, masks=(None, None), p: float = 0.0, dtype=None):
    """LipNet's head in torch (float64 by default) with the given keep masks: returns (log-probs, modules) where
    modules = (gru1, gru2, fc) carry the parameters of ``state`` (LipNet state_dict keys) with requires_grad."""
    import torch
    import torch.nn as nn
    dtype = dtype or torch.float64
    H = state["gru1.weight_hh_l0"].shape[1]
    in_dim = state["gru1.weight_ih_l0"].shape[1]
    V = state["fc.weight"].shape[0]
    dev = emb.device
    gru1 = nn.GRU(in_dim, H, batch_first=True, bidirectional=True).to(dev, dtype)
    gru2 = nn.GRU(2 * H, H, batch_first=True, bidirectional=True).to(dev, dtype)
    fc = nn.Linear(2 * H, V).to(dev, dtype)
    with torch.no_grad():
        for name, mod in (("gru1", gru1), ("gru2", gru2), ("fc", fc)):
            for k, prm in mod.named_parameters():
                prm.copy_(state[f"{name}.{k}"].to(dev, dtype))
    x, _ = gru1(emb.to(dtype))
    if masks[0] is not None:
        x = x * masks[0].to(dtype) * (1.0 / (1.0 - p))
    x, _ = gru2(x)
    if masks[1] is not None:
        x = x * masks[1].to(dtype) * (1.0 / (1.0 - p))
    return torch.log_softmax(fc(x), dim=-1), (gru1, gru2, fc)
