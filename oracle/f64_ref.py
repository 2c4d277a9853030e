"""float64 CPU restatements of the Bi-GRU head (K3) and the shift-sweep detector score (K4).

TEST INFRASTRUCTURE (oracle).  Independent of ``lipnet_ref`` / ``sweep_ref``: the head is built from
``torch.nn.GRU`` / ``torch.nn.functional.log_softmax`` in float64 rather than the hand-written float32 recurrence of
``lipnet_ref._gru_dir``, and the detector score is written out in float64 from its definition.  The kernels' float32
results are compared against these, so that an error of the float32 oracle cannot hide the same error in a kernel.
K1 needs no counterpart here: ``mfcc_ref`` already computes librosa's chain in float64 where librosa does.
"""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch
import torch.nn.functional as F


def _bigru_f64(params: Dict[str, torch.Tensor], prefix: str, x: torch.Tensor) -> torch.Tensor:
    H = params[f"{prefix}.weight_hh_l0"].shape[1]
    gru = torch.nn.GRU(x.shape[-1], H, bidirectional=True, batch_first=True).double()
    gru.load_state_dict({k[len(prefix) + 1:]: v.detach().double() for k, v in params.items()
                         if k.startswith(prefix + ".")})
    return gru(x)[0]


def bigru_head_f64(params: Dict[str, torch.Tensor], emb) -> torch.Tensor:
    """gru1 -> gru2 -> fc -> log_softmax of ``LipNet`` (model.py:84-95), eval mode, all in float64.
    ``params`` holds the ``gru1.* / gru2.* / fc.*`` entries of a LipNet state dict; emb [B, T, in] -> [B, T, vocab]."""
    with torch.no_grad():
        x = torch.as_tensor(emb).detach().cpu().double()
        x = _bigru_f64(params, "gru1", x)
        x = _bigru_f64(params, "gru2", x)
        x = x @ params["fc.weight"].double().t() + params["fc.bias"].double()
        return F.log_softmax(x, dim=-1)


def detector_scores_f64(w1, b1, w2, b2, v, a) -> np.ndarray:
    """sigmoid(w2 . relu(W1 . cat[v, a_k] + b1) + b2) for every clip and shift, in float64.

    w1 [H, Dv + Da], b1 [H], w2 [1, H] or [H], b2 [1]; v [B, Dv], a [B, K, Da] -> scores [B, K].
    W1 . cat[v, a_k] is evaluated as W1[:, :Dv] . v + W1[:, Dv:] . a_k (the same sum, grouped), so that the visual
    product is formed once per clip rather than once per shift."""
    f64 = [np.asarray(torch.as_tensor(t).detach().cpu().double()) for t in (w1, b1, w2, b2, v, a)]
    w1, b1, w2, b2, v, a = f64
    Dv = v.shape[1]
    hv = v @ w1[:, :Dv].T + b1                              # [B, H]
    h = np.maximum(hv[:, None, :] + a @ w1[:, Dv:].T, 0.0)   # [B, K, H]
    logit = h @ w2.reshape(-1) + b2.reshape(-1)[0]
    return 1.0 / (1.0 + np.exp(-logit))
