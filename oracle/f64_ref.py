"""float64 CPU restatements of the STCNN layers (K2), the Bi-GRU head (K3) and the shift-sweep detector score (K4).

TEST INFRASTRUCTURE (oracle).  Independent of ``lipnet_ref`` / ``sweep_ref``: the head is built from
``torch.nn.GRU`` / ``torch.nn.functional.log_softmax`` in float64 rather than the hand-written float32 recurrence of
``lipnet_ref._gru_dir``, and the detector score is written out in float64 from its definition.  The kernels' float32
results are compared against these, so that an error of the float32 oracle cannot hide the same error in a kernel.
The STCNN layer forms its operands the way the tensor-core kernels do (bf16 rounding, hi/lo split) and sums in float64,
so that a kernel's error against it is its own accumulation and output rounding only.
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


# ---------------------------------------------------------------------------------------------------- K2: STCNN layer
def bf16_round(x: torch.Tensor) -> torch.Tensor:
    """float32 -> nearest bfloat16, ties to even, back as float32: the kernels' ``__float2bfloat16_rn`` and the host's
    ``f2bf`` (conv_umma.cu) on finite values."""
    return x.float().to(torch.bfloat16).float()


def stcnn_operands(v: torch.Tensor, precision: str):
    """The operand(s) a layer multiplies for the float32 tensor ``v`` (activations or weights), as float64 terms whose
    products the kernel sums: fp32 [v]; bf16 [bf16(v)]; bf16x3 [hi, lo] with hi = bf16(v), lo = bf16(v - hi) (the
    difference is exact in float32)."""
    v = v.float()
    if precision == "fp32":
        return [v.double()]
    hi = bf16_round(v)
    if precision == "bf16":
        return [hi.double()]
    if precision == "bf16x3":
        return [hi.double(), bf16_round(v - hi).double()]
    raise ValueError(precision)


def stcnn_layer_f64(x, w, b, precision: str, t_out=None):
    """One STCNN layer in float64: Conv3d (3 x KH x KW, "same" padding), + bias, ReLU, MaxPool3d((1, 2, 2)).

    x [B, Cin, T, H, W], w [Cout, Cin, 3, KH, KW], b [Cout] (float32 values; the activations the kernel reads).  The
    operands are formed as the kernel forms them (stcnn_operands): fp32 as given, bf16 rounded, bf16x3 split into hi
    and lo with the sum x_hi.w_hi + x_hi.w_lo + x_lo.w_hi (the lo.lo product is not computed, as in the kernel).  Every
    product and sum is then float64.  ``t_out`` (a list of output time steps, default all) computes only those steps:
    each needs input planes t - 1 .. t + 1, zero outside the clip.

    Returns (out [B, Cout, len(t_out), H // 2, W // 2], S of the same shape): S is the error scale of an output,
    sum |x . w| + |b| over the taps of a conv output, the largest over the outputs of its pool window (a maximum is at
    most as far off as the farthest of its candidates, whichever of them wins)."""
    x = torch.as_tensor(x).detach().cpu().float()
    w = torch.as_tensor(w).detach().cpu().float()
    b = torch.as_tensor(b).detach().cpu().double()
    B, Cin, T, H, W = x.shape
    KH, KW = w.shape[3], w.shape[4]
    steps = list(range(T)) if t_out is None else [int(t) for t in t_out]
    # the three input planes of every requested step, zero planes outside [0, T): [B * n, Cin, 3, H, W]
    xz = torch.cat([x.new_zeros(B, Cin, 1, H, W), x, x.new_zeros(B, Cin, 1, H, W)], dim=2)
    xs = torch.stack([xz[:, :, t:t + 3] for t in steps], dim=1).reshape(B * len(steps), Cin, 3, H, W)
    xo, wo = stcnn_operands(xs, precision), stcnn_operands(w, precision)
    pad = (0, KH // 2, KW // 2)
    with torch.no_grad():
        if precision == "bf16x3":
            acc = F.conv3d(xo[0], wo[0] + wo[1], padding=pad) + F.conv3d(xo[1], wo[0], padding=pad)
            xa, wa = (xo[0] + xo[1]).abs(), (wo[0] + wo[1]).abs()
        else:
            acc = F.conv3d(xo[0], wo[0], padding=pad)
            xa, wa = xo[0].abs(), wo[0].abs()
        s = F.conv3d(xa, wa, padding=pad) + b.abs().view(1, -1, 1, 1, 1)
        out = F.relu(F.max_pool3d(acc + b.view(1, -1, 1, 1, 1), (1, 2, 2)))
        s = F.max_pool3d(s, (1, 2, 2))
    Cout, Ho, Wo = out.shape[1], out.shape[3], out.shape[4]
    out = out.reshape(B, len(steps), Cout, Ho, Wo).permute(0, 2, 1, 3, 4).contiguous()
    s = s.reshape(B, len(steps), Cout, Ho, Wo).permute(0, 2, 1, 3, 4).contiguous()
    return out, s
