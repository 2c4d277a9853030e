"""`model.LipNet` drop-in (reference: model.py:7-97) running on hand-written sm_100a kernels.

Same constructor, attribute names and ``state_dict`` keys as the reference module (so
``lipnet_final.pth`` loads in both the bare and the ``{'model_state_dict': ...}`` form,
misalignment_detection_train.py:299-309), but ``forward`` does not call ATen/cuDNN: the
STCNN runs in ``avs_stcnn_forward`` (K2) and the Bi-GRU head in ``avs_bigru_forward`` (K3).
``forward``, ``stcnn`` and ``gru_head`` are eval mode only; ``gru_head_train`` trains the Bi-GRU head on frozen STCNN
embeddings (``avs_bigru_train_forward`` / ``avs_bigru_train_backward``, K3b).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _native as N


class LipNet(nn.Module):
    def __init__(self, vocab_size: int, hidden_dim: int = 256, dropout_rate: float = 0.5,
                 precision: str = "bf16x3"):
        super().__init__()
        if precision not in N.PREC:
            raise ValueError(f"precision must be one of {sorted(N.PREC)}")
        self.precision = precision
        # parameter containers only — registered in the reference's order so default init and
        # state_dict keys are identical (model.py:22-48)
        self.conv1 = nn.Conv3d(1, 32, kernel_size=(3, 5, 5), padding=(1, 2, 2))
        self.pool1 = nn.MaxPool3d(kernel_size=(1, 2, 2))
        self.dropout1 = nn.Dropout3d(dropout_rate)
        self.conv2 = nn.Conv3d(32, 64, kernel_size=(3, 5, 5), padding=(1, 2, 2))
        self.pool2 = nn.MaxPool3d(kernel_size=(1, 2, 2))
        self.dropout2 = nn.Dropout3d(dropout_rate)
        self.conv3 = nn.Conv3d(64, 96, kernel_size=(3, 3, 3), padding=(1, 1, 1))
        self.pool3 = nn.MaxPool3d(kernel_size=(1, 2, 2))
        self.dropout3 = nn.Dropout3d(dropout_rate)
        self.conv_output_dim = 96 * 6 * 12          # model.py:50-55
        self.gru1 = nn.GRU(self.conv_output_dim, hidden_dim, batch_first=True, bidirectional=True)
        self.dropout_gru1 = nn.Dropout(dropout_rate)
        self.gru2 = nn.GRU(hidden_dim * 2, hidden_dim, batch_first=True, bidirectional=True)
        self.dropout_gru2 = nn.Dropout(dropout_rate)
        self.fc = nn.Linear(hidden_dim * 2, vocab_size)
        self.hidden_dim = hidden_dim
        self.vocab_size = vocab_size
        self._native = {}

    # ------------------------------------------------------------------ native handles
    def _key(self, params):
        return tuple((p.data_ptr(), p._version) for p in params) + (self.precision,)

    def _stcnn(self) -> N.Handle:
        params = [self.conv1.weight, self.conv1.bias, self.conv2.weight, self.conv2.bias,
                  self.conv3.weight, self.conv3.bias]
        key = self._key(params)
        cached = self._native.get("stcnn")
        if cached is None or cached[0] != key:
            N.device_check()
            for p in params:
                N.require_cuda(p, "LipNet parameters")
            keep = [N.f32c(p) for p in params]
            h = N.c_void_p()
            N.check(N.lib().avs_stcnn_create(*[N.ptr(t) for t in keep], N.PREC[self.precision],
                                             N.stream_ptr(), N.ctypes.byref(h)), "stcnn_create")
            cached = (key, N.Handle(h, N.lib().avs_stcnn_destroy, keep))
            self._native["stcnn"] = cached
        return cached[1]

    def _bigru(self) -> N.Handle:
        g1, g2 = self.gru1, self.gru2
        names = ["weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"]
        params = [getattr(g, n + s) for g in (g1, g2) for n in names for s in ("", "_reverse")]
        params += [self.fc.weight, self.fc.bias]
        key = self._key(params)
        cached = self._native.get("bigru")
        if cached is None or cached[0] != key:
            N.device_check()
            for p in params:
                N.require_cuda(p, "LipNet parameters")
            keep = []
            for g in (g1, g2):          # [2][...]: forward then reverse, as avsync.h documents
                for n in names:
                    keep.append(torch.stack([N.f32c(getattr(g, n)), N.f32c(getattr(g, n + "_reverse"))]).contiguous())
            keep += [N.f32c(self.fc.weight), N.f32c(self.fc.bias)]
            h = N.c_void_p()
            N.check(N.lib().avs_bigru_create(self.conv_output_dim, self.hidden_dim, self.vocab_size,
                                             *[N.ptr(t) for t in keep], N.PREC[self.precision],
                                             N.stream_ptr(), N.ctypes.byref(h)), "bigru_create")
            cached = (key, N.Handle(h, N.lib().avs_bigru_destroy, keep))
            self._native["bigru"] = cached
        return cached[1]

    # ------------------------------------------------------------------ kernels
    def _check_frames(self, x: torch.Tensor) -> torch.Tensor:
        N.require_cuda(x, "frames")
        if x.dim() != 5 or tuple(x.shape[1:]) != (1, 75, 50, 100):
            # same failure class as the reference's conv1/view on a wrong shape (model.py:22,52)
            raise RuntimeError(f"expected frames of shape (B, 1, 75, 50, 100), got {tuple(x.shape)}")
        if x.dtype == torch.uint8:         # the 8-bit pixels the reference divides by 255 (dataset.py:226-231)
            return x.detach().contiguous()
        return N.f32c(x)

    def stcnn(self, x: torch.Tensor, want_vstats: bool = False, debug: bool = False):
        """Conv half of ``forward`` (model.py:67-82): [B,1,75,50,100] -> emb [B,75,6912]
        (and, optionally, the time-pooled statistics of misalignment_detection_train.py:165).
        ``x`` may also be the uint8 pixels (same shape) the reference's f32 frames are made from
        (``float32(u8 / 255.0)``): same bits out, a quarter of the bytes in."""
        if self.training:
            raise RuntimeError("the B200 LipNet implements eval-mode forward only; call .eval()")
        x = self._check_frames(x)
        B = x.shape[0]
        net = self._stcnn()
        L = N.lib()
        emb = torch.empty((B, 75, self.conv_output_dim), dtype=torch.float32, device=x.device)
        vst = torch.empty((B, 2 * self.conv_output_dim), dtype=torch.float32, device=x.device) if want_vstats else None
        ws = N.workspace(L.avs_stcnn_workspace_bytes(net.h, B), x.device)
        if debug:
            if x.dtype == torch.uint8:
                raise RuntimeError("debug=True takes f32 frames")
            p1 = torch.empty((B, 32, 75, 25, 50), dtype=torch.float32, device=x.device)
            p2 = torch.empty((B, 64, 75, 12, 25), dtype=torch.float32, device=x.device)
            N.check(L.avs_stcnn_forward_debug(net.h, N.ptr(x), B, N.ptr(emb), N.ptr(vst), N.ptr(p1), N.ptr(p2),
                                              N.ptr(ws), ws.numel(), N.stream_ptr()), "stcnn_forward_debug")
            return emb, vst, p1, p2
        if x.dtype == torch.uint8:
            N.check(L.avs_stcnn_forward_u8(net.h, N.ptr(x), B, N.ptr(emb), N.ptr(vst), N.ptr(ws), ws.numel(),
                                           N.stream_ptr()), "stcnn_forward_u8")
            return (emb, vst) if want_vstats else emb
        N.check(L.avs_stcnn_forward(net.h, N.ptr(x), B, N.ptr(emb), N.ptr(vst), N.ptr(ws), ws.numel(),
                                    N.stream_ptr()), "stcnn_forward")
        return (emb, vst) if want_vstats else emb

    def gru_head(self, emb: torch.Tensor) -> torch.Tensor:
        """gru1 -> gru2 -> fc -> log_softmax (model.py:84-95): [B,T,6912] -> [B,T,vocab]."""
        if self.training:
            raise RuntimeError("the B200 LipNet implements eval-mode forward only; call .eval()")
        N.require_cuda(emb, "emb")
        emb = N.f32c(emb)
        B, T, _ = emb.shape
        head = self._bigru()
        L = N.lib()
        out = torch.empty((B, T, self.vocab_size), dtype=torch.float32, device=emb.device)
        ws = N.workspace(L.avs_bigru_workspace_bytes(head.h, B, T), emb.device)
        N.check(L.avs_bigru_forward(head.h, N.ptr(emb), B, T, N.ptr(out), N.ptr(ws), ws.numel(), N.stream_ptr()),
                "bigru_forward")
        return out

    def _head_params(self):
        names = ["weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"]
        return ([getattr(g, n + s) for g in (self.gru1, self.gru2) for n in names for s in ("", "_reverse")]
                + [self.fc.weight, self.fc.bias])

    def gru_head_train(self, emb: torch.Tensor, dropout: float = 0.0) -> torch.Tensor:
        """gru1 -> dropout -> gru2 -> dropout -> fc -> log_softmax (model.py:84-95) with gradients: [B,T,6912] -> log-probs
        [B,T,vocab] with a ``grad_fn`` whose backward (K3b) fills the ``.grad`` of ``gru1.*``, ``gru2.*`` and ``fc.*``.
        The STCNN is frozen: ``emb`` must not require grad (take it from ``stcnn`` under ``torch.no_grad()``).  Works
        whatever ``self.training`` is.  ``dropout`` is the reference's ``dropout_gru1`` / ``dropout_gru2`` rate; the keep
        masks are drawn with torch's RNG.  With ``dropout=0`` the log-probs equal ``gru_head``'s bit for bit."""
        if emb.requires_grad:
            raise ValueError("emb requires grad, but the STCNN backward is not implemented: pass a detached embedding")
        if not 0.0 <= dropout < 1.0:
            raise ValueError(f"dropout must be in [0, 1), got {dropout}")
        N.require_cuda(emb, "emb")
        if emb.dim() != 3 or emb.shape[2] != self.conv_output_dim:
            raise ValueError(f"emb must be [B, T, {self.conv_output_dim}], got {tuple(emb.shape)}")
        N.device_check()
        params = self._head_params()
        for p in params:
            N.require_cuda(p, "LipNet parameters")
        B, T, _ = emb.shape
        masks = (None, None)
        if dropout > 0.0:
            shape = (B, T, 2 * self.hidden_dim)
            masks = tuple(torch.empty(shape, dtype=torch.uint8, device=emb.device).bernoulli_(1.0 - dropout)
                          for _ in range(2))
        stacked = [torch.stack([params[i], params[i + 1]]) for i in range(0, 16, 2)]   # [2][...]: forward, reverse
        return _HeadTrain.apply(self, N.f32c(emb), masks, float(dropout), *stacked, params[16], params[17])

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """(B, 1, T, H, W) float32 -> (B, T, vocab) log-probabilities (model.py:57-97)."""
        with torch.no_grad():
            return self.gru_head(self.stcnn(x))


class _HeadTrain(torch.autograd.Function):
    """The head's training forward and backward over the 10 parameter tensors in avsync.h's stacked layout."""

    @staticmethod
    def forward(ctx, net, emb, masks, p, *params):
        B, T, _ = emb.shape
        L = N.lib()
        w = [N.f32c(t) for t in params]
        dims = (net.conv_output_dim, net.hidden_dim, net.vocab_size, N.PREC[net.precision])
        out = torch.empty((B, T, net.vocab_size), dtype=torch.float32, device=emb.device)
        ws = N.workspace(L.avs_bigru_train_workspace_bytes(*dims, B, T), emb.device)
        N.check(L.avs_bigru_train_forward(*dims, *[N.ptr(t) for t in w], N.ptr(emb), B, T, N.ptr(masks[0]),
                                          N.ptr(masks[1]), p, N.ptr(out), N.ptr(ws), ws.numel(), N.stream_ptr()),
                "bigru_train_forward")
        ctx.dims, ctx.p, ctx.masks, ctx.ws, ctx.w, ctx.emb = dims, p, masks, ws, w, emb
        ctx.shapes = [t.shape for t in params]
        return out

    @staticmethod
    def backward(ctx, grad_out):
        B, T, _ = ctx.emb.shape
        g = grad_out.to(torch.float32).contiguous()
        grads = [torch.empty(s, dtype=torch.float32, device=g.device) for s in ctx.shapes]
        N.check(N.lib().avs_bigru_train_backward(*ctx.dims, *[N.ptr(t) for t in ctx.w], N.ptr(ctx.emb), B, T,
                                                 N.ptr(ctx.masks[0]), N.ptr(ctx.masks[1]), ctx.p, N.ptr(g),
                                                 *[N.ptr(t) for t in grads], N.ptr(ctx.ws), ctx.ws.numel(),
                                                 N.stream_ptr()), "bigru_train_backward")
        return (None, None, None, None, *grads)
