"""Argument checks and workspace sizes of the CTC loss (avs_ctc_loss) and the head's training entry points
(avs_bigru_train_*), through ctypes: every check runs before any CUDA call, so no device is needed."""
import ctypes
import os

import pytest

FAKE = ctypes.c_void_p(256)     # never dereferenced: every call below fails its argument checks first


@pytest.fixture(scope="module")
def native():
    import avsync_b200
    N = avsync_b200._native
    if not os.path.isfile(N.LIB_PATH):
        N.build()
    return N


def test_ctc_loss_rejects_bad_arguments_without_a_device(native):
    L = native.lib()

    def call(n_clips=4, n_steps=75, vocab=39, blank=0, stride=40, ws_bytes=1 << 40, out=FAKE, grad=FAKE, scale=FAKE,
             ws=FAKE, targets=FAKE):
        rc = L.avs_ctc_loss(FAKE, n_clips, n_steps, vocab, blank, None, targets, stride, FAKE, scale, 0, out, grad, ws,
                            ws_bytes, None)
        return rc, L.avs_last_error_string().decode()

    for kw, text in (({"n_steps": 0}, "n_steps must be in [1, 1024]"), ({"n_steps": 1025}, "n_steps must be in [1, 1024]"),
                     ({"vocab": 1}, "vocab must be in [2, 64]"), ({"vocab": 65}, "vocab must be in [2, 64]"),
                     ({"blank": -1}, "blank must be in [0, vocab)"), ({"blank": 39}, "blank must be in [0, vocab)"),
                     ({"stride": -1}, "target_stride must be in [0, 512]"),
                     ({"stride": 513}, "target_stride must be in [0, 512]"),
                     ({"n_clips": -1}, "n_clips"), ({"out": None}, "null argument"),
                     ({"scale": None}, "null argument"), ({"targets": None}, "null argument")):
        rc, msg = call(**kw)
        assert rc == -1 and text in msg, (kw, msg)
    rc, msg = call(n_steps=1024, stride=512, ws_bytes=1 << 20)
    assert rc == -4 and "workspace too small" in msg
    rc, msg = call(ws=None)
    assert rc == -4 and "workspace too small" in msg
    assert call(n_clips=0, out=None, ws=None)[0] == 0     # an empty batch needs no buffers and launches nothing


def test_ctc_loss_workspace_bytes(native):
    L = native.lib()
    per_clip = L.avs_ctc_loss_workspace_bytes(1, 75, 40)
    assert per_clip >= 75 * 81 * 8 and per_clip % 256 == 0
    assert L.avs_ctc_loss_workspace_bytes(64, 75, 40) == 64 * per_clip
    assert L.avs_ctc_loss_workspace_bytes(1, 1024, 512) >= 1024 * 1025 * 8
    assert L.avs_ctc_loss_workspace_bytes(0, 75, 40) == 0
    for args in ((-1, 75, 40), (1, 0, 40), (1, 1025, 40), (1, 75, -1), (1, 1024, 513)):
        assert L.avs_ctc_loss_workspace_bytes(*args) == 0


def _train_call(L, fn, in_dim=6912, hidden=256, vocab=39, prec=2, n_clips=4, n_steps=75, masks=(None, None), p=0.0,
                ws_bytes=1 << 40, ws=FAKE, null_param=None):
    params = [FAKE] * 11
    if null_param is not None:
        params[null_param] = None
    head = [in_dim, hidden, vocab, prec] + params + [n_clips, n_steps, masks[0], masks[1], ctypes.c_float(p)]
    if fn == "forward":
        rc = L.avs_bigru_train_forward(*head, FAKE, ws, ws_bytes, None)
    else:
        rc = L.avs_bigru_train_backward(*head, FAKE, *([FAKE] * 10), ws, ws_bytes, None)
    return rc, L.avs_last_error_string().decode()


@pytest.mark.parametrize("fn", ["forward", "backward"])
def test_train_rejects_bad_arguments_without_a_device(native, fn):
    L = native.lib()
    for kw, text in (({"hidden": 0}, "hidden must be"), ({"hidden": 48}, "hidden must be"), ({"hidden": 1056}, "hidden must be"),
                     ({"in_dim": 0}, "in_dim"), ({"in_dim": 12}, "in_dim"), ({"in_dim": 40}, "in_dim % 32"),
                     ({"vocab": 0}, "vocab"), ({"vocab": 4097}, "vocab"), ({"prec": 3}, "precision"), ({"prec": -1}, "precision"),
                     ({"n_clips": -1}, "n_clips"), ({"n_steps": 0}, "n_steps"),
                     ({"n_clips": 100000, "n_steps": 75}, "2^31"),
                     ({"masks": (FAKE, None)}, "both keep masks"), ({"masks": (None, FAKE)}, "both keep masks"),
                     ({"masks": (FAKE, FAKE), "p": 1.0}, "dropout_p"), ({"masks": (FAKE, FAKE), "p": -0.1}, "dropout_p"),
                     ({"null_param": 0}, "null argument"), ({"null_param": 10}, "null argument")):
        rc, msg = _train_call(L, fn, **kw)
        assert rc == -1 and text in msg, (kw, msg)
    rc, msg = _train_call(L, fn, ws_bytes=1 << 20)
    assert rc == -4 and "workspace too small" in msg
    rc, msg = _train_call(L, fn, in_dim=40, prec=0, ws_bytes=1 << 10)   # fp32 projections take in_dim % 8 == 0
    assert rc == -4, msg
    if fn == "forward":
        assert _train_call(L, fn, n_clips=0, ws=None)[0] == 0


# sgemm_nt's tiled kernel has gridDim.y = ceil(rows / 128) and runs over all n_clips * n_steps rows (fc, the fp32
# projections, the backward's dh2 and dx); transpose_pad_kernel has gridDim.y = ceil(cols / 32) and the backward transposes
# the embedding (in_dim columns).  gridDim.y <= 65535.
MAX_ROWS = 65535 * 128       # 8 388 480
MAX_IN_DIM = 65535 * 32      # 2 097 120
PAST_LIMITS = [  # (in_dim, hidden, vocab, prec, n_clips, n_steps), each just past one limit; message text
    ((8, 32, 1, 0, MAX_ROWS + 1, 1), "n_clips * n_steps must be <= 8388480"),
    ((8, 32, 1, 0, 1, MAX_ROWS + 1), "n_clips * n_steps must be <= 8388480"),
    ((32, 32, 1, 2, 2796161, 3), "n_clips * n_steps must be <= 8388480"),   # 8 388 483 rows
    ((MAX_IN_DIM + 8, 32, 1, 0, 1, 1), "in_dim must be <= 2097120"),
    ((2097152, 32, 1, 2, 1, 1), "in_dim must be <= 2097120"),
]
INSIDE_LIMITS = [(8, 32, 1, 0, MAX_ROWS, 1), (8, 32, 1, 0, 1, MAX_ROWS), (32, 32, 1, 2, 2796160, 3),
                 (MAX_IN_DIM, 32, 1, 0, 1, 1), (MAX_IN_DIM, 32, 1, 2, 1, 1)]


@pytest.mark.parametrize("fn", ["forward", "backward"])
def test_train_rejects_shapes_past_the_launch_limits_without_a_device(native, fn):
    """Both shapes pass the older 2^31 bound on align8(rows) * width, but would fail a launch after kernels were queued."""
    L = native.lib()
    for (in_dim, H, V, prec, B, T), text in PAST_LIMITS:
        assert L.avs_bigru_train_workspace_bytes(in_dim, H, V, prec, B, T) == 0, (in_dim, B, T)
        rc, msg = _train_call(L, fn, in_dim=in_dim, hidden=H, vocab=V, prec=prec, n_clips=B, n_steps=T)
        assert rc == -1 and text in msg, (in_dim, B, T, msg)


def test_train_workspace_bytes_at_the_launch_limits(native):
    """Just inside each limit the shape is accepted (no call: it would launch kernels on the fake pointers)."""
    L = native.lib()
    for args in INSIDE_LIMITS:
        assert L.avs_bigru_train_workspace_bytes(*args) > 0, args


def test_train_workspace_bytes(native):
    L = native.lib()
    small = L.avs_bigru_train_workspace_bytes(6912, 256, 39, 2, 1, 75)
    big = L.avs_bigru_train_workspace_bytes(6912, 256, 39, 2, 64, 75)
    fp32 = L.avs_bigru_train_workspace_bytes(6912, 256, 39, 0, 64, 75)
    assert 0 < small < big and fp32 < big and big % 256 == 0
    # the transposed embedding alone (6912 x B*T floats) is part of it
    assert big >= 6912 * 4800 * 4
    for args in ((6912, 256, 39, 2, 0, 75), (6912, 48, 39, 2, 1, 75), (6912, 256, 0, 2, 1, 75), (6912, 256, 39, 3, 1, 75),
                 (6912, 256, 39, 2, 1, 0), (40, 256, 39, 2, 1, 75), (6912, 256, 39, 2, 100000, 75)):
        assert L.avs_bigru_train_workspace_bytes(*args) == 0
