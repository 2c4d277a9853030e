"""K3b, the Bi-GRU head's training backward (csrc/gru_train.cu), against float64 torch autograd at the shapes,
precisions, keep masks and upstream gradients avs_bigru_train_backward accepts.

LipNet.gru_head_train only reaches in_dim 6912, vocab 39 and CTC gradients, so the cases here drive
avs_bigru_train_forward / _backward through ctypes (TrainHead), with any in_dim, vocab, keep masks and dL/dlogp.  The
reference is oracle/ctc_loss_ref.head_reference in float64 on the GPU with the same masks, back-propagated from the same
upstream gradient; the training forward's log-probs are compared with its log-probs too.

Every case names in its id the kernels it launches: the forward's recurrence and projections (gru.cu), and for each
sgemm_nt product of the backward (dW_fc, dh2, dW_ih of layer 1 and 2, dW_hh, dx, in that order) whether it runs on the
one-thread-per-output kernel (s) or the tiled one (t).  A test without a device restates that dispatch from the source
(pinned with source_has) and checks that the cases reach every kernel, lane pass, padding and clip-group boundary.

Errors are max |g - g64| / max |g64| over each gate block (r, z, n) of each direction of a GRU parameter and over the
whole tensor for fc.*, so that a wrong block cannot hide under a larger one.  Tolerances sit at about twice the largest
error measured on an NVIDIA B200 (1000 W power limit) per precision and saturation group; report() prints each case's.
The exact properties of the code (clip isolation, scaling by powers of two, masks of all ones or all zeros, vocab 1,
bf16 against bf16x3) are checked bit for bit with torch.equal.  The _HeadTrain plumbing of LipNet.gru_head_train is
checked under losses other than CTC, repeated backwards and interleaved graphs."""
import os

import numpy as np
import pytest
import torch

from oracle import ctc_loss_ref as R
from oracle import lipnet_ref

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    "alignment-between-speech-and-visual-mouth-movements_b200", "csrc")

STACKED = [(g, n) for g in ("gru1", "gru2") for n in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")]
NAMES = [f"{g}.{n}{s}" for g, n in STACKED for s in ("", "_reverse")] + ["fc.weight", "fc.bias"]

# Largest errors measured on an NVIDIA B200 (1000 W power limit) over the cases of this file, see DESIGN §4.3:
#   gradients, max |g - g64| / max |g64| per gate block: fp32 4.1e-6, saturating 2.9e-6; bf16x3 4.1e-5, saturating
#   6.0e-5 (the backward recomputes the gates in fp32 from the tcgen05 forward's projections and outputs);
#   log-probs with keep masks, max |lp - lp64|: fp32 1.2e-6, saturating 2.0e-6; bf16x3 7.5e-5 (p = 0.9 scales layer
#   2's and fc's inputs by 10, at in_dim 6912), saturating 3.5e-5.
GRAD_TOL = {("fp32", False): 8e-6, ("fp32", True): 6e-6, ("bf16x3", False): 8e-5, ("bf16x3", True): 1.2e-4}
LP_TOL = {("fp32", False): 2.5e-6, ("fp32", True): 4e-6, ("bf16x3", False): 1.5e-4, ("bf16x3", True): 7e-5}


def source_has(name, *fragments):
    """The dispatch rules restated below are pinned to the CUDA source: if one of these lines changes, the
    restatement (and with it the coverage the cases are checked for) must be revisited."""
    src = " ".join(open(os.path.join(CSRC, name)).read().split())
    for f in fragments:
        assert " ".join(f.split()) in src, f"{name} no longer contains `{f}`: update the dispatch rule of this test"


@pytest.fixture(scope="module")
def A():
    import avsync_b200
    avsync_b200._native.device_check()
    return avsync_b200


# ---------------------------------------------------------------------------------------------------- dispatch
BPTT_CLIPS = 2            # gru_train.cu kBpttClips: clips per CTA of gru_bptt_kernel
SKINNY_OUTPUTS = 16384    # sgemm.cu kSkinnyOutputs: M * N up to which sgemm_nt runs one thread per output
FWD_GROUP = {"generic": 4, "cluster_fp32": 16, "cluster_umma": 32}   # gru.cu kGruClips, kCluClips; gru_umma.cu 16 x 2
FWD_B_BOUNDARIES = {"generic": {1, 4, 5}, "cluster_fp32": {1, 16, 17, 32, 33}, "cluster_umma": {1, 16, 17, 32, 33}}
GEMMS = ("dW_fc", "dh2", "dW_ih1", "dW_ih2", "dW_hh", "dx")


def recurrence(H, prec):
    """The forward's recurrence kernel (gru.cu head_forward; the training forward packs w_hh for H = 256 only)."""
    if H == 256:
        return "cluster_fp32" if prec == "fp32" else "cluster_umma"
    return "generic"


def gemm_kernels(H, B, T, V, in_dim):
    """Each sgemm_nt product of avs_bigru_train_backward as (M, N) -> 's' (skinny kernel) or 't' (tiled)."""
    BT = B * T
    shapes = {"dW_fc": (V, 2 * H), "dh2": (BT, 2 * H), "dW_ih1": (6 * H, in_dim), "dW_ih2": (6 * H, 2 * H),
              "dW_hh": (3 * H, H), "dx": (BT, 2 * H)}
    return {k: "s" if m * n <= SKINNY_OUTPUTS else "t" for k, (m, n) in shapes.items()}


# (hidden, precision, B, T, vocab, in_dim, dropout p, upstream gradient, saturating)
#   upstream gradient: "dense" normal (both signs, non-zero row sums), "zero" the same with whole rows and a clip of
#   zeros, "ctc" the CTC gradient of the kernel's log-probs (rows summing to -1 inside input_len, 0 after)
CASES = [
    (32, "fp32", 5, 75, 39, 40, 0.0, "dense", False),
    (32, "fp32", 1, 75, 100, 40, 0.3, "zero", False),
    (32, "bf16x3", 4, 2, 33, 256, 0.9, "dense", False),
    (32, "bf16x3", 1, 1, 8, 256, 0.0, "dense", False),
    (128, "fp32", 4, 1, 4096, 256, 0.0, "dense", False),
    (128, "bf16x3", 5, 75, 39, 6912, 0.3, "ctc", False),
    (128, "fp32", 1, 200, 8, 256, 0.0, "dense", False),
    (128, "bf16x3", 2, 200, 1, 256, 0.3, "dense", False),
    (512, "fp32", 5, 2, 100, 256, 0.9, "zero", False),
    (512, "bf16x3", 4, 75, 39, 6912, 0.0, "ctc", False),
    (1024, "fp32", 1, 75, 33, 256, 0.3, "dense", False),
    (1024, "bf16x3", 5, 1, 4096, 256, 0.0, "dense", False),
    (128, "fp32", 5, 75, 39, 256, 0.0, "dense", True),
    (128, "bf16x3", 4, 75, 100, 256, 0.3, "dense", True),
    (256, "fp32", 16, 75, 39, 256, 0.0, "dense", False),
    (256, "fp32", 17, 2, 100, 256, 0.3, "zero", False),
    (256, "fp32", 32, 1, 8, 256, 0.9, "dense", False),
    (256, "fp32", 33, 75, 4096, 256, 0.0, "dense", False),
    (256, "fp32", 1, 200, 33, 6912, 0.3, "ctc", False),
    (256, "fp32", 17, 75, 39, 256, 0.0, "dense", True),
    (256, "bf16x3", 16, 2, 39, 256, 0.3, "dense", False),
    (256, "bf16x3", 17, 75, 1, 256, 0.0, "zero", False),
    (256, "bf16x3", 32, 75, 100, 6912, 0.9, "ctc", False),
    (256, "bf16x3", 33, 1, 33, 256, 0.3, "dense", False),
    (256, "bf16x3", 1, 200, 4096, 256, 0.0, "dense", False),
    (256, "bf16x3", 17, 75, 39, 256, 0.3, "dense", True),
]


def case_id(c):
    H, prec, B, T, V, in_dim, p, gk, sat = c
    proj = "sgemm" if prec == "fp32" else "tcgen05"
    nt = "".join(gemm_kernels(H, B, T, V, in_dim)[k] for k in GEMMS)
    return (f"{recurrence(H, prec)}+{proj}+bptt-{prec}-H{H}-B{B}-T{T}-V{V}-in{in_dim}-p{p}-{gk}"
            + ("-saturating" if sat else "") + f"-nt{nt}")


def test_k3b_cases_reach_every_kernel_and_boundary():
    source_has("gru_train.cu", "constexpr int kBpttClips = 2;",
               "gru_bptt_kernel<kBpttClips><<<dim3(cdiv(B, kBpttClips), 2), H, smem, st>>>(",
               "log_softmax_backward_kernel<<<cdiv(BT, 4), 128, 0, st>>>(grad_logp, w.logp, BT, V, Vp, w.dz);",
               "for (int v = lane; v < Vp; v += 32)",
               "sgemm_nt(w.tr_a, BTp, w.tr_b, BTp, nullptr, d_fc_w, 2 * H, V, 2 * H, BTp, st)",
               "sgemm_nt(w.dz, Vp, w.fcw_t, Vp, nullptr, w.dh, 2 * H, BT, 2 * H, Vp, st)",
               "sgemm_nt(w.tr_a, BTp, w.tr_b, BTp, nullptr, d_wih[l], ins[l], 6 * H, ins[l], BTp, st)",
               "BTp, nullptr, d_whh[l] + static_cast<size_t>(dir) * 3 * H * H, H, 3 * H, H, BTp, st)",
               "sgemm_nt(w.dgi, 6 * H, w.wih2_t, 6 * H, nullptr, w.dh, 2 * H, BT, 2 * H, 6 * H, st)",
               "for (int l = 0; l < 2 && precision != AVS_PREC_FP32; ++l) {", "if (H == 256) {")
    source_has("sgemm.cu", "constexpr int kSkinnyOutputs = 16384;",
               "if (static_cast<long long>(M) * N <= kSkinnyOutputs) {")
    source_has("gru.cu", "constexpr int kGruClips = 4;", "kCluClips = 16,", "kCluH = 256,",
               "if (g->w_hh_packed[l] != nullptr && !force_fma) {", "} else if (H == kCluH) {")
    source_has("gru_umma.cu", "constexpr int kGrpClips = 16, kGroups = 2;")
    for prec in ("fp32", "bf16x3"):
        assert {c[0] for c in CASES if c[1] == prec} == {32, 128, 256, 512, 1024}, prec
    for kern, need in FWD_B_BOUNDARIES.items():
        cases = [c for c in CASES if recurrence(c[0], c[1]) == kern]
        assert {c[2] for c in cases} >= need, kern
        assert {c[2] % FWD_GROUP[kern] for c in cases} >= {0, 1}, kern                 # full and ragged last group
        assert {c[2] % BPTT_CLIPS for c in cases} == {0, 1}, kern                      # full and half-empty BPTT pair
        assert {c[3] for c in cases} >= {1, 2, 75, 200}, kern
        assert any(c[8] for c in cases), kern                                          # a saturating case
    # vocab: no padding (8, 4096), padding to align8 (1, 33, 39, 100); one, two, four and 128 lane passes
    assert {c[4] for c in CASES} == {1, 8, 33, 39, 100, 4096}
    assert {-(-((c[4] + 7) // 8 * 8) // 32) for c in CASES} >= {1, 2, 4, 128}
    assert {c[5] for c in CASES} == {40, 256, 6912} and all(c[1] == "fp32" for c in CASES if c[5] % 32)
    assert {c[6] for c in CASES} == {0.0, 0.3, 0.9} and {c[7] for c in CASES} == {"dense", "zero", "ctc"}
    for k in GEMMS:
        assert {gemm_kernels(*[c[i] for i in (0, 2, 3, 4, 5)])[k] for c in CASES} == {"s", "t"}, k
    for c in CASES:
        assert c[0] < 1024 or c[2] <= 5, "keep hidden-1024 cases small in B"
        assert c[3] < 200 or c[2] <= 2, "keep T = 200 cases small in B"
        assert c[7] != "ctc" or (c[4] > 1 and c[3] >= 75), "CTC needs labels besides the blank and frames for them"


# ---------------------------------------------------------------------------------------------------- harness
def gru_params(hidden, in_dim, vocab, seed, saturating=False):
    """A LipNet head's gru1 / gru2 / fc entries under PyTorch's default initialisation; `saturating` multiplies the
    input and recurrent weights by 4, so that the gates' arguments reach the flat ends of sigmoid and tanh."""
    torch.manual_seed(seed)
    p = {}
    for name, mod in (("gru1", torch.nn.GRU(in_dim, hidden, batch_first=True, bidirectional=True)),
                      ("gru2", torch.nn.GRU(2 * hidden, hidden, batch_first=True, bidirectional=True)),
                      ("fc", torch.nn.Linear(2 * hidden, vocab))):
        for k, v in mod.state_dict().items():
            v = v.detach().clone()
            if saturating and k.startswith("weight_"):
                v *= 4.0
            p[f"{name}.{k}"] = v
    return p


class TrainHead:
    """avs_bigru_train_forward / _backward over a parameter dict, in avsync.h's stacked layout ([2][...]: forward,
    reverse).  backward() uses the workspace of the last forward(), as the ABI requires."""

    def __init__(self, N, params, in_dim, hidden, vocab, precision):
        self.N, self.dims = N, (in_dim, hidden, vocab, N.PREC[precision])
        self.w = [torch.stack([params[f"{g}.{n}"], params[f"{g}.{n}_reverse"]]).float().contiguous().cuda()
                  for g, n in STACKED]
        self.w += [params["fc.weight"].float().contiguous().cuda(), params["fc.bias"].float().contiguous().cuda()]

    def forward(self, emb, masks=(None, None), p=0.0):
        N, L = self.N, self.N.lib()
        B, T, _ = emb.shape
        self.ws = N.workspace(L.avs_bigru_train_workspace_bytes(*self.dims, B, T), "cuda")
        self.args = (emb, masks, p)
        out = torch.full((B, T, self.dims[2]), float("nan"), device="cuda")
        N.check(L.avs_bigru_train_forward(*self.dims, *[N.ptr(t) for t in self.w], N.ptr(emb), B, T, N.ptr(masks[0]),
                                          N.ptr(masks[1]), p, N.ptr(out), N.ptr(self.ws), self.ws.numel(),
                                          N.stream_ptr()), "bigru_train_forward")
        return out

    def backward(self, g):
        N, L = self.N, self.N.lib()
        emb, masks, p = self.args
        B, T, _ = emb.shape
        grads = [torch.full_like(t, float("nan")) for t in self.w]    # an entry the kernels skip stays NaN
        N.check(L.avs_bigru_train_backward(*self.dims, *[N.ptr(t) for t in self.w], N.ptr(emb), B, T, N.ptr(masks[0]),
                                           N.ptr(masks[1]), p, N.ptr(g.contiguous()), *[N.ptr(t) for t in grads],
                                           N.ptr(self.ws), self.ws.numel(), N.stream_ptr()), "bigru_train_backward")
        out = {}
        for (g_, n), t in zip(STACKED, grads):
            out[f"{g_}.{n}"], out[f"{g_}.{n}_reverse"] = t[0], t[1]
        out["fc.weight"], out["fc.bias"] = grads[8], grads[9]
        return out


def reference(params, emb, masks, p, g):
    """float64 log-probs and the 18 gradients of <lp, g> (autograd through nn.GRU, Linear, log_softmax)."""
    lp64, mods = R.head_reference(params, emb, masks, p)
    lp64.backward(gradient=g.double())
    return lp64.detach(), {f"{name}.{k}": q.grad for name, m in zip(("gru1", "gru2", "fc"), mods)
                           for k, q in m.named_parameters()}


def keep_masks(p, B, T, H, seed):
    if p == 0:
        return (None, None)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return tuple(torch.empty((B, T, 2 * H), dtype=torch.uint8, device="cuda").bernoulli_(1.0 - p, generator=gen)
                 for _ in range(2))


def upstream(kind, lp, seed):
    """dL/dlogp, float32 [B, T, V] on the device."""
    B, T, V = lp.shape
    rng = np.random.default_rng(seed)
    if kind == "ctc":
        lens = rng.integers(1, T // 3 + 1, B)
        targets = rng.integers(1, V, (B, int(lens.max()))).astype(np.int32)
        il = np.full(B, T)
        il[: B // 2] = T - rng.integers(0, T // 4 + 1, B // 2)
        _, g = R.loss_grad_batch(lp.cpu().numpy(), targets, lens, il)
        assert np.isfinite(g).all()
    else:
        g = rng.normal(size=(B, T, V))
        if kind == "zero":
            g[rng.random((B, T)) < 0.3] = 0.0
            g[:, T - T // 4:] = 0.0
            if B > 1:
                g[B // 2] = 0.0
    return torch.from_numpy(g.astype(np.float32)).cuda()


def block_errors(got, want, H):
    """max |g - g64| / max |g64| per gate block (r, z, n) of each GRU parameter (each direction is its own name) and per
    fc tensor; a block whose reference is exactly zero must be exactly zero."""
    errs = {}
    for n in NAMES:
        a, b = got[n].double(), want[n]
        blocks = [("", slice(None))] if n.startswith("fc.") else [(f"[{gate}]", slice(i * H, (i + 1) * H))
                                                                   for i, gate in enumerate("rzn")]
        for tag, sl in blocks:
            ref, d = float(b[sl].abs().max()), float((a[sl] - b[sl]).abs().max())
            errs[n + tag] = d / ref if ref > 0 else (0.0 if d == 0 else float("inf"))
    return errs


def report(name, errs, lp_err):
    worst = max(errs, key=errs.get)
    print(f"[k3b] {name}: worst gradient block {worst} {errs[worst]:.3e}, max |lp - lp64| {lp_err:.3e}")
    return errs[worst]


def check_vs_f64(name, got, want, lp, lp64, H, group, skip=()):
    for n in NAMES:
        assert torch.isfinite(got[n]).all(), (name, n)
    lp_err = float((lp.double() - lp64).abs().max())
    errs = block_errors(got, want, H)
    worst = report(name, {k: v for k, v in errs.items() if not k.startswith(skip)} or {"-": 0.0}, lp_err)
    assert lp_err <= LP_TOL[group], (name, lp_err)
    assert worst <= GRAD_TOL[group], (name, errs)


def case_seed(H, B, T, V, in_dim, p, sat):
    return (H * 7 + B * 131 + T * 17 + V + in_dim + int(p * 10) * 1000 + (5000 if sat else 0)) % 100003


def rand_emb(B, T, in_dim, seed):
    return (torch.rand((B, T, in_dim), generator=torch.Generator().manual_seed(seed)) * 0.2).cuda()


# ---------------------------------------------------------------------------------------------------- vs float64
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
def test_k3b_gradients_vs_f64(A, case):
    H, prec, B, T, V, in_dim, p, gk, sat = case
    name = case_id(case)
    seed = case_seed(H, B, T, V, in_dim, p, sat)
    params = gru_params(H, in_dim, V, seed, sat)
    emb = rand_emb(B, T, in_dim, seed)
    masks = keep_masks(p, B, T, H, seed)
    head = TrainHead(A._native, params, in_dim, H, V, prec)
    lp = head.forward(emb, masks, p)
    g = upstream(gk, lp, seed)
    got = head.backward(g)
    lp64, want = reference(params, emb, masks, p, g)
    check_vs_f64(name, got, want, lp, lp64, H, (prec, sat))
    if V == 1:   # log_softmax of one logit is 0, and dz = g - exp(0) * g = 0: nothing reaches any parameter
        assert torch.equal(lp, torch.zeros_like(lp)), name
        for n in NAMES:
            assert torch.equal(got[n], torch.zeros_like(got[n])), (name, n)


# ---------------------------------------------------------------------------------------------------- exact properties
# (recurrence kernel, hidden, precision, B): every position of a BPTT pair and of a forward group
ISOLATION = [("generic", 128, "fp32", 5), ("cluster_fp32", 256, "fp32", 17), ("cluster_umma", 256, "bf16x3", 33)]


@pytest.mark.gpu
@pytest.mark.parametrize("kern,H,prec,B", ISOLATION, ids=[c[0] for c in ISOLATION])
def test_clip_isolation_bit_for_bit(A, kern, H, prec, B):
    """A clip x among clips whose grad_logp rows are all zero gets the 18 gradients of x alone, at every position.  The
    forward is batch-independent bit for bit; a zero clip adds ±0 products to the ascending-k fmaf chains of sgemm_nt and
    ±0 rows to the fp64 column sums, and the zero rows that pad B*T to a multiple of 8 add nothing either."""
    assert recurrence(H, prec) == kern
    T, V, in_dim, p = 3, 39, 256, 0.3
    params = gru_params(H, in_dim, V, seed=B)
    head = TrainHead(A._native, params, in_dim, H, V, prec)
    emb_x = rand_emb(1, T, in_dim, seed=1)
    m_x = keep_masks(p, 1, T, H, seed=2)
    lp_x = head.forward(emb_x, m_x, p)
    g_x = upstream("dense", lp_x, seed=3)
    want = head.backward(g_x)
    for i in range(B):
        emb = rand_emb(B, T, in_dim, seed=10 + i)
        masks = keep_masks(p, B, T, H, seed=100 + i)
        emb[i], masks[0][i], masks[1][i] = emb_x[0], m_x[0][0], m_x[1][0]
        lp = head.forward(emb, masks, p)
        assert torch.equal(lp[i], lp_x[0]), (kern, i)
        g = torch.zeros((B, T, V), device="cuda")
        g[i] = g_x[0]
        got = head.backward(g)
        for n in NAMES:
            assert torch.equal(got[n], want[n]), (kern, i, n)


@pytest.mark.gpu
@pytest.mark.parametrize("H,prec", [(128, "fp32"), (256, "bf16x3")])
def test_backward_scales_with_powers_of_two(A, H, prec):
    """backward(2^k g) == 2^k backward(g): every step of the backward is a product, a sum or a chain of fmaf that is
    linear in g, and scaling by 2^k commutes with fp32 and fp64 rounding while nothing is subnormal (non-saturating
    parameters)."""
    B, T, V, in_dim, p = 5, 75, 39, 256, 0.3
    params = gru_params(H, in_dim, V, seed=7)
    head = TrainHead(A._native, params, in_dim, H, V, prec)
    lp = head.forward(rand_emb(B, T, in_dim, seed=7), keep_masks(p, B, T, H, seed=7), p)
    g = upstream("dense", lp, seed=7)
    base = head.backward(g)
    for k in (-3, 5):
        got = head.backward(g * 2.0 ** k)
        for n in NAMES:
            assert torch.equal(got[n], base[n] * 2.0 ** k), (k, n)


@pytest.mark.gpu
@pytest.mark.parametrize("H,prec", [(128, "fp32"), (256, "bf16x3")])
def test_masks_of_all_ones_at_p0_are_the_mask_free_call(A, H, prec):
    """keep_scale = 1 / (1 - 0) = 1, and x * 1 * 1 is x: the log-probs and gradients are those of the call without
    masks."""
    B, T, V, in_dim = 5, 75, 39, 256
    params = gru_params(H, in_dim, V, seed=8)
    head = TrainHead(A._native, params, in_dim, H, V, prec)
    emb = rand_emb(B, T, in_dim, seed=8)
    lp0 = head.forward(emb)
    g = upstream("dense", lp0, seed=8)
    want = head.backward(g)
    ones = tuple(torch.ones((B, T, 2 * H), dtype=torch.uint8, device="cuda") for _ in range(2))
    lp1 = head.forward(emb, ones, 0.0)
    got = head.backward(g)
    assert torch.equal(lp1, lp0)
    for n in NAMES:
        assert torch.equal(got[n], want[n]), n


@pytest.mark.gpu
@pytest.mark.parametrize("which", [1, 2])
@pytest.mark.parametrize("H,prec", [(128, "fp32"), (256, "bf16x3")])
def test_all_zero_keep_mask(A, which, H, prec):
    """Mask 1 all zero: layer 2 sees zeros, so every gru1.* gradient and gru2.weight_ih* are exactly 0.  Mask 2 all
    zero: fc sees zeros, so every GRU gradient and fc.weight are exactly 0.  The rest matches float64."""
    B, T, V, in_dim, p = 5, 75, 39, 256, 0.3
    params = gru_params(H, in_dim, V, seed=9)
    head = TrainHead(A._native, params, in_dim, H, V, prec)
    emb = rand_emb(B, T, in_dim, seed=9)
    masks = list(keep_masks(p, B, T, H, seed=9))
    masks[which - 1] = torch.zeros_like(masks[which - 1])
    lp = head.forward(emb, tuple(masks), p)
    g = upstream("dense", lp, seed=9)
    got = head.backward(g)
    zero = (("gru1.", "gru2.weight_ih") if which == 1 else ("gru1.", "gru2.", "fc.weight"))
    for n in NAMES:
        if n.startswith(zero):
            assert torch.equal(got[n], torch.zeros_like(got[n])), n
    lp64, want = reference(params, emb, tuple(masks), p, g)
    check_vs_f64(f"mask{which}-zero-{prec}-H{H}", got, want, lp, lp64, H, (prec, False), skip=zero)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [128, 256])
def test_bf16_backward_is_the_bf16x3_backward(A, H):
    """precision 'bf16' runs the head exactly as 'bf16x3' does (test_k3_bf16_head_is_the_bf16x3_head), and the backward
    does not depend on the precision: same bits."""
    B, T, V, in_dim, p = 17, 75, 39, 256, 0.3
    params = gru_params(H, in_dim, V, seed=10)
    emb = rand_emb(B, T, in_dim, seed=10)
    masks = keep_masks(p, B, T, H, seed=10)
    out = []
    for prec in ("bf16", "bf16x3"):
        head = TrainHead(A._native, params, in_dim, H, V, prec)
        lp = head.forward(emb, masks, p)
        out.append((lp, head.backward(upstream("dense", lp, seed=10))))
    assert torch.equal(out[0][0], out[1][0])
    for n in NAMES:
        assert torch.equal(out[0][1][n], out[1][1][n]), n


# ---------------------------------------------------------------------------------------------------- _HeadTrain
PLUMB_H = 32


@pytest.fixture(scope="module")
def lipnet(A):
    sd = lipnet_ref.init_lipnet_state(39, PLUMB_H, seed=12)
    net = A.LipNet(39, hidden_dim=PLUMB_H, precision="fp32")
    net.load_state_dict(sd)
    return net.cuda(), {k: v for k, v in sd.items() if k.split(".")[0] in ("gru1", "gru2", "fc")}


def net_grads(net):
    return {n: q.grad.detach().clone() for n, q in net.named_parameters() if n in NAMES and q.grad is not None}


def clear_grads(net):
    for q in net.parameters():
        q.grad = None


LOSSES = {
    "sum": lambda lp, w: lp.sum(),                                  # grad_out has stride 0
    "strided": lambda lp, w: (lp[:, ::2] * w[:, ::2]).sum(),        # grad_out is zero on every other frame
    "weighted": lambda lp, w: (lp * w).sum(),
}


@pytest.mark.gpu
@pytest.mark.parametrize("loss", list(LOSSES))
def test_head_train_losses_other_than_ctc_vs_f64(A, lipnet, loss):
    net, sd = lipnet
    B, T = 3, 20
    emb = rand_emb(B, T, 6912, seed=13) * 0.25
    w = torch.randn((B, T, 39), generator=torch.Generator().manual_seed(13)).cuda()
    clear_grads(net)
    lp = net.gru_head_train(emb)
    LOSSES[loss](lp, w).backward()
    got = net_grads(net)
    assert sorted(got) == sorted(NAMES)
    lp64, mods = R.head_reference(sd, emb)
    LOSSES[loss](lp64, w.double()).backward()
    want = {f"{name}.{k}": q.grad for name, m in zip(("gru1", "gru2", "fc"), mods) for k, q in m.named_parameters()}
    check_vs_f64(f"_HeadTrain-{loss}", got, want, lp.detach(), lp64.detach(), PLUMB_H, ("fp32", False))


@pytest.mark.gpu
def test_head_train_retain_graph_accumulates_twice(A, lipnet):
    net, _ = lipnet
    emb = rand_emb(3, 20, 6912, seed=14) * 0.25
    w = torch.randn((3, 20, 39), generator=torch.Generator().manual_seed(14)).cuda()
    clear_grads(net)
    (net.gru_head_train(emb) * w).sum().backward()
    once = net_grads(net)
    clear_grads(net)
    loss = (net.gru_head_train(emb) * w).sum()
    loss.backward(retain_graph=True)
    loss.backward()
    twice = net_grads(net)
    for n in NAMES:
        assert torch.equal(twice[n], 2 * once[n]), n


@pytest.mark.gpu
def test_head_train_interleaved_graphs(A, lipnet):
    """Two forwards, then their backwards in reverse order: each graph keeps its own workspace and masks, so each gives
    the bits of its own sequential run."""
    net, _ = lipnet
    embs = [rand_emb(3, 20, 6912, seed=15 + i) * 0.25 for i in range(2)]
    ws = [torch.randn((3, 20, 39), generator=torch.Generator().manual_seed(17 + i)).cuda() for i in range(2)]
    seq = []
    for i in range(2):
        clear_grads(net)
        torch.manual_seed(20 + i)
        (net.gru_head_train(embs[i], dropout=0.3) * ws[i]).sum().backward()
        seq.append(net_grads(net))
    losses = []
    for i in range(2):
        torch.manual_seed(20 + i)
        losses.append((net.gru_head_train(embs[i], dropout=0.3) * ws[i]).sum())
    for i in (1, 0):
        clear_grads(net)
        losses[i].backward()
        got = net_grads(net)
        for n in NAMES:
            assert torch.equal(got[n], seq[i][n]), (i, n)
