"""Kernel variants outside the headline configuration, against float64 references (oracle/f64_ref.py, oracle/mfcc_ref.py).

The dispatch code picks a kernel from the shape: K3's recurrence from the GRU hidden size and the precision, K4's score
kernel from the detector's hidden size, the shift count and n_mfcc, K1's kernels from n_mfcc.  Every case below names
the kernel it launches in its id, and for each family one test recomputes the dispatch rule of the CUDA source
(gru.cu: avs_bigru_forward, score.cu: sweep_score_impl, mfcc.cu) and checks that the cases reach every branch and
every clip-group boundary, so that a change of a threshold cannot leave a branch untested.

Measured errors are printed with report(); each tolerance sits at about twice the error measured on an NVIDIA B200
(see the constants below).  Tests without a device are unmarked; the others are marked gpu."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import f64_ref, mfcc_ref, sweep_ref


def _sm_count():
    """Streaming multiprocessors the persistent K4 grid is sized by (score.cu asks the device); 148 on a B200, the value
    used where no device is present."""
    if torch.cuda.is_available():
        return torch.cuda.get_device_properties(0).multi_processor_count
    return 148


N_SMS = _sm_count()
SR = 16000
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    "alignment-between-speech-and-visual-mouth-movements_b200", "csrc")


def source_has(name, *fragments):
    """The dispatch rules restated below are pinned to the CUDA source: if one of these lines changes, the
    restatement (and with it the coverage the cases are checked for) must be revisited."""
    src = " ".join(open(os.path.join(CSRC, name)).read().split())
    for f in fragments:
        assert " ".join(f.split()) in src, f"{name} no longer contains `{f}`: update the dispatch rule of this test"


@pytest.fixture(scope="module")
def native():
    import avsync_b200
    N = avsync_b200._native
    if not os.path.isfile(N.LIB_PATH):
        N.build()
    return N


@pytest.fixture(scope="module")
def A():
    import avsync_b200
    avsync_b200._native.device_check()
    return avsync_b200


def report(name, got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    err = np.abs(got - want)
    big = np.abs(want) > 1e-2
    rel = err / np.maximum(np.abs(want), 1e-6)
    print(f"[variants] {name}: max_abs={err.max():.3e} mean_abs={err.mean():.3e} "
          f"max_rel(|want|>1e-2)={rel[big].max() if big.any() else 0:.3e} ref_absmax={np.abs(want).max():.3e}")
    return float(err.max())


# ============================================================================================== K3: Bi-GRU head
# Tolerances: absolute bounds on log-probabilities against float64, about twice the largest error measured on an NVIDIA
# B200 (1000 W) per group of cases; all are tighter than the suite's fp32-grade bar for log-probs (rtol 1e-3 / atol 1e-4).
# Measured: fp32 5.2e-7, saturating 1.6e-6; bf16x3 1.9e-6, saturating 2.8e-5, LipNet head at in_dim 6912 1.2e-5 (the
# tcgen05 projections keep three of the four hi/lo bf16 products, ~2^-16 of the magnitude of the sum: larger inputs,
# weights and reductions give larger errors).
K3_ATOL = {("fp32", False): 1e-6, ("fp32", True): 3.5e-6, ("bf16x3", False): 4e-6, ("bf16x3", True): 6e-5}
K3_ATOL_LIPNET = 2.5e-5
K3_SUM_TOL = 6e-7                      # |sum_v exp(logp) - 1|, measured 2.9e-7


def k3_recurrence(hidden, precision):
    """The recurrence kernel avs_bigru_forward (gru.cu) launches."""
    if hidden == 256:                  # kCluH: resident-weight cluster kernels
        return "cluster_fp32" if precision == "fp32" else "cluster_umma"
    return "generic"                   # gru_recurrence_kernel<kGruClips = 4>, every precision


def k3_projection(precision):
    return "sgemm" if precision == "fp32" else "tcgen05"


# clips per CTA / group of each recurrence kernel: gru.cu kGruClips, kCluClips; gru_umma.cu kGrpClips x kGroups
K3_GROUP = {"generic": 4, "cluster_fp32": 16, "cluster_umma": 32}
K3_B_BOUNDARIES = {"generic": {1, 4, 5}, "cluster_fp32": {1, 16, 17, 32, 33}, "cluster_umma": {1, 16, 17, 32, 33}}

# (hidden, precision, B, T, vocab, in_dim, saturating)
K3_CASES = [
    (32, "fp32", 5, 75, 39, 40, False),
    (128, "fp32", 4, 1, 1, 256, False),
    (512, "fp32", 5, 2, 100, 256, False),
    (1024, "fp32", 1, 75, 28, 256, False),
    (128, "fp32", 1, 200, 39, 256, False),
    (128, "fp32", 5, 75, 39, 256, True),
    (32, "bf16x3", 1, 75, 100, 256, False),
    (128, "bf16x3", 5, 75, 39, 256, False),
    (512, "bf16x3", 4, 2, 28, 256, False),
    (1024, "bf16x3", 5, 1, 1, 64, False),
    (128, "bf16x3", 1, 200, 39, 256, False),
    (128, "bf16x3", 5, 75, 100, 256, True),
    (256, "fp32", 16, 75, 39, 256, False),
    (256, "fp32", 17, 2, 100, 256, False),
    (256, "fp32", 32, 1, 28, 256, False),
    (256, "fp32", 33, 75, 1, 256, False),
    (256, "fp32", 1, 200, 39, 256, False),
    (256, "fp32", 17, 75, 39, 256, True),
    (256, "bf16x3", 16, 75, 39, 256, False),
    (256, "bf16x3", 17, 1, 100, 256, False),
    (256, "bf16x3", 32, 2, 28, 256, False),
    (256, "bf16x3", 33, 75, 39, 256, False),
    (256, "bf16x3", 1, 200, 1, 256, False),
    (256, "bf16x3", 17, 75, 39, 256, True),
]


def k3_id(c):
    H, prec, B, T, V, ind, sat = c
    return (f"{k3_recurrence(H, prec)}+{k3_projection(prec)}-{prec}-H{H}-B{B}-T{T}-V{V}-in{ind}" + ("-saturating" if sat else ""))


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


class Head:
    """A native Bi-GRU head (avs_bigru_create) with any in_dim, built from a parameter dict as LipNet._bigru builds it."""

    def __init__(self, N, params, in_dim, hidden, vocab, precision):
        self.N, self.vocab = N, vocab
        keep = []
        for g in ("gru1", "gru2"):                   # [2][...]: forward then reverse (include/avsync.h)
            for n in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"):
                keep.append(torch.stack([params[f"{g}.{n}"], params[f"{g}.{n}_reverse"]]).float().contiguous().cuda())
        keep += [params["fc.weight"].float().contiguous().cuda(), params["fc.bias"].float().contiguous().cuda()]
        h = N.c_void_p()
        N.check(N.lib().avs_bigru_create(in_dim, hidden, vocab, *[N.ptr(t) for t in keep], N.PREC[precision],
                                         N.stream_ptr(), ctypes.byref(h)), "bigru_create")
        self.handle = N.Handle(h, N.lib().avs_bigru_destroy, keep)

    def __call__(self, emb):
        N, L = self.N, self.N.lib()
        B, T, _ = emb.shape
        out = torch.full((B, T, self.vocab), float("nan"), device="cuda")    # a row the kernels skip stays NaN
        ws = N.workspace(L.avs_bigru_workspace_bytes(self.handle.h, B, T), "cuda")
        N.check(L.avs_bigru_forward(self.handle.h, N.ptr(emb), B, T, N.ptr(out), N.ptr(ws), ws.numel(), N.stream_ptr()),
                "bigru_forward")
        return out


def k3_check(name, got, want, atol):
    got = got.cpu().numpy()
    want = want.numpy()
    assert np.isfinite(got).all(), name
    report(f"logp[{name}]", got, want)
    np.testing.assert_allclose(got, want, rtol=0, atol=atol, err_msg=name)
    s = np.abs(np.exp(got.astype(np.float64)).sum(-1) - 1.0).max()
    print(f"[variants] rowsum[{name}]: max |sum exp - 1| = {s:.3e}")
    assert s <= K3_SUM_TOL, (name, s)


def test_k3_cases_reach_every_recurrence_kernel_and_boundary():
    source_has("gru.cu", "constexpr int kGruClips = 4;", "kCluClips = 16,", "kCluH = 256,",
               "if (g->w_hh_packed[l] != nullptr && !force_fma) {", "} else if (H == kCluH) {",
               "if (!rc && hidden == 256) {", "if (g->precision == AVS_PREC_FP32) {")
    source_has("gru_umma.cu", "constexpr int kGrpClips = 16, kGroups = 2;")
    kernels = {k3_recurrence(c[0], c[1]) for c in K3_CASES}
    assert kernels == {"generic", "cluster_fp32", "cluster_umma"}
    for prec in ("fp32", "bf16x3"):
        assert {c[0] for c in K3_CASES if c[1] == prec} == {32, 128, 256, 512, 1024}, prec
    for kern, need in K3_B_BOUNDARIES.items():
        cases = [c for c in K3_CASES if k3_recurrence(c[0], c[1]) == kern]
        assert {c[2] for c in cases} >= need, kern
        assert all(any(c[2] % K3_GROUP[kern] == r for c in cases) for r in (0, 1)), kern   # full and ragged last group
        assert {c[3] for c in cases} >= {1, 2, 75, 200}, kern
        assert {c[4] for c in cases} >= {1, 28, 39, 100}, kern
        assert any(c[6] for c in cases), kern                                                 # a saturating case
    # vocab 100 spans more than two 32-lane passes of log_softmax_kernel; 39 does not
    assert any(c[4] > 64 for c in K3_CASES)
    for c in K3_CASES:
        assert c[0] < 1024 or c[2] <= 5, "keep hidden-1024 cases small in B"
        assert c[3] < 200 or c[2] == 1, "keep T = 200 cases small in B"


def test_f64_head_matches_the_float32_oracle():
    """The float64 head agrees with oracle/lipnet_ref's float32 recurrence (a different implementation) to float32
    rounding: it restates the same model."""
    from oracle import lipnet_ref
    p = gru_params(64, 48, 30, seed=1)
    emb = torch.rand((3, 9, 48), generator=torch.Generator().manual_seed(2)) * 0.2
    want = f64_ref.bigru_head_f64(p, emb)
    assert want.dtype == torch.float64
    got = lipnet_ref.gru_head(p, emb)
    np.testing.assert_allclose(got.numpy(), want.numpy(), rtol=0, atol=2e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("case", K3_CASES, ids=[k3_id(c) for c in K3_CASES])
def test_k3_head_vs_f64(A, case):
    H, prec, B, T, V, in_dim, sat = case
    name = k3_id(case)
    seed = (H * 7 + B * 131 + T * 17 + V + in_dim + (1000 if sat else 0)) % 100003
    p = gru_params(H, in_dim, V, seed, sat)
    emb = torch.rand((B, T, in_dim), generator=torch.Generator().manual_seed(seed)) * 0.2
    want = f64_ref.bigru_head_f64(p, emb)
    head = Head(A._native, p, in_dim, H, V, prec)
    embd = emb.cuda()
    got = head(embd)
    k3_check(name, got, want, K3_ATOL[(prec, sat)])
    # batch independence, bit for bit: a clip's rows do not depend on the batch (every group boundary of the kernel)
    for i in sorted({0, 3, 4, 15, 16, 31, 32, B - 1}):
        if B > 1 and i < B:
            assert torch.equal(head(embd[i:i + 1].contiguous())[0], got[i]), (name, i)


@pytest.mark.gpu
def test_k3_bf16_head_is_the_bf16x3_head(A):
    """LipNet(precision='bf16') runs its head exactly as 'bf16x3' does (only the STCNN differs): same bits."""
    p = gru_params(256, 256, 39, seed=5)
    emb = (torch.rand((17, 75, 256), generator=torch.Generator().manual_seed(5)) * 0.2).cuda()
    a = Head(A._native, p, 256, 256, 39, "bf16")(emb)
    b = Head(A._native, p, 256, 256, 39, "bf16x3")(emb)
    assert torch.equal(a, b)
    c = Head(A._native, gru_params(128, 256, 39, seed=6), 256, 128, 39, "bf16")(emb)
    d = Head(A._native, gru_params(128, 256, 39, seed=6), 256, 128, 39, "bf16x3")(emb)
    assert torch.equal(c, d)


@pytest.mark.gpu
def test_k3_refuses_rows_past_the_fc_grid_limit(A):
    """The fc product runs on sgemm_nt's tiled kernel over all n_clips * n_steps rows, gridDim.y = ceil(rows / 128) <=
    65535: one row more is refused before any launch (the pointers past the handle are never touched)."""
    N = A._native
    head = Head(N, gru_params(32, 8, 1, seed=1), 8, 32, 1, "fp32")
    fake = ctypes.c_void_p(256)
    for B, T in ((65535 * 128 + 1, 1), (1, 65535 * 128 + 1), (2796161, 3)):
        assert N.lib().avs_bigru_forward(head.handle.h, fake, B, T, fake, fake, 1 << 40, N.stream_ptr()) == -1
        assert "n_clips * n_steps must be <= 8388480" in N.lib().avs_last_error_string().decode()
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_k3_lipnet_hidden128_gru_head_vs_f64(A):
    """The drop-in module with a non-default hidden size: LipNet(39, hidden_dim=128).gru_head at in_dim 6912 (generic
    recurrence, tcgen05 projections with N = 768)."""
    from oracle import lipnet_ref
    sd = lipnet_ref.init_lipnet_state(39, 128, seed=3)
    net = A.LipNet(39, hidden_dim=128, precision="bf16x3")
    net.load_state_dict(sd)
    net = net.cuda().eval()
    emb = torch.rand((2, 75, 6912), generator=torch.Generator().manual_seed(3)) * 0.2
    want = f64_ref.bigru_head_f64({k: v for k, v in sd.items() if k.split(".")[0] in ("gru1", "gru2", "fc")}, emb)
    got = net.gru_head(emb.cuda())
    k3_check("generic+tcgen05-bf16x3-lipnet-H128-B2-T75-V39-in6912", got, want, K3_ATOL_LIPNET)


# ============================================================================================== K4: sweep score
# Tolerances: absolute bounds on scores against float64, about twice the error measured on an NVIDIA B200 (1000 W):
# fp32 K4 2.3e-7 (the suite's bar: rtol 1e-3 / atol 1e-5), the bf16 sweep's tensor-core K4 on its own statistics 1.6e-7
# (the suite's bar: 2e-6).
K4_ATOL = 5e-7
K4_TC_ATOL = 3.5e-7


def k4_variant(hidden, n_shifts, a_dim):
    """The score kernel sweep_score_impl (score.cu) launches for the fp32 K4, or 'reject'."""
    sm = (n_shifts * a_dim + n_shifts) * 4
    if sm > 48 * 1024:
        return "reject"
    sm_p = sm + a_dim * (hidden + 1) * 4
    if sm_p > 200 * 1024:
        return "fallback"                                         # sweep_score_kernel, one CTA per clip
    return "persistent16x6" if hidden == 512 and n_shifts <= 48 else "persistent"


def k4_grid_loops(hidden, n_shifts, a_dim, n_clips):
    """Whether a persistent CTA scores more than one clip (grid = min(clips, SMs x (2 if sm_p <= 100 KB else 1)))."""
    sm_p = (n_shifts * a_dim + n_shifts) * 4 + a_dim * (hidden + 1) * 4
    return n_clips > N_SMS * (2 if sm_p <= 100 * 1024 else 1)


# (hidden, n_mfcc, K, clips, Dv)
K4_CASES = [
    (512, 20, 41, 297, 13824),      # the reference's detector: register-blocked kernel, the grid loops
    (512, 20, 48, 3, 13824),        # last shift count of the register-blocked kernel
    (512, 20, 49, 3, 13824),        # first shift count past it
    (512, 40, 41, 2, 13824),        # register-blocked, one CTA per SM
    (512, 13, 1, 1, 264),
    (256, 20, 41, 297, 13824),      # the reference's default detector (hidden 256): generic kernel, the grid loops
    (100, 13, 21, 2, 264),
    (64, 40, 121, 3, 13824),
    (64, 20, 299, 3, 264),          # s_a at its 48 KB limit
    (1000, 20, 41, 2, 13824),       # generic kernel, one CTA per SM
    (1000, 20, 299, 1, 13824),      # hidden 1000 with 299 shifts no longer fits: fallback kernel
    (2048, 20, 41, 3, 13824),
    (2048, 13, 1, 1, 264),
    (2048, 40, 48, 2, 264),
]


def k4_id(c):
    H, nm, K, B, Dv = c
    v = k4_variant(H, K, 2 * nm)
    return f"{v}{'-loops' if k4_grid_loops(H, K, 2 * nm, B) else ''}-H{H}-nmfcc{nm}-K{K}-clips{B}-Dv{Dv}"


def test_k4_cases_reach_every_score_kernel():
    source_has("score.cu", "const size_t sm = (static_cast<size_t>(n_shifts) * a_dim + n_shifts) * sizeof(float);",
               "AVS_REQUIRE(sm <= 48 * 1024,", "const size_t sm_p = sm + static_cast<size_t>(a_dim) * (hidden + 1) * sizeof(float);",
               "if (sm_p <= 200 * 1024) {", "std::min(n_clips, n_sms * (sm_p <= 100 * 1024 ? 2 : 1));",
               "(hidden == 512 && n_shifts <= 48) ? sweep_score_persistent_kernel<16, 6> : sweep_score_persistent_kernel<0, 1>;")
    variants = {k4_variant(c[0], c[2], 2 * c[1]) for c in K4_CASES}
    assert variants == {"persistent16x6", "persistent", "fallback"}
    assert k4_variant(64, 300, 40) == "reject" and k4_variant(64, 299, 40) != "reject"   # test_k4_rejects_...
    for v in ("persistent16x6", "persistent"):
        assert any(k4_variant(c[0], c[2], 2 * c[1]) == v and k4_grid_loops(c[0], c[2], 2 * c[1], c[3]) for c in K4_CASES), v
    assert {c[0] for c in K4_CASES} >= {64, 100, 256, 512, 1000, 2048}
    assert {c[1] for c in K4_CASES} >= {13, 20, 40}
    assert {c[2] for c in K4_CASES} >= {1, 21, 41, 48, 49, 121, 299}
    assert {c[3] for c in K4_CASES} >= {1, 2, 3, 297}
    assert {c[4] for c in K4_CASES} == {264, 13824}
    # hidden 512 at 48 and 49 shifts sit on both sides of the register-blocked kernel's limit
    assert k4_variant(512, 48, 40) == "persistent16x6" and k4_variant(512, 49, 40) == "persistent"


def test_f64_detector_matches_the_float32_oracle():
    det = sweep_ref.init_detector_state(30 + 8, 16, seed=3)
    g = torch.Generator().manual_seed(3)
    v, a = torch.rand((2, 30), generator=g), torch.randn((2, 5, 8), generator=g) * 20
    want = f64_ref.detector_scores_f64(det["classifier.0.weight"], det["classifier.0.bias"], det["classifier.3.weight"],
                                       det["classifier.3.bias"], v, a)
    x = torch.cat([v[:, None, :].expand(-1, 5, -1), a], dim=-1)
    np.testing.assert_allclose(torch.sigmoid(sweep_ref.detector_logits(det, x)).numpy(), want, rtol=0, atol=1e-6)


def detector_state(in_dim, hidden, seed):
    return sweep_ref.init_detector_state(in_dim, hidden, seed=seed)


def det_weights(sd):
    return [sd[k] for k in ("classifier.0.weight", "classifier.0.bias", "classifier.3.weight", "classifier.3.bias")]


def sweep_score_native(N, w, v, a):
    """avs_sweep_score with NaN / -1 in the outputs beforehand, so that a score or offset the kernel skips cannot pass."""
    L = N.lib()
    w1, b1, w2, b2 = [t.float().contiguous().cuda() for t in w]
    B, K, Da = a.shape
    H = w1.shape[0]
    scores = torch.full((B, K), float("nan"), device="cuda")
    best = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    ws = N.workspace(L.avs_sweep_score_workspace_bytes(B, H), "cuda")
    N.check(L.avs_sweep_score(N.ptr(v), N.ptr(a), B, K, v.shape[1], Da, N.ptr(w1), N.ptr(b1), N.ptr(w2), N.ptr(b2), H,
                              N.ptr(scores), N.ptr(best), N.ptr(ws), ws.numel(), N.stream_ptr()), "sweep_score")
    return scores, best


def check_best(name, best, want, err):
    """best must be the float64 arg-max wherever the float64 top-2 margin exceeds 10x the measured error; that must be
    most rows, so that the check stays live."""
    K = want.shape[1]
    if K == 1:
        assert (best == 0).all(), name
        return
    srt = np.sort(want, axis=1)
    clear = (srt[:, -1] - srt[:, -2]) > 10 * max(err, 1e-9)
    print(f"[variants] best[{name}]: {int(clear.sum())}/{len(clear)} rows resolvable")
    assert clear.mean() > 0.5, (name, clear.mean())
    assert (best[clear] == want.argmax(1)[clear]).all(), name


@pytest.mark.gpu
@pytest.mark.parametrize("case", K4_CASES, ids=[k4_id(c) for c in K4_CASES])
def test_k4_sweep_score_vs_f64(A, case):
    H, nm, K, B, Dv = case
    name = k4_id(case)
    Da = 2 * nm
    seed = (H + 3 * nm + 7 * K + 11 * B + Dv) % 100003
    sd = detector_state(Dv + Da, H, seed)
    w = det_weights(sd)
    g = torch.Generator().manual_seed(seed)
    v = torch.rand((B, Dv), generator=g) * 0.3                  # visual statistics: non-negative, ~0.3
    a = torch.randn((B, K, Da), generator=g) * 20               # audio statistics
    want = f64_ref.detector_scores_f64(*w, v, a)
    tie = None
    if K > 1:                                                   # clip 0: an exact tie at its maximum
        m = int(want[0].argmax())
        j = 0 if m > 0 else K - 1
        a[0, j] = a[0, m]
        want[0] = f64_ref.detector_scores_f64(*w, v[:1], a[:1])[0]
        tie = min(j, m)
    vd, ad = v.cuda(), a.cuda()
    sc, best = sweep_score_native(A._native, w, vd, ad)
    got, best = sc.cpu().numpy(), best.cpu().numpy()
    assert np.isfinite(got).all(), name
    err = report(f"scores[{name}]", got, want)
    np.testing.assert_allclose(got, want, rtol=0, atol=K4_ATOL, err_msg=name)
    rows = slice(None)
    if tie is not None:                                         # the first of the tied maxima (np.argmax)
        top = np.flatnonzero(got[0] == got[0].max())
        assert len(top) >= 2 and best[0] == top[0] == tie, (name, top, best[0], tie)
        rows = slice(1, None)
    if len(best[rows]):
        check_best(name, best[rows], want[rows], err)
    # the module-level entry point gives the same bits
    det = A.MisalignmentDetector(Dv + Da, H)
    det.load_state_dict(sd)
    sc2, best2 = A.sweep_score(vd, ad, det.cuda().eval())
    assert torch.equal(sc2.cpu(), torch.from_numpy(got)) and np.array_equal(best2.cpu().numpy(), best), name


@pytest.mark.gpu
def test_k4_rejects_shift_tables_over_48kb_and_recovers(A):
    """300 shifts x 40 audio features do not fit the 48 KB shift table: a clean RuntimeError, and the same call at 299
    shifts still works afterwards."""
    H, Dv, Da = 64, 264, 40
    sd = detector_state(Dv + Da, H, seed=8)
    det = A.MisalignmentDetector(Dv + Da, H)
    det.load_state_dict(sd)
    det = det.cuda().eval()
    g = torch.Generator().manual_seed(8)
    v = (torch.rand((2, Dv), generator=g) * 0.3).cuda()
    a = (torch.randn((2, 300, Da), generator=g) * 20).cuda()
    with pytest.raises(RuntimeError, match="n_shifts \\* a_dim too large"):
        A.sweep_score(v, a, det)
    sc, best = A.sweep_score(v, a[:, :299].contiguous(), det)
    want = f64_ref.detector_scores_f64(*det_weights(sd), v.cpu(), a[:, :299].cpu())
    report("scores[persistent-H64-nmfcc20-K299 after a rejected call]", sc.cpu().numpy(), want)
    np.testing.assert_allclose(sc.cpu().numpy(), want, rtol=0, atol=K4_ATOL)


# bf16 sweep: the detector's hidden layer on the tensor cores (split-K hi/lo tcgen05 GEMM) when hidden % 4 == 0, else the
# fp32 GEMM; N tails (hidden 100, 1000), M tails (clips not a multiple of 128) with chunks of 128 clips.
def k4_sweep_gemm(hidden):
    """The hidden-layer GEMM of a bf16 SyncSweeper (sweep.cu: tensor_k4, score.cu: sweep_score_tensor_gemm_ok)."""
    return "tcgen05splitk" if hidden % 4 == 0 else "sgemm"


K4_SWEEP_CASES = [(100, 1), (100, 300), (256, 129), (1000, 1), (1000, 129), (130, 129)]


def test_k4_sweep_cases_reach_both_gemms():
    source_has("score.cu", "return v_dim % 32 == 0 && (v_dim + a_dim) % 4 == 0 && hidden % 4 == 0;")
    source_has("sweep.cu", "stcnn_precision(net) == AVS_PREC_BF16 && sweep_score_tensor_gemm_ok(AVS_VSTATS, 2 * s->n_mfcc, hidden);")
    assert {k4_sweep_gemm(h) for h, _ in K4_SWEEP_CASES} == {"tcgen05splitk", "sgemm"}
    tc = [(h, n) for h, n in K4_SWEEP_CASES if k4_sweep_gemm(h) == "tcgen05splitk"]
    assert {h for h, _ in tc} >= {100, 256, 1000} and {n for _, n in tc} >= {1, 129, 300}
    assert any(h % 256 for h, _ in tc) and any(n % 128 for _, n in tc)       # N and M tails


@pytest.fixture(scope="module")
def bf16_net(A):
    from oracle import lipnet_ref
    net = A.LipNet(39, precision="bf16")
    net.load_state_dict(lipnet_ref.init_lipnet_state(39, 256, seed=0))
    return net.cuda().eval()


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,n_clips", K4_SWEEP_CASES,
                         ids=[f"{k4_sweep_gemm(h)}-H{h}-clips{n}-chunk128" for h, n in K4_SWEEP_CASES])
def test_k4_bf16_sweep_vs_f64(A, bf16_net, hidden, n_clips):
    S = 20
    sd = detector_state(13864, hidden, seed=hidden)
    det = A.MisalignmentDetector(13864, hidden)
    det.load_state_dict(sd)
    det = det.cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(n_clips)
    frames = torch.randint(0, 256, (n_clips, 1, 75, 50, 100), generator=g, dtype=torch.uint8, device="cuda")
    audio = torch.from_numpy(sweep_ref.synth_audio(n_clips, seed=hidden + n_clips, kind="speechlike")).cuda()
    sw = A.SyncSweeper(bf16_net, det, S, chunk_clips=128)
    sc, best = sw.run(frames, audio)
    v = A.visual_stats(bf16_net, frames)
    a = A.audio_stats_sweep(audio, [640 * k for k in range(-S, S + 1)])
    want = f64_ref.detector_scores_f64(*det_weights(sd), v.cpu(), a.cpu())
    name = f"{k4_sweep_gemm(hidden)}-H{hidden}-clips{n_clips}"
    got = sc.cpu().numpy()
    err = report(f"bf16 sweep scores[{name}]", got, want)
    assert err <= K4_TC_ATOL, (name, err)
    if n_clips > 1:
        check_best(name, best.cpu().numpy() + S, want, err)


# ============================================================================================== K1: MFCC statistics
# Tolerances: absolute bounds on the statistics (values up to ~490 in magnitude) against the float64 oracle, about twice
# the error measured on an NVIDIA B200 (1000 W): 6.7e-4 on 3-s clips, 5.9e-5 on the long clips at the frame limit.
# The suite's bar for MFCC statistics is rtol 1e-3 / atol 2e-3.
K1_ATOL = 1.4e-3
K1_LIMIT_ATOL = 1.2e-4
K1_NMFCC = [1, 13, 20, 21, 40]
SHIFT_FRAMES = list(range(-20, 21))


def k1_kernels(n_mfcc):
    """The instantiation of the log-mel and statistics kernels (mfcc.cu: NQ = 20 up to n_mfcc 20, else kMaxQ = 40)."""
    return "nq20" if n_mfcc <= 20 else "nq40"


def k1_max_frames(n_mfcc):
    """STFT frames the statistics kernel holds in 227 KB of shared memory: (128 mel rows + F frames) x NQ floats."""
    nq = 20 if n_mfcc <= 20 else 40
    return 227 * 1024 // (nq * 4) - 128


def test_k1_cases_reach_both_instantiations():
    source_has("mfcc.cu", "if (p->n_mfcc <= 20) mfcc_logmel_warp_kernel<false, 20>", "const int nq = n_mfcc <= 20 ? 20 : kMaxQ;",
               "constexpr int kStatsSmemLimit = 227 * 1024;", "return kStatsSmemLimit / (nq * static_cast<int>(sizeof(float))) - kMels;")
    assert {k1_kernels(n) for n in K1_NMFCC} == {"nq20", "nq40"}
    assert {1, 20, 21, 40} <= set(K1_NMFCC)          # both ends of both instantiations
    assert k1_max_frames(20) == 2777 and k1_max_frames(40) == 1324 and k1_max_frames(1) == 2777


_mfcc_cache = {}


def mfcc40_ref(key, y, sr=SR):
    """mfcc_ref's 40 coefficients per frame (librosa's chain, which returns float32); n_mfcc < 40 is a prefix of them."""
    if key not in _mfcc_cache:
        _mfcc_cache[key] = mfcc_ref.mfcc(y, sr, 40, max(1, sr // 40)).astype(np.float64)
    return _mfcc_cache[key]


def stats_f64(m):
    """[mean, unbiased std] over frames of an [n_mfcc, F] table, in float64."""
    return np.concatenate([m.mean(1), m.std(1, ddof=1)])


def k1_audio(n, seed):
    """One speech-like clip and one half-silent clip (its silent third drives the top_db clamp)."""
    return [sweep_ref.synth_audio(1, seed=seed, n_samples=n, kind="speechlike")[0],
            sweep_ref.synth_audio(1, seed=seed + 1, n_samples=n, kind="halfsilent")[0]]


def k1_oracle(tag, clips, fps_list, n_mfcc):
    out = np.empty((len(clips), len(SHIFT_FRAMES), 2 * n_mfcc))
    for i, (x, fps) in enumerate(zip(clips, fps_list)):
        for j, k in enumerate(SHIFT_FRAMES):
            m = mfcc40_ref((tag, i, k), sweep_ref.shift_audio(x, k, fps, SR))
            out[i, j] = stats_f64(m[:n_mfcc])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n_mfcc", K1_NMFCC, ids=[f"{k1_kernels(n)}-nmfcc{n}" for n in K1_NMFCC])
def test_k1_uniform_sweep_vs_oracle(A, n_mfcc):
    clips = k1_audio(48000, seed=300)
    got = A.audio_stats_sweep(torch.from_numpy(np.stack(clips)).cuda(), [640 * k for k in SHIFT_FRAMES], SR, n_mfcc)
    want = k1_oracle("uniform", clips, [25.0, 25.0], n_mfcc)
    name = f"{k1_kernels(n_mfcc)}-nmfcc{n_mfcc}-uniform"
    report(f"astats[{name}]", got.cpu().numpy(), want)
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=0, atol=K1_ATOL, err_msg=name)


@pytest.mark.gpu
@pytest.mark.parametrize("n_mfcc", K1_NMFCC, ids=[f"{k1_kernels(n)}-nmfcc{n}" for n in K1_NMFCC])
def test_k1_ragged_sweep_vs_oracle(A, n_mfcc):
    from avsync_b200 import shift_samples
    lengths, fps_list = (40000, 52000, 45001, 47999), (25.0, 29.97, 29.97, 25.0)
    clips = k1_audio(40000, 310)[:1] + k1_audio(52000, 311)[1:] + k1_audio(45001, 312)[:1] + k1_audio(47999, 313)[1:]
    assert tuple(len(x) for x in clips) == lengths
    rows = [[shift_samples(k, f, SR) for k in SHIFT_FRAMES] for f in fps_list]
    got = A.audio_stats_sweep_ragged([torch.from_numpy(x).cuda() for x in clips], rows, SR, n_mfcc)
    want = k1_oracle("ragged", clips, fps_list, n_mfcc)
    name = f"{k1_kernels(n_mfcc)}-nmfcc{n_mfcc}-ragged"
    report(f"astats[{name}]", got.cpu().numpy(), want)
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=0, atol=K1_ATOL, err_msg=name)


@pytest.mark.gpu
@pytest.mark.parametrize("n_mfcc", [20, 40], ids=["nq20-nmfcc20-2777frames", "nq40-nmfcc40-1324frames"])
def test_k1_clip_at_the_frame_limit(A, n_mfcc):
    """A clip of exactly the most frames the statistics kernel holds, through the uniform and the ragged plan: the two
    agree bit for bit and match the oracle."""
    F = k1_max_frames(n_mfcc)
    n = (F - 1) * (SR // 40)
    x = sweep_ref.synth_audio(1, seed=n_mfcc, n_samples=n, kind="speechlike")[0]
    ks = (-20, -1, 0, 7, 20)
    shifts = [sweep_ref.shift_samples(k, 25.0, SR) for k in ks]
    xd = torch.from_numpy(x).cuda()
    uni = A.audio_stats_sweep(xd[None], shifts, SR, n_mfcc)
    rag = A.audio_stats_sweep_ragged([xd], [shifts], SR, n_mfcc)
    assert torch.equal(uni, rag)
    from avsync_b200.misalignment_detection_train import mfcc_plan
    assert mfcc_plan(n, SR, n_mfcc, shifts).n_frames == F
    want = np.stack([stats_f64(mfcc_ref.mfcc(sweep_ref.shift_audio(x, k, 25.0, SR), SR, n_mfcc, SR // 40).astype(np.float64))
                     for k in ks])
    report(f"astats[{k1_kernels(n_mfcc)}-nmfcc{n_mfcc}-{F}frames]", uni[0].cpu().numpy(), want)
    np.testing.assert_allclose(uni[0].cpu().numpy(), want, rtol=0, atol=K1_LIMIT_ATOL)


def test_uniform_plan_refuses_clips_over_the_frame_limit_without_a_device(native):
    """avs_mfcc_plan_create rejects a clip with more STFT frames than the statistics kernel holds with AVS_EINVAL (-1)
    and a message naming the limit, before any CUDA call, as the ragged plan does."""
    L = native.lib()
    h = ctypes.c_void_p()
    arr = (ctypes.c_int32 * 3)(0, 640, -640)
    for frames, nm, limit, sr in ((2778, 20, 2777, 16000), (2778, 1, 2777, 16000), (1325, 40, 1324, 16000),
                                  (1325, 21, 1324, 16000), (2778, 20, 2777, 8000), (3000, 13, 2777, 16000)):
        n = (frames - 1) * (sr // 40)
        assert L.avs_mfcc_plan_create(n, sr, nm, arr, 3, ctypes.byref(h)) == -1, (frames, nm, sr)
        msg = L.avs_last_error_string()
        assert str(limit).encode() in msg and str(frames).encode() in msg, msg
    # the ragged plan draws the line at the same clip
    ln = (ctypes.c_int32 * 1)(2777 * 400)
    assert L.avs_mfcc_ragged_plan_create(1, ln, 16000, 20, arr, 3, None, ctypes.byref(h)) == -1
    assert b"2777" in L.avs_last_error_string()


@pytest.mark.gpu
def test_compute_audio_stats_refuses_a_70s_clip(A):
    x = sweep_ref.synth_audio(1, seed=70, n_samples=70 * SR, kind="speechlike")[0]
    with pytest.raises(RuntimeError, match="at most 2777 frames"):
        A.compute_audio_stats(x, SR, 20)
    with pytest.raises(RuntimeError, match="at most 1324 frames"):
        A.compute_audio_stats(x[:40 * SR], SR, 40)
    assert torch.isfinite(A.compute_audio_stats(x[:48000], SR, 20)).all()     # the device is still usable
