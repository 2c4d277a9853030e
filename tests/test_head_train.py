"""Head fine-tuning on the B200: the CTC loss and gradient (K5e, csrc/ctc_loss.cu) against the float64 oracle
(oracle/ctc_loss_ref.py) and torch, bit-equality with K5c's log-likelihood; the head's training forward against
gru_head bit for bit; all 18 head gradients (K3b, csrc/gru_train.cu) against float64 torch autograd; determinism, error
paths and a small training run."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ctc_align_ref, ctc_beam_ref, lipnet_ref
from oracle import ctc_loss_ref as R

pytestmark = pytest.mark.gpu

# Largest errors measured on an NVIDIA B200 (1000 W power limit), see DESIGN §4.3:
#   ctc_loss: relative error of the loss 5.5e-8 (the fp32 rounding of an fp64 result), absolute error of the gradient
#   6.0e-8 against the float64 oracle;
#   head gradients: max |g - g64| / max |g64| per parameter, over the cases of test_head_gradients_vs_float64:
#   3.0e-6 with the fp32 forward, 1.9e-5 with the bf16x3 forward (its tcgen05 projections and recurrence round
#   differently from the fp32 recomputation of the gates in the backward).
LOSS_REL_TOL = 1.2e-7
GRAD_ABS_TOL = 1.2e-7
HEAD_GRAD_TOL = {"fp32": 6e-6, "bf16x3": 4e-5, "bf16": 4e-5}   # the bf16 head is the bf16x3 head

NAMES = [f"{g}.{n}{s}" for g in ("gru1", "gru2") for n in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")
         for s in ("", "_reverse")] + ["fc.weight", "fc.bias"]


@pytest.fixture(scope="module")
def A():
    import avsync_b200
    avsync_b200._native.device_check()
    return avsync_b200


@pytest.fixture(scope="module")
def c2i():
    from avsync_b200.dataset import create_vocab
    return create_vocab()[0]


def rand_logp(rng, B, T, V, scale=2.0):
    x = rng.normal(size=(B, T, V)) * scale
    return (x - np.logaddexp.reduce(x, axis=-1, keepdims=True)).astype(np.float32)


def logits_grad(lp, g):
    return g - np.exp(lp.astype(np.float64)) * g.sum(-1, keepdims=True)


def grid_batch(c2i, B, T=75, seed=0):
    _, targets, lens = ctc_align_ref.grid_targets(B, c2i, seed=seed)
    lp = rand_logp(np.random.default_rng(seed), B, T, 39)
    return lp, targets, lens


# ---------------------------------------------------------------------------------------------------- K5e
@pytest.mark.parametrize("zero_infinity", [False, True])
def test_ctc_loss_vs_oracle_with_mixed_statuses(A, c2i, zero_infinity):
    B, T = 64, 75
    lp, targets, lens = grid_batch(c2i, B, T, seed=1)
    il = np.full(B, T, np.int32)
    il[3] = 20           # infeasible: too short for its sentence
    lp[5, 10, 7] = np.nan     # NaN inside input_len
    il[6], lp[6, 70, 2] = 60, np.nan   # NaN past input_len: no effect
    targets[8, 2] = 39   # invalid id
    lens[9] = targets.shape[1] + 1   # invalid length
    targets[10, 0] = 0   # the blank as a label
    il[11] = 76          # invalid input length
    il[12], lens[12] = 0, 0   # no frames, empty target
    lens[13] = 0
    il[14] = 45
    scale = np.random.default_rng(2).uniform(0.1, 2.0, B).astype(np.float32)
    want_nll, want_g = R.loss_grad_batch(lp, targets, lens, il, scale=scale, zero_infinity=zero_infinity)
    x = torch.from_numpy(lp).cuda().requires_grad_()
    loss = A.ctc_loss(x, torch.from_numpy(targets), torch.from_numpy(il), torch.from_numpy(lens), reduction="none",
                      zero_infinity=zero_infinity)
    loss.backward(torch.from_numpy(scale).cuda())
    got_nll, got_g = loss.detach().cpu().numpy(), x.grad.cpu().numpy()
    np.testing.assert_array_equal(np.isnan(got_nll), np.isnan(want_nll))
    np.testing.assert_array_equal(np.isinf(got_nll), np.isinf(want_nll))
    fin = np.isfinite(want_nll)
    assert np.all(np.abs(got_nll[fin] - want_nll[fin]) <= LOSS_REL_TOL * np.maximum(1, np.abs(want_nll[fin])))
    np.testing.assert_array_equal(np.isnan(got_g), np.isnan(want_g))
    ok = ~np.isnan(want_g)
    rel = np.abs(got_nll[fin] - want_nll[fin]) / np.maximum(1, np.abs(want_nll[fin]))
    print(f"ctc_loss: max rel loss error {rel.max():.2e}, max abs gradient error {np.abs(got_g[ok] - want_g[ok]).max():.2e}")
    assert np.abs(got_g[ok] - want_g[ok]).max() <= GRAD_ABS_TOL
    assert (got_g[6, 60:] == 0).all() and (got_g[14, 45:] == 0).all()
    assert np.isnan(got_g[8]).all() and np.isnan(got_g[11]).all()
    assert np.isfinite(got_nll[6]) and np.isfinite(got_g[6]).all()


@pytest.mark.parametrize("reduction", ["mean", "sum", "none"])
def test_ctc_loss_vs_torch_float64(A, c2i, reduction):
    B, T = 17, 75
    rng = np.random.default_rng(3)
    logits = rng.normal(size=(B, T, 39)) * 2.0
    _, targets, lens = ctc_align_ref.grid_targets(B, c2i, seed=3)
    lens[0] = 0
    il = rng.integers(55, T + 1, B).astype(np.int32)
    x64 = torch.tensor(logits, requires_grad=True)
    want = F.ctc_loss(torch.log_softmax(x64, -1).transpose(0, 1), torch.from_numpy(targets).long(),
                      torch.from_numpy(il).long(), torch.from_numpy(lens).long(), reduction=reduction)
    want.sum().backward()
    x = torch.tensor(logits, dtype=torch.float32, device="cuda", requires_grad=True)
    got = A.ctc_loss(torch.log_softmax(x, -1), torch.from_numpy(targets), torch.from_numpy(il),
                     torch.from_numpy(lens), reduction=reduction)
    got.sum().backward()
    np.testing.assert_allclose(got.detach().cpu().numpy(), want.detach().numpy(), rtol=1e-6)
    np.testing.assert_allclose(x.grad.cpu().numpy(), x64.grad.numpy(), rtol=0,
                               atol=1e-6 * float(np.abs(x64.grad.numpy()).max()))


def test_nll_equals_minus_forced_align_loglik_bit_for_bit(A, c2i):
    B, T = 256, 75
    lp, targets, lens = grid_batch(c2i, B, T, seed=4)
    il = np.random.default_rng(4).integers(30, T + 1, B).astype(np.int32)
    dev = lambda a: torch.from_numpy(a).cuda()   # noqa: E731
    nll = A.ctc_loss(dev(lp), dev(targets), dev(il), dev(lens), reduction="none")
    ll = A.ctc_forced_align(dev(lp), dev(targets), dev(lens), dev(il)).loglik
    n, l = nll.cpu().numpy(), ll.cpu().numpy()
    fin = np.isfinite(l)
    assert fin.sum() > B // 2
    np.testing.assert_array_equal(n[fin], -l[fin])
    assert np.all(n[~fin] == np.inf)


def test_ctc_loss_corners_and_repeat_runs(A):
    rng = np.random.default_rng(5)
    lp = rand_logp(rng, 3, 1024, 64)
    targets = rng.integers(1, 64, size=(3, 512)).astype(np.int32)
    lens = np.array([512, 0, 100], np.int32)
    il = np.array([1024, 1024, 1], np.int32)
    dev = lambda a: torch.from_numpy(a).cuda()   # noqa: E731
    want_nll, want_g = R.loss_grad_batch(lp, targets, lens, il)
    outs = []
    for _ in range(2):
        x = dev(lp).requires_grad_()
        loss = A.ctc_loss(x, dev(targets), dev(il), dev(lens), reduction="none")
        loss.backward(torch.ones(3, device="cuda"))
        outs.append((loss.detach().cpu().numpy(), x.grad.cpu().numpy()))
    np.testing.assert_array_equal(outs[0][0], outs[1][0])
    np.testing.assert_array_equal(outs[0][1], outs[1][1])
    fin = np.isfinite(want_nll)
    np.testing.assert_allclose(outs[0][0][fin], want_nll[fin], rtol=LOSS_REL_TOL)
    assert outs[0][0][2] == np.inf
    ok = ~np.isnan(want_g)
    assert np.abs(outs[0][1][ok] - want_g[ok]).max() <= GRAD_ABS_TOL


def test_ctc_loss_errors_and_empty_batch(A):
    x = torch.zeros((2, 5, 4), device="cuda")
    t = torch.ones((2, 2), dtype=torch.int32)
    with pytest.raises(ValueError):
        A.ctc_loss(x[0], t, [5, 5], [2, 2])
    with pytest.raises(ValueError):
        A.ctc_loss(x, t, [5, 5], [2, 2], reduction="avg")
    with pytest.raises(ValueError):
        A.ctc_loss(x, t[0], [5, 5], [2, 2])
    with pytest.raises(RuntimeError, match="vocab"):
        A.ctc_loss(torch.zeros((2, 5, 65), device="cuda"), t, [5, 5], [2, 2])
    with pytest.raises(RuntimeError, match="n_steps"):
        A.ctc_loss(torch.zeros((2, 1025, 4), device="cuda"), t, [5, 5], [2, 2])
    e = torch.zeros((0, 5, 4), device="cuda", requires_grad=True)
    loss = A.ctc_loss(e, torch.zeros((0, 2), dtype=torch.int32), torch.zeros(0), torch.zeros(0), reduction="sum")
    loss.backward()
    assert float(loss) == 0 and e.grad.shape == (0, 5, 4)


# ---------------------------------------------------------------------------------------------------- K3 train / K3b
def make_net(A, H, precision, seed=0):
    sd = lipnet_ref.init_lipnet_state(39, H, seed=seed)
    net = A.LipNet(39, hidden_dim=H, precision=precision)
    net.load_state_dict(sd)
    return net.cuda(), sd


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("H", [256, 128])
def test_train_forward_equals_gru_head_bit_for_bit(A, precision, H):
    net, _ = make_net(A, H, precision)
    emb = torch.randn((17, 75, 6912), device="cuda") * 0.05
    net.eval()
    with torch.no_grad():
        want = net.gru_head(emb)
    got = net.gru_head_train(emb)
    assert got.grad_fn is not None
    torch.testing.assert_close(got.detach(), want, rtol=0, atol=0)
    net.train()
    got = net.gru_head_train(emb)
    torch.testing.assert_close(got.detach(), want, rtol=0, atol=0)


def head_grads(A, net, emb, targets, il, lens, p, seed):
    torch.manual_seed(seed)
    for q in net.parameters():
        q.grad = None
    lp = net.gru_head_train(emb, dropout=p)
    A.ctc_loss(lp, targets, il, lens, zero_infinity=True).backward()
    return lp, {n: q.grad.detach().clone() for n, q in net.named_parameters() if q.grad is not None}


def masks_of(seed, p, B, T, H):
    """The keep masks gru_head_train draws under torch.manual_seed(seed)."""
    if p == 0:
        return (None, None)
    torch.manual_seed(seed)
    return tuple(torch.empty((B, T, 2 * H), dtype=torch.uint8, device="cuda").bernoulli_(1.0 - p) for _ in range(2))


GRAD_CASES = [  # (H, precision, B, T, dropout): 256 runs the tcgen05 (bf16x3) and cluster (fp32) forwards, others the generic
    (256, "bf16x3", 17, 75, 0.5), (256, "fp32", 64, 75, 0.0), (32, "fp32", 1, 1, 0.0), (32, "bf16x3", 64, 200, 0.3),
    (128, "bf16x3", 17, 75, 0.5), (128, "fp32", 1, 200, 0.0), (1024, "fp32", 1, 75, 0.5), (1024, "bf16x3", 17, 1, 0.0),
    (512, "fp32", 5, 75, 0.9), (512, "bf16x3", 4, 75, 0.9), (256, "bf16", 17, 75, 0.3)]


@pytest.mark.parametrize("H,precision,B,T,p", GRAD_CASES)
def test_head_gradients_vs_float64(A, c2i, H, precision, B, T, p):
    net, sd = make_net(A, H, precision, seed=H + B)
    rng = np.random.default_rng(H * 7 + B + T)
    emb = torch.from_numpy(rng.normal(size=(B, T, 6912)).astype(np.float32) * 0.05).cuda()
    _, targets, lens = ctc_align_ref.grid_targets(B, c2i, seed=B + T)
    lens = np.minimum(lens, max(T // 2, 0)).astype(np.int32)   # feasible at every T (T = 1: empty targets)
    il = np.full(B, T, np.int32)
    il[: B // 2] = np.maximum(1, T - rng.integers(0, T // 4 + 1, B // 2))
    targets, lens, il = (torch.from_numpy(a).cuda() for a in (targets, lens, il))
    _, got = head_grads(A, net, emb, targets, il, lens, p, seed=11)
    masks = masks_of(11, p, B, T, H)
    lp64, mods = R.head_reference(sd, emb, masks, p)
    F.ctc_loss(lp64.transpose(0, 1), targets.long(), il.long(), lens.long(), zero_infinity=True).backward()
    want = {f"{name}.{k}": q.grad for name, m in zip(("gru1", "gru2", "fc"), mods) for k, q in m.named_parameters()}
    assert sorted(got) == sorted(NAMES)
    errs = {n: float((got[n].double() - want[n]).abs().max() / want[n].abs().max().clamp(min=1e-30)) for n in NAMES}
    worst = max(errs, key=errs.get)
    print(f"H={H} {precision} B={B} T={T} p={p}: worst {worst} {errs[worst]:.3e}")
    assert errs[worst] <= HEAD_GRAD_TOL[precision], errs


def test_two_runs_bit_identical(A, c2i):
    net, _ = make_net(A, 256, "bf16x3", seed=5)
    emb = torch.randn((17, 75, 6912), device="cuda") * 0.05
    _, targets, lens = ctc_align_ref.grid_targets(17, c2i, seed=5)
    args = (torch.from_numpy(targets).cuda(), torch.full((17,), 75, device="cuda"), torch.from_numpy(lens).cuda())
    lp0, g0 = head_grads(A, net, emb, *args, p=0.5, seed=3)
    lp1, g1 = head_grads(A, net, emb, *args, p=0.5, seed=3)
    torch.testing.assert_close(lp0, lp1, rtol=0, atol=0)
    for n in NAMES:
        torch.testing.assert_close(g0[n], g1[n], rtol=0, atol=0)


def test_train_errors_and_empty_batch(A):
    net, _ = make_net(A, 32, "fp32")
    emb = torch.zeros((2, 5, 6912), device="cuda")
    with pytest.raises(ValueError, match="requires grad"):
        net.gru_head_train(emb.clone().requires_grad_())
    with pytest.raises(ValueError):
        net.gru_head_train(emb, dropout=1.0)
    with pytest.raises(ValueError):
        net.gru_head_train(torch.zeros((2, 5, 100), device="cuda"))
    with pytest.raises(RuntimeError):
        net.gru_head_train(emb.cpu())
    lp = net.gru_head_train(torch.zeros((0, 5, 6912), device="cuda"), dropout=0.5)
    assert lp.shape == (0, 5, 39)
    lp.sum().backward()
    for n, q in net.named_parameters():
        if n.startswith(("gru", "fc")):
            assert q.grad is not None and not q.grad.any(), n
    net.eval()   # eval-mode forward still refuses training mode; gru_head_train does not care
    net.train()
    with pytest.raises(RuntimeError):
        net.gru_head(emb)


def synth_grid(c2i, n, seed):
    """Embeddings that encode GRID sentences: frame 2i carries a code vector of the sentence's i-th character, the other
    frames the blank's, plus noise."""
    rng = np.random.default_rng(seed)
    code = rng.normal(size=(39, 6912)) * 0.05
    sents = ctc_beam_ref.grid_sentences(n, seed)
    lab = np.zeros((n, 75), np.int64)
    targets = np.zeros((n, 40), np.int32)
    for b, s in enumerate(sents):
        ids = [c2i[ch] for ch in s]
        lab[b, 0:2 * len(ids):2] = ids
        targets[b, :len(ids)] = ids
    emb = code[lab] + rng.normal(size=(n, 75, 6912)) * 0.01
    return sents, torch.from_numpy(emb.astype(np.float32)).cuda(), torch.from_numpy(targets).cuda(), \
        torch.tensor([len(s) for s in sents], dtype=torch.int32).cuda()


def test_training_run_learns_grid_sentences(A, c2i):
    from avsync_b200.dataset import create_vocab
    i2c = create_vocab()[1]
    torch.manual_seed(0)
    net, _ = make_net(A, 64, "bf16x3", seed=0)
    sents, emb, targets, lens = synth_grid(c2i, 8, seed=3)
    head = [q for n, q in net.named_parameters() if n.startswith(("gru", "fc"))]
    opt = torch.optim.Adam(head, lr=3e-3)
    il = torch.full((8,), 75, dtype=torch.int32, device="cuda")
    losses = []
    for _ in range(100):
        lp = net.gru_head_train(emb)
        loss = A.ctc_loss(lp, targets, il, lens, zero_infinity=True)
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(head, 1.0)
        opt.step()
        losses.append(float(loss))
    print(f"loss {losses[0]:.3f} -> {losses[-1]:.4f}")
    assert losses[-1] < 0.05 * losses[0]
    ids, n = A.ctc_greedy_decode(net.gru_head_train(emb).detach())
    got = ["".join(i2c[int(i)] for i in ids[b, :int(n[b])]) for b in range(8)]
    assert got == sents
