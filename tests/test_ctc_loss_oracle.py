"""CTC loss and gradient (K5e) without a device: the float64 restatement of alpha / beta / gamma (oracle/ctc_loss_ref.py)
against torch.nn.functional.ctc_loss in float64, losses and gradients (compared as gradients of the logits under
log_softmax), over repeats, L = 0, short inputs, infeasible clips, each reduction and zero_infinity."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ctc_loss_ref as R


def torch_ref(logits, targets, in_lens, tgt_lens, reduction="none", zero_infinity=False):
    """torch's loss in float64 and its gradient with respect to the logits (under log_softmax)."""
    x = torch.tensor(logits, dtype=torch.float64, requires_grad=True)
    lp = torch.log_softmax(x, dim=-1)
    loss = F.ctc_loss(lp.transpose(0, 1), torch.as_tensor(targets, dtype=torch.long), torch.as_tensor(in_lens),
                      torch.as_tensor(tgt_lens), blank=0, reduction=reduction, zero_infinity=zero_infinity)
    loss.sum().backward()
    return loss.detach().numpy(), x.grad.numpy(), lp.detach().numpy()


def logits_grad(lp, g):   # dL/dlogits from dL/dlogp under log_softmax
    return g - np.exp(lp) * g.sum(-1, keepdims=True)


CASES = [  # (T, V, y, input_len): repeats, input_len < T, L = 0, infeasible, T = 1
    (10, 5, [1, 2, 2], 10), (12, 4, [3, 3, 3], 12), (6, 4, [3, 3, 3], 6), (20, 6, [1, 1, 2, 1, 1], 11),
    (7, 3, [], 7), (7, 3, [], 3), (1, 2, [1], 1), (3, 2, [1, 1], 3), (75, 39, [5, 12, 12, 15], 40),
    (9, 5, [4, 4, 4, 4], 9), (5, 4, [3, 3, 3], 5), (4, 5, [1, 2, 3], 2)]


@pytest.mark.parametrize("T,V,y,n", CASES)
@pytest.mark.parametrize("zero_infinity", [False, True])
def test_loss_and_gradient_equal_torch(T, V, y, n, zero_infinity):
    rng = np.random.default_rng(T * 31 + V + len(y))
    logits = rng.normal(size=(1, T, V)) * 2.0
    targets = np.array([list(y) or [1]])
    want_loss, want_g, lp = torch_ref(logits, targets, [n], [len(y)], zero_infinity=zero_infinity)
    nll, g = R.loss_grad(lp[0], y, n, zero_infinity=zero_infinity)
    if np.isinf(want_loss[0]):
        assert nll == np.inf and np.isnan(g[:n]).all() and (g[n:] == 0).all()
        return
    assert abs(nll - want_loss[0]) <= 1e-10 * max(1.0, abs(want_loss[0]))
    if not zero_infinity or want_loss[0] != 0 or len(y) == 0:
        np.testing.assert_allclose(logits_grad(lp[0], g), want_g[0], rtol=0, atol=1e-10)
    assert (g[n:] == 0).all()
    if nll > 0 or len(y) == 0:   # gamma sums to 1 at every frame inside input_len
        np.testing.assert_allclose(-g[:n].sum(-1), 1.0, atol=1e-12)


@pytest.mark.parametrize("reduction", ["none", "sum", "mean"])
def test_reductions_match_torch(reduction):
    rng = np.random.default_rng(7)
    B, T, V, Lmax = 6, 30, 8, 6
    logits = rng.normal(size=(B, T, V))
    tl = np.array([6, 0, 3, 1, 5, 4])
    il = np.array([30, 12, 4, 30, 25, 2])   # clip 5: 4 labels in 2 frames, infeasible
    targets = rng.integers(1, V, size=(B, Lmax))
    for zi in (False, True):
        want, want_g, lp = torch_ref(logits, targets, il, tl, reduction, zi)
        nll, _ = R.loss_grad_batch(lp, targets, tl, il, zero_infinity=zi)
        w = {"none": np.ones(B), "sum": np.ones(B), "mean": 1.0 / (np.maximum(tl, 1) * B)}[reduction]
        _, g = R.loss_grad_batch(lp, targets, tl, il, scale=w, zero_infinity=zi)
        red = {"none": nll, "sum": nll.sum(), "mean": (nll / np.maximum(tl, 1)).mean()}[reduction]
        if not zi:
            assert np.isinf(red).any() if reduction != "none" else np.isinf(red[5])
            continue
        np.testing.assert_allclose(red, want, rtol=1e-12)
        np.testing.assert_allclose(logits_grad(lp, g), want_g, rtol=0, atol=1e-12)


def test_mean_divides_by_clamped_target_length():
    # an L = 0 clip divides its loss by 1, not 0
    lp = np.log(np.full((1, 5, 3), 1 / 3))
    nll, _ = R.loss_grad(lp[0], [], 5)
    assert nll == pytest.approx(5 * np.log(3))
    want, _, _ = torch_ref(np.zeros((1, 5, 3)), np.array([[1]]), [5], [0], "mean")
    assert float(want) == pytest.approx(nll / max(0, 1))


def test_statuses():
    lp = np.log(np.full((6, 4), 0.25))
    nll, g = R.loss_grad(lp, [1, 4], 6)           # id out of range
    assert np.isnan(nll) and np.isnan(g).all()
    nll, g = R.loss_grad(lp, [0, 1], 6)           # the blank as a label
    assert np.isnan(nll) and np.isnan(g).all()
    nll, g = R.loss_grad(lp, [1], 7)              # input_len > T
    assert np.isnan(nll) and np.isnan(g).all()
    bad = lp.copy()
    bad[2, 3] = np.nan                            # a NaN inside input_len, even on a label the target does not use
    nll, g = R.loss_grad(bad, [1, 2], 4)
    assert np.isnan(nll) and np.isnan(g[:4]).all() and (g[4:] == 0).all()
    nll, g = R.loss_grad(bad, [1, 2], 2)          # ... but not past it
    assert np.isfinite(nll) and np.isfinite(g).all()
    nll, g = R.loss_grad(lp, [1, 1, 1], 4)        # needs 5 frames
    assert nll == np.inf and np.isnan(g[:4]).all() and (g[4:] == 0).all()
    nll, g = R.loss_grad(lp, [1, 1, 1], 4, zero_infinity=True)
    assert nll == 0 and (g == 0).all()
