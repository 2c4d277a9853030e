"""CTC forced alignment (K5c) without a device: the float64 oracle against torch's CTC loss, torchaudio's forced aligner
and merge_tokens, and brute-force enumeration; the GRID .align reader; the argument checks of avs_ctc_align and
avs_ctc_align_workspace_bytes (include/avsync.h), which run before any CUDA call."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import ctc_align_ref as R

FAKE = ctypes.c_void_p(256)     # never dereferenced: every call below fails its argument checks first


def rand_logp(rng, T, V, scale=2.0):
    x = rng.normal(size=(T, V)) * scale
    return x - np.logaddexp.reduce(x, axis=1, keepdims=True)


def ctc_loss(lp, y, n=None):
    T = lp.shape[0]
    return float(torch.nn.functional.ctc_loss(torch.from_numpy(lp)[:, None], torch.tensor([list(y) or [1]]),
                                              torch.tensor([T if n is None else n]), torch.tensor([len(y)]), blank=0,
                                              reduction="none", zero_infinity=False)[0])


CASES = [  # (T, V, y, input_len): repeated labels, input_len < T, L = 0, infeasible targets
    (10, 5, [1, 2, 2], None), (12, 4, [3, 3, 3], None), (6, 4, [3, 3, 3], None), (5, 4, [3, 3, 3], None),
    (20, 6, [1, 1, 2, 1, 1], 11), (20, 6, [1, 1, 2, 1, 1], 8), (7, 3, [], None), (7, 3, [], 3), (7, 3, [1], 0),
    (7, 3, [], 0), (1, 2, [1], None), (1, 2, [1, 1], None), (3, 2, [1, 1], None), (75, 39, [5, 12, 12, 15], 40)]


@pytest.mark.parametrize("T,V,y,n", CASES)
def test_loglik_equals_minus_ctc_loss(T, V, y, n):
    lp = rand_logp(np.random.default_rng(T * 31 + V), T, V)
    want = -ctc_loss(lp, y, n)
    got = R.align(lp, y, n)
    if np.isinf(want):
        assert got.loglik == got.path_score == -np.inf
        assert (got.frame_token == -2).all() and (got.span == -1).all() and np.isnan(got.token_prob).all()
    else:
        assert abs(got.loglik - want) <= 1e-10 * max(1.0, abs(want))
        assert got.path_score <= got.loglik
        assert ((got.frame_token[n if n is not None else T:]) == -2).all()


@pytest.mark.parametrize("seed", range(30))
def test_loglik_on_random_targets(seed):
    rng = np.random.default_rng(1000 + seed)
    T, V = int(rng.integers(1, 80)), int(rng.integers(2, 40))
    L = int(rng.integers(0, 12))
    y = rng.integers(1, V, L) if rng.random() < 0.5 else np.repeat(rng.integers(1, V, (L + 1) // 2), 2)[:L]
    n = int(rng.integers(0, T + 1))
    lp = rand_logp(rng, T, V)
    want, got = -ctc_loss(lp, y, n), R.align(lp, y, n).loglik
    assert (np.isinf(want) and got == -np.inf) or abs(got - want) <= 1e-10 * max(1.0, abs(want)), (got, want)


def _torchaudio():   # imported per test, so that only these tests skip without torchaudio
    F = pytest.importorskip("torchaudio.functional")
    if not hasattr(F, "forced_align"):
        pytest.skip("this torchaudio has no forced_align")
    return F


def aligned_cases(n, seed):
    """(logp, y, input_len) with continuous random log-probs (no exact ties) and a feasible target."""
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        T, V = int(rng.integers(2, 80)), int(rng.integers(3, 40))
        L = int(rng.integers(1, 15))
        y = rng.integers(1, V, L)
        if rng.random() < 0.3:
            y[1::2] = y[0::2][:len(y[1::2])]          # repeated labels
        nin = int(rng.integers(1, T + 1))
        if nin < L + int((y[1:] == y[:-1]).sum()):
            continue
        out.append((rand_logp(rng, T, V, 3.0), y, nin))
    return out


def test_viterbi_path_and_score_equal_torchaudio_forced_align():
    F = _torchaudio()
    for lp, y, n in aligned_cases(60, 7):
        r = R.align(lp, y, n)
        labels, scores = F.forced_align(torch.from_numpy(lp[:n])[None], torch.tensor(y[None], dtype=torch.int32),
                                        torch.tensor([n]), torch.tensor([len(y)]), blank=0)
        want = np.where(r.frame_token[:n] >= 0, y[np.maximum(r.frame_token[:n], 0)], 0)
        np.testing.assert_array_equal(labels[0].numpy(), want)
        assert abs(float(scores.sum()) - r.path_score) <= 1e-10 * max(1.0, abs(r.path_score))


def test_spans_and_scores_equal_torchaudio_merge_tokens():
    F = _torchaudio()
    for lp, y, n in aligned_cases(60, 8):
        r = R.align(lp, y, n)
        labels, scores = F.forced_align(torch.from_numpy(lp[:n])[None], torch.tensor(y[None], dtype=torch.int32),
                                        torch.tensor([n]), torch.tensor([len(y)]), blank=0)
        spans = F.merge_tokens(labels[0], scores[0].exp(), blank=0)
        assert [s.token for s in spans] == list(y)
        np.testing.assert_array_equal(r.span, [[s.start, s.end] for s in spans])
        np.testing.assert_allclose(r.token_prob, [s.score for s in spans], rtol=1e-12, atol=0)


@pytest.mark.parametrize("seed", range(40))
def test_oracle_equals_brute_force(seed):
    rng = np.random.default_rng(2000 + seed)
    T, V = int(rng.integers(1, 9)), int(rng.integers(2, 5))
    L = int(rng.integers(0, 4))
    y = rng.integers(1, V, L)
    lp = rand_logp(rng, T, V)
    ll, ps, ft = R.brute_force(lp, y)
    r = R.align(lp, y)
    assert r.path_score == ps                  # the same adds in the same order
    np.testing.assert_array_equal(r.frame_token, ft)
    assert (ll == r.loglik == -np.inf) or abs(ll - r.loglik) <= 1e-12


def test_uniform_rows_follow_the_tie_rule():
    """All paths tie: the backtrace stays wherever it can, so the trailing blank holds every frame it can reach and
    each token sits as early as its successors allow."""
    lp = np.full((6, 3), np.log(1 / 3))
    r = R.align(lp, [1, 2])
    np.testing.assert_array_equal(r.frame_token, [0, 1, -1, -1, -1, -1])
    r = R.align(lp, [1, 1])       # a repeated label needs a blank between
    np.testing.assert_array_equal(r.frame_token, [0, -1, 1, -1, -1, -1])
    r = R.align(lp[:2], [1, 2])
    np.testing.assert_array_equal(r.frame_token, [0, 1])


def test_statuses_of_invalid_clips_and_nan():
    lp = rand_logp(np.random.default_rng(3), 10, 5)
    for y, n in (([1, 5], None), ([1, 0], None), ([-1], None), ([1], 11), ([1], -1)):
        r = R.align(lp, y, n)
        assert np.isnan(r.loglik) and np.isnan(r.path_score) and (r.frame_token == -2).all()
    holes = lp.copy()
    holes[4, :] = np.nan
    assert R.align(holes, [1, 2]).loglik == -np.inf
    holes = lp.copy()
    holes[4, 3] = np.nan
    a, b = R.align(holes, [1, 2]), R.align(np.where(np.isnan(holes), -np.inf, holes), [1, 2])
    assert a.loglik == b.loglik and (a.frame_token == b.frame_token).all()
    ll, ps, ft, span, prob = R.align_batch(lp[None].repeat(2, 0), np.array([[1, 2], [1, 2]]), [3, 2])
    assert np.isnan(ll[0]) and np.isfinite(ll[1]) and (span[0] == -1).all() and (span[1] >= 0).all()


def test_read_grid_align(tmp_path):
    from avsync_b200.dataset import read_grid_align
    p = tmp_path / "bbaf2n.align"
    p.write_text("0 23750 sil\n23750 29500 bin\n29500 34000 blue\n34000 35500 at\n35500 41000 f\n"
                 "41000 47250 two\n47250 53000 sp\n53000 55500 now\n55500 74500 sil\n")
    text, words = read_grid_align(str(p))
    assert text == "bin blue at f two now"
    assert words == [("bin", 23.75, 29.5), ("blue", 29.5, 34.0), ("at", 34.0, 35.5), ("f", 35.5, 41.0),
                     ("two", 41.0, 47.25), ("now", 53.0, 55.5)]
    bad = tmp_path / "bad.align"
    bad.write_text("0 100\n")
    with pytest.raises(ValueError):
        read_grid_align(str(bad))


# ---------------------------------------------------------------- argument checks through ctypes, no device needed

@pytest.fixture(scope="module")
def native():
    import avsync_b200
    N = avsync_b200._native
    if not os.path.isfile(N.LIB_PATH):
        N.build()
    return N


def test_align_rejects_bad_arguments_without_a_device(native):
    L = native.lib()

    def call(n_clips=4, n_steps=75, vocab=39, blank=0, stride=40, ws_bytes=1 << 40, out=FAKE, ws=FAKE):
        rc = L.avs_ctc_align(FAKE, n_clips, n_steps, vocab, blank, None, FAKE, stride, FAKE, out, out, out, out, out,
                             ws, ws_bytes, None)
        return rc, L.avs_last_error_string().decode()

    for kw, text in (({"n_steps": 0}, "n_steps must be in [1, 1024]"), ({"n_steps": 1025}, "n_steps must be in [1, 1024]"),
                     ({"vocab": 1}, "vocab must be in [2, 64]"), ({"vocab": 65}, "vocab must be in [2, 64]"),
                     ({"blank": -1}, "blank must be in [0, vocab)"), ({"blank": 39}, "blank must be in [0, vocab)"),
                     ({"stride": -1}, "target_stride must be in [0, 512]"),
                     ({"stride": 513}, "target_stride must be in [0, 512]"),
                     ({"n_clips": -1}, "n_clips"), ({"out": None}, "null argument")):
        rc, msg = call(**kw)
        assert rc == -1 and text in msg, (kw, msg)
    rc, msg = call(n_steps=1024, stride=512, ws_bytes=1 << 20)
    assert rc == -4 and "workspace too small" in msg
    rc, msg = call(n_steps=1024, stride=512, ws=None)
    assert rc == -4 and "workspace too small" in msg
    assert call(n_clips=0, out=None)[0] == 0          # an empty batch needs no buffers and launches nothing


def test_align_workspace_bytes(native):
    L = native.lib()
    # GRID clips keep their backpointers (one byte per frame and state) in shared memory
    assert L.avs_ctc_align_workspace_bytes(4096, 75, 40) == 0
    assert L.avs_ctc_align_workspace_bytes(1, 32, 511) == 0                 # 32 * 1023 bytes < 32 KB
    per_clip = L.avs_ctc_align_workspace_bytes(1, 1024, 512)
    assert per_clip >= 1024 * 1025 and L.avs_ctc_align_workspace_bytes(7, 1024, 512) == 7 * per_clip
    assert L.avs_ctc_align_workspace_bytes(1, 33, 511) >= 33 * 1023
    for args in ((-1, 75, 40), (1, 0, 40), (1, 1025, 40), (1, 75, -1), (1, 1024, 513)):
        assert L.avs_ctc_align_workspace_bytes(*args) == 0
