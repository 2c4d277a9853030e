"""CTC forced alignment (K5c, csrc/ctc_align.cu) on the B200 against the float64 oracle (oracle/ctc_align_ref.py),
torch's CUDA ctc_loss and brute-force enumeration; the tie rule, statuses, corners, NaN, determinism, error paths and
align_words."""
import numpy as np
import pytest
import torch

from oracle import ctc_align_ref as R
from oracle import ctc_beam_ref

pytestmark = pytest.mark.gpu

# Largest relative error measured on an NVIDIA B200 (1000 W power limit) over the cases below: 5.9e-8 for loglik and
# token_prob against the float64 oracle, 5.5e-8 for loglik against torch's CUDA ctc_loss in float64.  The kernel runs in
# fp64, so that is the fp32 rounding of its outputs (at most 2^-24 = 6.0e-8).  The tolerance is twice that error.
REL_TOL = 1.2e-7


@pytest.fixture(scope="module")
def A():
    import avsync_b200
    avsync_b200._native.device_check()
    return avsync_b200


@pytest.fixture(scope="module")
def c2i():
    from avsync_b200.dataset import create_vocab
    return create_vocab()[0]


def run(A, lp, targets, lens, input_lens=None, blank=0):
    dev = lambda x: None if x is None else torch.as_tensor(np.asarray(x)).cuda()   # noqa: E731
    out = A.ctc_forced_align(torch.from_numpy(np.ascontiguousarray(lp)).cuda(), dev(targets), dev(lens),
                             dev(input_lens), blank)
    return tuple(t.cpu().numpy() for t in out)


def rel_err(got, want, floor=1.0):
    fin = np.isfinite(want)
    assert np.array_equal(fin, np.isfinite(got)) and np.array_equal(np.isnan(want), np.isnan(got))
    assert np.array_equal(np.sign(want[~fin & ~np.isnan(want)]), np.sign(got[~fin & ~np.isnan(got)]))
    if not fin.any():
        return 0.0
    err = np.abs(got[fin].astype(np.float64) - want[fin]) / np.maximum(np.abs(want[fin]), floor)
    return float(err.max())


def assert_matches_oracle(got, want, floor_prob=0.0):
    ll, ps, ft, span, prob = got
    o_ll, o_ps, o_ft, o_span, o_prob = want
    np.testing.assert_array_equal(ft, o_ft)
    np.testing.assert_array_equal(span, o_span)
    np.testing.assert_array_equal(ps, o_ps.astype(np.float32))      # the same fp64 adds, rounded once
    e_ll, e_prob = rel_err(ll, o_ll), rel_err(prob, o_prob, floor=floor_prob)
    assert e_ll <= REL_TOL and e_prob <= REL_TOL, (e_ll, e_prob)
    return e_ll, e_prob


def grid_batch(c2i, n, seed):
    """n GRID-shaped clips (T = 75, V = 39): GRID sentence targets (Lmax 40, zero-padded), the first half over
    log-probs of those sentences being spoken (ctc_beam_ref.grid_sentence_logp), the second half over unrelated peaked
    log-probs; random input lengths, some too short for their sentence."""
    sentences, targets, lens = R.grid_targets(n, c2i, seed=seed, lmax=40)
    spoken = ctc_beam_ref.grid_sentence_logp(sentences[:n // 2], c2i, seed=seed + 1)
    lp = np.concatenate([spoken, ctc_beam_ref.peaked_logp(n - n // 2, 75, 39, seed=seed + 2)])
    input_lens = np.random.default_rng(seed + 3).integers(16, 76, n).astype(np.int32)
    return lp, targets, lens, input_lens


def test_grid_clips_vs_oracle(A, c2i):
    lp, targets, lens, input_lens = grid_batch(c2i, 1024, 0)
    got = run(A, lp, targets, lens, input_lens)
    want = R.align_batch(lp, targets, lens, input_lens)
    e_ll, e_prob = assert_matches_oracle(got, want)
    n_inf = int(np.isneginf(want[0]).sum())
    assert 50 <= n_inf <= 500, n_inf          # some inputs are too short for their sentence
    print(f"1024 GRID clips, {n_inf} without an alignment: max rel err loglik {e_ll:.2e}, token_prob {e_prob:.2e}")


def test_loglik_equals_torch_cuda_ctc_loss(A, c2i):
    lp, targets, lens, input_lens = grid_batch(c2i, 512, 10)
    ll = run(A, lp, targets, lens, input_lens)[0]
    loss = torch.nn.functional.ctc_loss(torch.from_numpy(lp).cuda().double().transpose(0, 1),
                                        torch.from_numpy(targets).cuda().long(), torch.from_numpy(input_lens).cuda(),
                                        torch.from_numpy(lens).cuda(), blank=0, reduction="none", zero_infinity=False)
    want = -loss.cpu().numpy()
    err = rel_err(ll, want)
    assert err <= REL_TOL, err
    print(f"max rel err against torch's CUDA ctc_loss (float64): {err:.2e}")


def test_brute_force_on_the_gpu(A):
    rng = np.random.default_rng(20)
    for _ in range(40):
        T, V = int(rng.integers(1, 9)), int(rng.integers(2, 5))
        L = int(rng.integers(0, 4))
        y = rng.integers(1, V, L).astype(np.int32)
        x = rng.normal(size=(T, V)) * 2.0
        lp = (x - np.logaddexp.reduce(x, axis=1, keepdims=True)).astype(np.float32)
        b_ll, b_ps, b_ft = R.brute_force(lp, y)
        ll, ps, ft, span, _ = run(A, lp[None], y[None].reshape(1, L), [L])
        np.testing.assert_array_equal(ft[0], b_ft)
        assert ps[0] == np.float32(b_ps)
        assert (b_ll == ll[0] == -np.inf) or abs(ll[0] - b_ll) <= REL_TOL * max(1.0, abs(b_ll))


def test_exact_ties_follow_the_tie_rule(A):
    """Uniform rows: every path of a target ties.  The backtrace takes the stay, then s-1, then s-2, and ends in the
    trailing blank, so each token sits as early as the tokens after it allow."""
    rng = np.random.default_rng(21)
    cases = [(6, 3, [1, 2], [0, 1, -1, -1, -1, -1]), (6, 3, [1, 1], [0, -1, 1, -1, -1, -1]), (2, 3, [1, 2], [0, 1]),
             (3, 3, [2, 2], [0, -1, 1]), (4, 2, [], [-1, -1, -1, -1])]
    for _ in range(30):
        T, V = int(rng.integers(1, 20)), int(rng.integers(2, 6))
        y = list(rng.integers(1, V, int(rng.integers(0, 6))))
        cases.append((T, V, y, None))
    for T, V, y, want_ft in cases:
        for lp in (np.full((T, V), np.log(1.0 / V), np.float32), np.zeros((T, V), np.float32)):
            y32 = np.asarray(y, np.int32).reshape(1, len(y))
            got = run(A, lp[None], y32, [len(y)])
            assert_matches_oracle(got, R.align_batch(lp[None], y32, [len(y)]))
            if want_ft is not None:
                np.testing.assert_array_equal(got[2][0], want_ft)


def test_corners_and_invalid_clips_next_to_valid_ones(A, c2i):
    lp = ctc_beam_ref.peaked_logp(10, 75, 39, seed=22)
    _, targets, lens = R.grid_targets(10, c2i, seed=22, lmax=40)
    input_lens = np.full(10, 75, np.int32)
    lens[1] = 0                                  # empty target
    input_lens[2] = 0                            # no frames, non-empty target: no alignment
    lens[3], input_lens[3] = 0, 0                # no frames, empty target: probability 1
    targets[4, 3] = 39                           # id outside the vocabulary
    targets[5, 0] = 0                            # the blank
    lens[6] = 41                                 # longer than the stride
    lens[7] = -1
    input_lens[8] = 76                           # longer than the clip
    targets[9, :4] = 7                           # "gggg" needs 7 frames
    input_lens[9] = 6
    lens[9] = 4
    got = run(A, lp, targets, lens, input_lens)
    want = R.align_batch(lp, targets, lens, input_lens)
    assert_matches_oracle(got, want)
    ll, ps, ft, span, prob = got
    assert ll[0] < 0 and np.isfinite(ll[0]) and ll[1] < 0 and (ft[1] == -1).all()
    assert ll[3] == ps[3] == 0 and (ft[3] == -2).all()
    assert np.isneginf(ll[[2, 9]]).all() and np.isneginf(ps[[2, 9]]).all()
    assert np.isnan(ll[4:9]).all() and np.isnan(ps[4:9]).all()
    assert (ft[[2, 4, 5, 6, 7, 8, 9]] == -2).all() and (span[[2, 4, 5, 6, 7, 8, 9]] == -1).all()
    assert np.isnan(prob[[2, 4, 5, 6, 7, 8, 9]]).all()
    # the valid clip is unaffected by its neighbours
    solo = run(A, lp[:1], targets[:1], lens[:1], input_lens[:1])
    for a, b in zip(got, solo):
        assert np.array_equal(a[:1], b, equal_nan=np.issubdtype(a.dtype, np.floating))
    # no targets at all (Lmax 0)
    ll0, ps0, ft0, span0, prob0 = run(A, lp[:3], np.zeros((3, 0), np.int32), [0, 0, 0], [75, 10, 0])
    assert span0.shape == (3, 0, 2) and prob0.shape == (3, 0)
    np.testing.assert_allclose(ll0[:2], [lp[0, :, 0].astype(np.float64).sum(), lp[1, :10, 0].astype(np.float64).sum()],
                               rtol=REL_TOL)
    assert ll0[2] == 0 and (ft0[0] == -1).all() and (ft0[1, 10:] == -2).all()


def test_longest_clip_and_target(A):
    """T = 1024 and L = 512: the backpointers (1 MB per clip) live in the workspace."""
    rng = np.random.default_rng(23)
    lp = ctc_beam_ref.peaked_logp(3, 1024, 64, seed=23)
    targets = rng.integers(1, 64, (3, 512)).astype(np.int32)
    targets[2, 1::2] = targets[2, 0::2]          # 256 repeated pairs: needs 768 frames
    lens = np.array([512, 300, 512], np.int32)
    got = run(A, lp, targets, lens, [1024, 1000, 1024])
    assert_matches_oracle(got, R.align_batch(lp, targets, lens, [1024, 1000, 1024]))
    assert np.isfinite(got[0]).all()
    lp = ctc_beam_ref.peaked_logp(2, 1024, 39, seed=24)
    got = run(A, lp, targets[:2] % 38 + 1, [512, 20], [1024, 1024])
    assert_matches_oracle(got, R.align_batch(lp, targets[:2] % 38 + 1, [512, 20], [1024, 1024]))


def test_nan_counts_as_minus_infinity(A, c2i):
    lp, targets, lens, input_lens = grid_batch(c2i, 64, 30)
    rng = np.random.default_rng(25)
    holes = lp.copy()
    holes[rng.random(holes.shape) < 0.05] = np.nan
    as_inf = np.where(np.isnan(holes), -np.inf, holes).astype(np.float32)
    a, b = run(A, holes, targets, lens, input_lens), run(A, as_inf, targets, lens, input_lens)
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)
    assert_matches_oracle(a, R.align_batch(holes, targets, lens, input_lens))
    assert np.isfinite(a[0]).sum() >= 32
    dead = lp[:2].copy()
    dead[:, 30, :] = np.nan                      # a frame where nothing is possible
    ll, ps, ft, _, _ = run(A, dead, targets[:2], lens[:2])
    assert np.isneginf(ll).all() and np.isneginf(ps).all() and (ft == -2).all()


def test_batch_equals_solo_and_runs_repeat_bit_for_bit(A, c2i):
    lp, targets, lens, input_lens = grid_batch(c2i, 96, 40)
    full, again = run(A, lp, targets, lens, input_lens), run(A, lp, targets, lens, input_lens)
    for x, y in zip(full, again):
        assert np.array_equal(x, y, equal_nan=True)
    for c in (0, 47, 48, 95):
        solo = run(A, lp[c:c + 1], targets[c:c + 1], lens[c:c + 1], input_lens[c:c + 1])
        for x, y in zip(full, solo):
            assert np.array_equal(x[c:c + 1], y, equal_nan=True)


def test_error_paths_and_empty_batch(A, c2i):
    lp = torch.from_numpy(ctc_beam_ref.peaked_logp(2, 75, 39, seed=1)).cuda()
    tg = torch.ones((2, 5), dtype=torch.int32, device="cuda")
    tl = torch.full((2,), 5, dtype=torch.int32, device="cuda")
    with pytest.raises(RuntimeError, match="blank"):
        A.ctc_forced_align(lp, tg, tl, blank_index=39)
    with pytest.raises(RuntimeError, match="n_steps"):
        A.ctc_forced_align(torch.zeros((1, 1025, 39), device="cuda"), tg[:1], tl[:1])
    with pytest.raises(RuntimeError, match="vocab"):
        A.ctc_forced_align(torch.zeros((1, 75, 65), device="cuda"), tg[:1], tl[:1])
    with pytest.raises(RuntimeError, match="target_stride"):
        A.ctc_forced_align(lp, torch.ones((2, 513), dtype=torch.int32, device="cuda"), tl)
    with pytest.raises(RuntimeError, match="CUDA"):
        A.ctc_forced_align(lp.cpu(), tg, tl)
    with pytest.raises(ValueError):
        A.ctc_forced_align(lp[0], tg, tl)
    with pytest.raises(ValueError):
        A.ctc_forced_align(lp, tg[:1], tl)
    with pytest.raises(ValueError):
        A.ctc_forced_align(lp, tg, tl, input_lens=tl[:1])
    # the native call refuses a workspace smaller than avs_ctc_align_workspace_bytes
    N = A._native
    L = N.lib()
    big = torch.zeros((1, 1024, 39), device="cuda")
    tg_big = torch.ones((1, 512), dtype=torch.int32, device="cuda")
    need = L.avs_ctc_align_workspace_bytes(1, 1024, 512)
    ws = torch.empty(need - 1, dtype=torch.uint8, device="cuda")
    outs = [torch.empty(n, device="cuda") for n in (1, 1, 1024, 1024, 512)]
    rc = L.avs_ctc_align(N.ptr(big), 1, 1024, 39, 0, None, N.ptr(tg_big), 512, N.ptr(tl[:1]),
                         *(N.ptr(t) for t in outs), N.ptr(ws), ws.numel(), N.stream_ptr())
    assert rc == -4 and "workspace too small" in L.avs_last_error_string().decode()
    out = A.ctc_forced_align(lp[:0], tg[:0], tl[:0])
    assert out.frame_token.shape == (0, 75) and out.span.shape == (0, 5, 2) and out.loglik.shape == (0,)
    assert A.align_words(lp[:0], []) == []


def placed_logp(placements, T=75, V=39, peak=10.0):
    """Log-probs in which each (label, first frame, end frame) holds its label with logit ``peak`` over zeros, and the
    blank every other frame."""
    x = np.zeros((T, V))
    x[:, 0] = peak
    for c, a, b in placements:
        x[a:b, 0] = 0.0
        x[a:b, c] = peak
    return (x - np.logaddexp.reduce(x, axis=1, keepdims=True)).astype(np.float32)


def test_align_words_returns_the_placed_word_times(A, c2i):
    texts = ["bin blue at f two now", "set red by q nine again", "lay green  with e seven soon "]
    lps, want = [], []
    for b, text in enumerate(texts):
        t, placements = 3 + b, []
        for i, ch in enumerate(text):
            if i and text[i - 1] == ch:
                t += 1                                     # a repeated label needs a blank between
            n = 1 + (i + b) % 3
            placements.append((c2i[ch], t, t + n))
            t += n
        assert t <= 75
        lps.append(placed_logp(placements))
        words, i = [], 0
        for w in text.split(" "):
            if w:
                words.append((w, placements[i][1], placements[i + len(w) - 1][2]))
            i += len(w) + 1
        want.append(words)
    peak = float(np.exp(lps[0][3, c2i["b"]]))
    for fps in (25.0, 29.97):
        res = A.align_words(torch.from_numpy(np.stack(lps)).cuda(), texts, fps=fps)
        for (words, ll), exp in zip(res, want):
            assert np.isfinite(ll) and ll > -1.0
            assert [w for w, _, _, _ in words] == [w for w, _, _ in exp]
            for (w, s, e, score), (_, a, b) in zip(words, exp):
                assert s == pytest.approx(a / fps, abs=1e-12) and e == pytest.approx(b / fps, abs=1e-12), (w, s, e, a, b)
                assert score == pytest.approx(peak, rel=1e-6)
    # a clip too short for its text keeps its words, with NaN times; an unknown character raises
    (words, ll), = A.align_words(torch.from_numpy(lps[0][None, :10]).cuda(), texts[:1])
    assert ll == -np.inf and [w for w, _, _, _ in words] == texts[0].split(" ") and np.isnan(words[0][1])
    with pytest.raises(ValueError, match="outside"):
        A.align_words(torch.from_numpy(lps[0][None]).cuda(), ["bin blue!"])
