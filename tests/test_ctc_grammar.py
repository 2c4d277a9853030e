"""Exact CTC decoding under a word-slot grammar (K5d, csrc/ctc_grammar.cu) on the B200 against the float64 restatement
(oracle/ctc_grammar_ref.py) and against the full 64 000-sentence GRID grammar brute-forced with K5c; the planted
sentence where the lexicon beam breaks the grammar; tie rules, statuses, corners, NaN, determinism, error paths and the
decode entry points."""
import numpy as np
import pytest
import torch

from oracle import ctc_beam_ref
from oracle import ctc_grammar_ref as R

pytestmark = pytest.mark.gpu

# Largest errors against the float64 restatement measured on an NVIDIA B200 (1000 W power limit) over 1 024 GRID clips:
# loglik 5.7e-8 relative, posteriors 3.0e-8 absolute.  The kernel runs in fp64, so that is the fp32 rounding of its
# outputs (at most 2^-24 = 6.0e-8 relative).  The tolerances are twice that rounding bound.
REL_TOL = 1.2e-7
POST_TOL = 1.2e-7


@pytest.fixture(scope="module")
def A():
    import avsync_b200
    avsync_b200._native.device_check()
    return avsync_b200


@pytest.fixture(scope="module")
def c2i():
    from avsync_b200.dataset import create_vocab
    return create_vocab()[0]


@pytest.fixture(scope="module")
def grid(A, c2i):
    from avsync_b200.dataset import GRID_SLOTS
    return A.grid_grammar(), R.lattice(R.slots_to_ids(GRID_SLOTS, c2i), 0, c2i[" "])


def run(A, lp, grammar, input_lens=None):
    il = None if input_lens is None else torch.as_tensor(np.asarray(input_lens, np.int32)).cuda()
    out = A.ctc_grammar_decode(torch.from_numpy(np.ascontiguousarray(lp)).cuda(), grammar, il)
    return tuple(t.cpu().numpy() for t in out)


def rel_err(got, want, floor=1.0):
    fin = np.isfinite(want)
    assert np.array_equal(fin, np.isfinite(got)) and np.array_equal(np.isnan(want), np.isnan(got))
    if not fin.any():
        return 0.0
    return float((np.abs(got[fin].astype(np.float64) - want[fin]) / np.maximum(np.abs(want[fin]), floor)).max())


def assert_matches_oracle(got, want, slot_off, min_mbr_share=1.0):
    words, span, ps, ll, post, mbr = got
    o_words, o_span, o_ps, o_ll, o_post, o_mbr = want
    np.testing.assert_array_equal(words, o_words)
    np.testing.assert_array_equal(span, o_span)
    np.testing.assert_array_equal(ps, o_ps.astype(np.float32))        # the same fp64 adds, rounded once
    e_ll = rel_err(ll, o_ll)
    fin = ~np.isnan(o_post)
    assert np.array_equal(fin, ~np.isnan(post))
    e_post = float(np.abs(post[fin] - o_post[fin]).max()) if fin.any() else 0.0
    assert e_ll <= REL_TOL and e_post <= POST_TOL, (e_ll, e_post)
    # MBR words: equal wherever the oracle's top two posteriors in each slot are further apart than the tolerance
    p32 = o_post.astype(np.float32)
    ok = np.ones(len(words), bool)
    for a, b in zip(slot_off[:-1], slot_off[1:]):
        if b - a > 1:
            top = np.sort(p32[:, a:b], axis=1)[:, -2:]
            ok &= ~fin[:, 0] | (top[:, 1] - top[:, 0] > 2 * POST_TOL)
    assert ok.mean() >= min_mbr_share, ok.mean()
    np.testing.assert_array_equal(mbr[ok], o_mbr[ok])
    return e_ll, e_post


def check(got, lp, lat, input_lens=None, min_mbr_share=1.0):
    return assert_matches_oracle(got, R.decode_batch(lp, lat, input_lens), lat.slot_off, min_mbr_share)


def grid_batch(c2i, n, seed):
    """n GRID-shaped clips (T = 75, V = 39), as in the K5c tests: the first half log-probs of random GRID sentences being
    spoken, the second half unrelated peaked log-probs; random input lengths, some too short for any sentence."""
    sentences = ctc_beam_ref.grid_sentences(n // 2, seed)
    spoken = ctc_beam_ref.grid_sentence_logp(sentences, c2i, seed=seed + 1)
    lp = np.concatenate([spoken, ctc_beam_ref.peaked_logp(n - n // 2, 75, 39, seed=seed + 2)])
    input_lens = np.random.default_rng(seed + 3).integers(16, 76, n).astype(np.int32)
    return sentences, lp, input_lens


def test_grid_clips_vs_oracle(A, c2i, grid):
    g, lat = grid
    _, lp, input_lens = grid_batch(c2i, 1024, 0)
    got = run(A, lp, g, input_lens)
    e_ll, e_post = check(got, lp, lat, input_lens, min_mbr_share=0.99)
    n_inf = int(np.isneginf(got[3]).sum())
    assert 20 <= n_inf <= 500, n_inf
    print(f"1024 GRID clips, {n_inf} without a path: max rel err loglik {e_ll:.2e}, max abs err posterior {e_post:.2e}")


def test_full_grid_grammar_brute_forced_with_k5c(A, c2i, grid):
    """Every one of the 64 000 GRID sentences aligned with ctc_forced_align (K5c) on the same clip."""
    from avsync_b200.dataset import GRID_SLOTS
    g, _ = grid
    slots = R.slots_to_ids(GRID_SLOTS, c2i)
    choices, targets = zip(*R.sentences(slots, c2i[" "]))
    choices = np.array(choices)
    lens = np.array([len(y) for y in targets], np.int32)
    tg = np.zeros((len(targets), lens.max()), np.int32)
    for i, y in enumerate(targets):
        tg[i, :len(y)] = y
    tg_d, lens_d = torch.from_numpy(tg).cuda(), torch.from_numpy(lens).cuda()
    off = np.cumsum([0] + [len(ws) for ws in GRID_SLOTS])
    word_of = torch.from_numpy(choices + off[:-1]).cuda()                      # [64000, 6] global word index
    sentences = ctc_beam_ref.grid_sentences(3, seed=7)
    lp = np.concatenate([ctc_beam_ref.grid_sentence_logp(sentences, c2i, seed=8),
                         ctc_beam_ref.peaked_logp(2, 75, 39, seed=9)])
    words, span, ps, ll, post, mbr = run(A, lp, g)
    for b in range(len(lp)):
        x = torch.from_numpy(lp[b:b + 1]).cuda().expand(len(targets), 75, 39)
        al = A.ctc_forced_align(x, tg_d, lens_d)
        bf_ps = float(al.path_score.max())
        assert ps[b] == bf_ps, (b, ps[b], bf_ps)
        lls = al.loglik.double()
        Z = torch.logsumexp(lls, 0)
        assert abs(ll[b] - float(Z)) <= 2 * REL_TOL * abs(float(Z)), (ll[b], float(Z))
        bf_post = torch.zeros(off[-1], dtype=torch.float64, device="cuda")
        bf_post.index_add_(0, word_of.reshape(-1), (lls - Z).exp().repeat_interleave(6))
        # each K5c loglik is rounded to fp32: a relative error of 2^-24 |loglik| in every sentence's probability
        tol = 2 * 2.0 ** -24 * float(lls.abs().max()) + POST_TOL
        err = float((torch.from_numpy(post[b]).cuda().double() - bf_post).abs().max())
        assert err <= tol, (err, tol)
        i = int(np.flatnonzero((choices == words[b]).all(1))[0])
        assert float(al.path_score[i]) == ps[b]                                # the decoded sentence's own K5c score
        if b < len(sentences):
            assert g.texts(words[b:b + 1]) == [sentences[b]]
        print(f"clip {b}: path score {ps[b]:.4f}, loglik {ll[b]:.4f} vs {float(Z):.4f}, posterior err {err:.1e}")


def planted_logp(c2i, n, seed):
    """GRID sentences spoken with an extra, weaker word of the same slot as its neighbour inserted: the lexicon accepts
    the seven-word text, the grammar does not."""
    from avsync_b200.dataset import GRID_SLOTS
    rng = np.random.default_rng(seed)
    sentences = ctc_beam_ref.grid_sentences(n, seed)
    out = np.empty((n, 75, 39), np.float32)
    for b, s in enumerate(sentences):
        words = s.split(" ")
        k = int(rng.integers(6))
        extra = [w for w in GRID_SLOTS[k] if w != words[k]][int(rng.integers(len(GRID_SLOTS[k]) - 1))]
        text = " ".join(words[:k + 1] + [extra] + words[k + 1:])
        a, e = len(" ".join(words[:k + 1])) + 1, len(" ".join(words[:k + 1])) + 1 + len(extra)
        path, strength = [], []
        for i, ch in enumerate(text):       # one frame per character, a blank between repeated ones
            path += [c2i[ch]] + ([0] if text[i + 1:i + 2] == ch else [])
            strength += [4.0 if a <= i < e else 10.0] * (2 if text[i + 1:i + 2] == ch else 1)
        assert len(path) <= 75
        x = rng.normal(0.0, 1.0, size=(75, 39))
        x[np.arange(len(path)), path] += strength
        x[len(path):, 0] += 8.0
        out[b] = x - np.logaddexp.reduce(x, axis=1, keepdims=True)
    return sentences, out


def test_grammar_keeps_the_planted_sentence_where_the_lexicon_beam_breaks_it(A, c2i, grid):
    from avsync_b200.dataset import GRID_SLOTS
    g, lat = grid
    sentences, lp = planted_logp(c2i, 64, seed=11)
    lp_d = torch.from_numpy(lp).cuda()
    i2c = {i: c for c, i in c2i.items()}
    ids, lens, _ = A.ctc_beam_decode(lp_d, 8, 1, lexicon=A.grid_lexicon())
    beam = ["".join(i2c[i] for i in ids[b, 0, :lens[b, 0]].tolist()) for b in range(64)]

    def in_grammar(t):
        ws = t.split(" ")
        return len(ws) == 6 and all(w in s for w, s in zip(ws, GRID_SLOTS))
    broken = sum(not in_grammar(t) for t in beam)
    assert broken >= 56, broken
    res = A.ctc_grammar_decode(lp_d, g)
    assert g.texts(res.words.cpu()) == sentences
    assert g.texts(res.mbr_words.cpu()) == sentences
    print(f"{broken}/64 beam texts break the grammar; the grammar decode returns every planted sentence")


def test_exact_ties_follow_the_tie_rule(A):
    """Uniform rows: every path ties.  In a chain the stay wins, then s-1, then s-2; at SP and at the end the stay,
    then the lowest word index, tb before c_last."""
    c2i = {c: i for i, c in enumerate("_ abcd")}
    cases = [([["ab", "cd"], ["a", "b"]], 8, [0, 0], [[0, 2], [3, 4]]),
             ([["b", "a"], ["c", "d"], ["a"]], 9, [0, 0, 0], [[0, 1], [2, 3], [4, 5]]),
             ([["a", "b", "c"]], 3, [0], [[0, 1]]),
             ([["aa", "ab"], ["b", "a"]], 7, [1, 0], [[0, 2], [3, 4]])]
    for slots, T, want_words, want_span in cases:
        g = A.CtcGrammar(slots, c2i)
        lat = R.lattice(R.slots_to_ids(slots, c2i), 0, 1)
        for lp in (np.full((1, T, 6), np.log(1 / 6), np.float32), np.zeros((1, T, 6), np.float32)):
            got = run(A, lp, g)
            check(got, lp, lat, min_mbr_share=0.0)      # tied posteriors: MBR words follow the kernel's own f32 values
            np.testing.assert_array_equal(got[0][0], want_words)
            np.testing.assert_array_equal(got[1][0], want_span)
            off = lat.slot_off
            assert [int(np.argmax(got[4][0, a:b])) for a, b in zip(off[:-1], off[1:])] == got[5][0].tolist()


def test_corners_and_invalid_clips_next_to_valid_ones(A, c2i, grid):
    g, lat = grid
    sentences, lp, _ = grid_batch(c2i, 8, 20)
    input_lens = np.full(8, 75, np.int32)
    input_lens[1] = 0                            # no frames
    input_lens[2] = 10                           # shorter than every sentence
    input_lens[3] = -1                           # out of range
    input_lens[5] = 76
    got = run(A, lp, g, input_lens)
    check(got, lp, lat, input_lens)
    words, span, ps, ll, post, mbr = got
    assert np.isneginf(ps[[1, 2]]).all() and np.isneginf(ll[[1, 2]]).all()
    assert np.isnan(ps[[3, 5]]).all() and np.isnan(ll[[3, 5]]).all()
    bad = [1, 2, 3, 5]
    assert (words[bad] == -1).all() and (mbr[bad] == -1).all() and (span[bad] == -1).all() and np.isnan(post[bad]).all()
    assert np.isfinite(ps[[0, 4, 6, 7]]).all() and g.texts(words[:1]) == sentences[:1]
    for c in (0, 4):                             # valid clips are unaffected by their neighbours
        solo = run(A, lp[c:c + 1], g, input_lens[c:c + 1])
        for a, b in zip(got, solo):
            assert np.array_equal(a[c:c + 1], b, equal_nan=True)


def test_longest_clip_takes_the_workspace(A, c2i, grid):
    """T = 1024: 357 KB of per-frame storage per clip, in the workspace."""
    g, lat = grid
    L = A._native.lib()
    assert L.avs_ctc_grammar_workspace_bytes(g.handle, 4096, 75) == 0                  # GRID at T = 75: shared memory
    per_clip = L.avs_ctc_grammar_workspace_bytes(g.handle, 1, 1024)
    assert per_clip >= 1024 * (299 + 10 * 5) and L.avs_ctc_grammar_workspace_bytes(g.handle, 3, 1024) == 3 * per_clip
    lp = ctc_beam_ref.peaked_logp(3, 1024, 39, seed=21)
    lp[0, :75] = ctc_beam_ref.grid_sentence_logp(ctc_beam_ref.grid_sentences(1, 21), c2i, seed=22)[0]
    input_lens = [1024, 700, 1024]
    got = run(A, lp, g, input_lens)
    check(got, lp, lat, input_lens)
    assert np.isfinite(got[2]).all()


def test_nan_counts_as_minus_infinity(A, c2i, grid):
    g, lat = grid
    _, lp, input_lens = grid_batch(c2i, 32, 30)
    rng = np.random.default_rng(31)
    holes = lp.copy()
    holes[rng.random(holes.shape) < 0.05] = np.nan
    as_inf = np.where(np.isnan(holes), -np.inf, holes).astype(np.float32)
    a, b = run(A, holes, g, input_lens), run(A, as_inf, g, input_lens)
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)
    check(a, holes, lat, input_lens)
    assert np.isfinite(a[2]).sum() >= 8
    dead = lp[:2].copy()
    dead[:, 30, :] = np.nan                      # a frame where nothing is possible
    words, _, ps, ll, post, _ = run(A, dead, g)
    assert np.isneginf(ps).all() and np.isneginf(ll).all() and (words == -1).all() and np.isnan(post).all()


def test_one_slot_one_word_and_a_grammar_at_the_limits(A):
    c2i = {c: i for i, c in enumerate("_ " + "abcdefghijklmnopqrstuvwxyz0123456789")}   # 38 ids, 36 letters
    rng = np.random.default_rng(40)
    g1 = A.CtcGrammar([["a"]], c2i)
    lp = ctc_beam_ref.peaked_logp(4, 20, 38, seed=40)
    got = run(A, lp, g1, [20, 1, 0, 21])
    check(got, lp, R.lattice([[[2]]], 0, 1), [20, 1, 0, 21])
    assert (got[4][:2] == 1.0).all() and (got[0][:2] == 0).all()

    # 16 slots, 255 words in slot 0 (36 of one letter, 219 of two), 64-letter words, 2 048 states exactly
    letters = "abcdefghijklmnopqrstuvwxyz0123456789"
    slot0 = list(letters) + [a + b for a in letters for b in letters][:219]
    rest = [["".join(rng.choice(list(letters), 64))], ["".join(rng.choice(list(letters), 64))]]
    used = sum(2 * len(w) + 1 for ws in [slot0] + rest for w in ws) + 15
    for k in range(13):                          # the last slot takes two words, to land on 2 048 exactly
        budget = 2048 - used
        m = (budget // (13 - k) - 1) // 2 if k < 12 else (budget - 4) // 2
        rest.append(["".join(rng.choice(list(letters), m))] + (["a"] if k == 12 else []))
        used += 2 * m + 1 + (3 if k == 12 else 0)
    slots = [slot0] + rest
    assert len(slots) == 16 and sum(2 * len(w) + 1 for ws in slots for w in ws) + 15 == 2048
    g = A.CtcGrammar(slots, c2i)
    assert A._native.lib().avs_ctc_grammar_workspace_bytes(g.handle, 1, 1024) > 0
    lat = R.lattice(R.slots_to_ids(slots, c2i), 0, 1)
    lp = ctc_beam_ref.peaked_logp(2, 1024, 38, seed=41)
    got = run(A, lp, g, [1024, 900])
    check(got, lp, lat, [1024, 900])
    assert np.isfinite(got[2]).all()
    with pytest.raises(RuntimeError, match="2048"):
        A.CtcGrammar(slots[:-1] + [slots[-1] + ["b"]], c2i)


def test_batch_equals_solo_and_runs_repeat_bit_for_bit(A, c2i, grid):
    g, _ = grid
    _, lp, input_lens = grid_batch(c2i, 96, 50)
    full, again = run(A, lp, g, input_lens), run(A, lp, g, input_lens)
    for x, y in zip(full, again):
        assert np.array_equal(x, y, equal_nan=True)
    for c in (0, 47, 48, 95):
        solo = run(A, lp[c:c + 1], g, input_lens[c:c + 1])
        for x, y in zip(full, solo):
            assert np.array_equal(x[c:c + 1], y, equal_nan=True)


def test_error_paths_and_empty_batch(A, grid):
    g, _ = grid
    lp = torch.from_numpy(ctc_beam_ref.peaked_logp(2, 75, 39, seed=1)).cuda()
    with pytest.raises(RuntimeError, match="vocab"):
        A.ctc_grammar_decode(torch.zeros((1, 75, 40), device="cuda"), g)
    with pytest.raises(RuntimeError, match="n_steps"):
        A.ctc_grammar_decode(torch.zeros((1, 1025, 39), device="cuda"), g)
    with pytest.raises(RuntimeError, match="CUDA"):
        A.ctc_grammar_decode(lp.cpu(), g)
    with pytest.raises(ValueError):
        A.ctc_grammar_decode(lp[0], g)
    with pytest.raises(ValueError, match="blank"):
        A.ctc_grammar_decode(lp, g, blank_index=1)
    with pytest.raises(ValueError):
        A.ctc_grammar_decode(lp, g, input_lens=torch.ones(3, dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError, match="outside"):
        A.CtcGrammar([["bin!"]], A.dataset.create_vocab()[0])
    with pytest.raises(RuntimeError, match="twice"):
        A.CtcGrammar([["bin", "bin"]], A.dataset.create_vocab()[0])
    other = A.grid_grammar()
    other.device = torch.device("cuda", torch.cuda.device_count())   # a grammar that lives on another device
    with pytest.raises(ValueError, match="lives on"):
        A.ctc_grammar_decode(lp, other)
    out = A.ctc_grammar_decode(lp[:0], g)
    assert out.words.shape == (0, 6) and out.span.shape == (0, 6, 2) and out.posterior.shape == (0, 51)
    assert out.loglik.shape == out.path_score.shape == (0,) and out.mbr_words.shape == (0, 6)
    L = A._native.lib()
    N = A._native
    need = L.avs_ctc_grammar_workspace_bytes(g.handle, 1, 1024)
    ws = torch.empty(need - 1, dtype=torch.uint8, device="cuda")
    big = torch.zeros((1, 1024, 39), device="cuda")
    outs = [torch.empty(64, device="cuda") for _ in range(6)]
    rc = L.avs_ctc_grammar_decode(g.handle, N.ptr(big), 1, 1024, 39, None, *(N.ptr(t) for t in outs), N.ptr(ws),
                                  ws.numel(), N.stream_ptr())
    assert rc == -4 and "workspace too small" in L.avs_last_error_string().decode()


class _Grid:
    def __init__(self):
        from avsync_b200.dataset import create_vocab
        self.char_to_idx, self.idx_to_char = create_vocab()


def test_decode_batch_and_evaluate_model_with_a_grammar(A, c2i, grid, capsys):
    g, _ = grid
    sentences, lp = planted_logp(c2i, 6, seed=60)
    lp = torch.from_numpy(lp).cuda()
    assert A.decode_batch(lp, _Grid(), grammar=g) == sentences
    with pytest.raises(ValueError, match="grammar"):
        A.decode_batch(lp, _Grid(), beam_width=8, grammar=g)
    with pytest.raises(ValueError, match="grammar"):
        A.decode_batch(lp, _Grid(), lexicon=A.grid_lexicon(), grammar=g)
    labels = torch.zeros((6, 40), dtype=torch.int64)
    label_lens = torch.tensor([len(s) for s in sentences])
    for b, s in enumerate(sentences):
        labels[b, :len(s)] = torch.tensor([c2i[ch] for ch in s])
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(lp.cpu(), labels, label_lens), batch_size=4)
    res = A.evaluate_model(torch.nn.Identity(), loader, _Grid(), torch.device("cuda"), num_samples=6, grammar=g)
    assert [r[1] for r in res] == sentences and all(r[2] == 100.0 for r in res)
    assert capsys.readouterr().out.count("Character accuracy: 100.00%") == 6
    with pytest.raises(ValueError, match="grammar"):
        A.evaluate_model(torch.nn.Identity(), loader, _Grid(), torch.device("cuda"), beam_width=8, grammar=g)
