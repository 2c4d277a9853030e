"""CTC prefix beam search (K5b, csrc/ctc_beam.cu) on the B200 against the float64 oracle (oracle/ctc_beam_ref.py) and
against brute-force enumeration; determinism, corners, NaN, error paths and the decode entry points that use it."""
import numpy as np
import pytest
import torch

from oracle import ctc_beam_ref as R

pytestmark = pytest.mark.gpu

# Largest score error against the float64 oracle measured on an NVIDIA B200 (1000 W power limit) over the oracle cases
# below: 3.0e-5 at scores near -500 (GRID lexicon), 9.5e-7 without the lexicon; relative to the score, 5.9e-8 at most,
# the fp32 rounding of the output (the search runs in fp64).  The tolerance is twice that relative error.
REL_TOL = 1.2e-7
# clips whose oracle margin (closest pruning or final-rank decision) is below this are not compared id for id
MARGIN = 1e-9


@pytest.fixture(scope="module")
def A():
    import avsync_b200
    avsync_b200._native.device_check()
    return avsync_b200


@pytest.fixture(scope="module")
def grid():
    from avsync_b200.dataset import GRID_WORDS, create_vocab
    c2i, i2c = create_vocab()
    return c2i, i2c, R.Lexicon.from_words(GRID_WORDS, c2i)


@pytest.fixture(scope="module")
def grid_lex(A):
    return A.grid_lexicon()


def decode(A, lp, bw, top_n, lexicon=None, blank=0):
    ids, lens, sc = A.ctc_beam_decode(torch.from_numpy(lp).cuda(), bw, top_n, blank, lexicon)
    return ids.cpu().numpy(), lens.cpu().numpy(), sc.cpu().numpy()


def assert_scores_close(got, want):
    fin = np.isfinite(want)
    assert np.array_equal(fin, np.isfinite(got))
    err = np.abs(got[fin].astype(np.float64) - want[fin])
    assert (err <= REL_TOL * np.maximum(np.abs(want[fin]), 1.0)).all(), err.max()
    return float(err.max()) if err.size else 0.0


@pytest.mark.parametrize("lexicon", [False, True], ids=["free", "grid"])
@pytest.mark.parametrize("bw", [1, 2, 8, 64, 128])
def test_beam_vs_oracle(A, grid, grid_lex, bw, lexicon):
    lp = R.peaked_logp(256, 75, 39, seed=bw)
    o_ids, o_lens, o_sc, margin = R.beam_search_batch(lp, bw, bw, 0, grid[2] if lexicon else None)
    ok = margin > MARGIN
    assert ok.mean() >= 0.95, ok.mean()
    worst = 0.0
    for top_n in sorted({1, bw}):
        ids, lens, sc = decode(A, lp, bw, top_n, grid_lex if lexicon else None)
        assert ids.shape == (256, top_n, 75) and lens.shape == sc.shape == (256, top_n)
        np.testing.assert_array_equal(ids[ok], o_ids[ok, :top_n])
        np.testing.assert_array_equal(lens[ok], o_lens[ok, :top_n])
        worst = max(worst, assert_scores_close(sc[ok], o_sc[ok, :top_n]))
        assert ((ids >= 0).sum(axis=2) == lens).all()
    print(f"bw {bw} lexicon {lexicon}: {ok.sum()}/256 clips compared, max |score - oracle| {worst:.2e}")


def tiny_cases(lexicon):
    """(logp, blank) of problems whose every prefix fits a 128-wide beam, so the search is exhaustive."""
    rng = np.random.default_rng(11 if lexicon else 10)
    out = []
    for i in range(24):
        if lexicon:
            T, V = int(rng.integers(1, 8)), 4
        else:
            V = int(rng.integers(2, 5))
            T = int(rng.integers(1, {2: 8, 3: 7, 4: 5}[V]))
        x = rng.normal(size=(T, V)) * 2.0
        out.append(((x - np.logaddexp.reduce(x, axis=1, keepdims=True)).astype(np.float32),
                    0 if lexicon else int(rng.integers(V))))
    return out


@pytest.mark.parametrize("lexicon", [False, True], ids=["free", "lexicon"])
def test_brute_force_on_the_gpu(A, lexicon):
    lex = R.Lexicon([[1], [2, 1], [1, 1, 2]], vocab=4, blank=0, space_id=3) if lexicon else None
    words = ["a", "ba", "aab"]
    g_lex = A.CtcLexicon(words, {"a": 1, "b": 2, " ": 3}, vocab=4) if lexicon else None
    for lp, blank in tiny_cases(lexicon):
        _, _, beams = R.beam_search(lp, 10 ** 6, 1, blank, lex, trace=True)
        assert max(len(b) for b in beams) <= 128           # the search below keeps every prefix
        want, want_lp = R.exact_best(lp, blank, lex)
        ids, lens, sc = decode(A, lp[None], 128, 1, g_lex, blank)
        assert tuple(ids[0, 0, :lens[0, 0]]) == want
        assert abs(float(sc[0, 0]) - want_lp) <= REL_TOL * max(abs(want_lp), 1.0) + 1e-7


def test_exact_ties_follow_the_index_order(A):
    """Rows whose non-blank labels share one probability: every extension of a beam ties with its siblings, and the
    survivors are the lowest (source rank, label) indices, as in the oracle."""
    rng = np.random.default_rng(12)
    for _ in range(24):
        T, V = int(rng.integers(1, 7)), int(rng.integers(3, 6))
        bw = int(rng.integers(1, 5))
        p_blank = rng.choice([0.25, 0.5])
        row = np.log(np.r_[p_blank, np.full(V - 1, (1 - p_blank) / (V - 1))])
        lp = np.tile(row, (T, 1)).astype(np.float32)
        o_ids, o_lens, o_sc, _ = R.beam_search_batch(lp[None], bw, bw)
        ids, lens, sc = decode(A, lp[None], bw, bw)
        assert np.array_equal(ids, o_ids) and np.array_equal(lens, o_lens), (T, V, bw)
        assert_scores_close(sc, o_sc)


def test_grid_sentences_are_recovered_by_the_lexicon(A, grid, grid_lex):
    c2i, i2c, _ = grid
    sentences = R.grid_sentences(128, seed=1)
    lp = R.grid_sentence_logp(sentences, c2i, seed=2)
    g_ids, g_lens = A.ctc_greedy_decode(torch.from_numpy(lp).cuda())
    greedy = ["".join(i2c.get(i, "") for i in g_ids[b, :g_lens[b]].tolist()) for b in range(128)]
    from avsync_b200.dataset import GRID_WORDS
    non_words = sum(any(w not in GRID_WORDS for w in t.split(" ")) for t in greedy)
    assert non_words >= 64, non_words
    for bw in (8, 32):
        ids, lens, _ = decode(A, lp, bw, 1, grid_lex)
        got = ["".join(i2c[i] for i in ids[b, 0, :lens[b, 0]]) for b in range(128)]
        assert got == sentences


def test_each_clip_equals_its_solo_run_and_runs_repeat_bit_for_bit(A, grid_lex):
    lp = R.peaked_logp(64, 75, 39, seed=5)
    for lex in (None, grid_lex):
        full = decode(A, lp, 64, 8, lex)
        again = decode(A, lp, 64, 8, lex)
        for a, b in zip(full, again):
            assert np.array_equal(a, b)
        for c in (0, 17, 63):
            solo = decode(A, lp[c:c + 1], 64, 8, lex)
            for a, b in zip(full, solo):
                assert np.array_equal(a[c:c + 1], b)
        ids = full[0]
        for c in range(64):   # the n-best list holds distinct label sequences
            seqs = {tuple(ids[c, o, :full[1][c, o]]) for o in range(8) if np.isfinite(full[2][c, o])}
            assert len(seqs) == np.isfinite(full[2][c]).sum()


def test_widest_beam_and_vocab(A):
    lp = R.peaked_logp(8, 75, 64, seed=3)
    o_ids, o_lens, o_sc, margin = R.beam_search_batch(lp, 128, 128, 5)
    ids, lens, sc = decode(A, lp, 128, 128, None, blank=5)
    ok = margin > MARGIN
    assert ok.sum() >= 7
    assert np.array_equal(ids[ok], o_ids[ok]) and np.array_equal(lens[ok], o_lens[ok])
    assert_scores_close(sc[ok], o_sc[ok])


def test_longest_sequence(A, grid, grid_lex):
    lp = R.peaked_logp(2, 1024, 39, seed=4)
    for bw, lex, g in ((8, None, None), (128, grid[2], grid_lex)):
        o_ids, o_lens, o_sc, margin = R.beam_search_batch(lp, bw, 4, 0, lex)
        ids, lens, sc = decode(A, lp, bw, 4, g)
        assert ids.shape == (2, 4, 1024)
        ok = margin > MARGIN
        assert ok.all(), margin
        assert np.array_equal(ids, o_ids) and np.array_equal(lens, o_lens)
        assert_scores_close(sc, o_sc)
        if lex is None:
            assert lens[:, 0].min() > 100


def test_nan_counts_as_minus_infinity(A, grid_lex):
    lp = R.peaked_logp(6, 75, 39, seed=9)
    rng = np.random.default_rng(0)
    holes = lp.copy()
    holes[rng.random(holes.shape) < 0.2] = np.nan
    holes[:, :, 0] = np.where(np.isnan(holes[:, :, 0]), lp[:, :, 0], holes[:, :, 0])   # keep the blank column whole
    as_inf = np.where(np.isnan(holes), -np.inf, holes).astype(np.float32)
    for lex in (None, grid_lex):
        for a, b in zip(decode(A, holes, 16, 4, lex), decode(A, as_inf, 16, 4, lex)):
            assert np.array_equal(a, b)
    # a step where nothing is possible empties the beam: every slot is -inf with length 0
    dead = lp.copy()
    dead[2, 40] = np.nan
    dead[3, 0] = -np.inf
    ids, lens, sc = decode(A, dead, 16, 4)
    assert np.isneginf(sc[2:4]).all() and (lens[2:4] == 0).all() and (ids[2:4] == -1).all()
    assert np.isfinite(sc[[0, 1, 4, 5], 0]).all()


def test_error_paths_and_empty_batch(A, grid_lex):
    lp = torch.from_numpy(R.peaked_logp(2, 75, 39, seed=1)).cuda()
    for kw, text in (({"beam_width": 0}, "beam_width"), ({"beam_width": 129}, "beam_width"),
                     ({"beam_width": 4, "top_n": 5}, "top_n"), ({"beam_width": 4, "blank_index": 39}, "blank")):
        args = {"beam_width": 8, **kw}
        with pytest.raises(RuntimeError, match=text):
            A.ctc_beam_decode(lp, **args)
    with pytest.raises(RuntimeError, match="vocab"):
        A.ctc_beam_decode(lp[:, :, :2].contiguous(), 4, lexicon=grid_lex)     # lexicon built for 39 labels
    with pytest.raises(RuntimeError, match="n_steps"):
        A.ctc_beam_decode(torch.zeros((1, 1025, 39), device="cuda"), 4)
    with pytest.raises(RuntimeError, match="vocab"):
        A.ctc_beam_decode(torch.zeros((1, 75, 65), device="cuda"), 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        A.ctc_beam_decode(lp.cpu(), 4)
    with pytest.raises(ValueError):
        A.ctc_beam_decode(lp[0], 4)
    with pytest.raises(RuntimeError, match="space_id"):
        A.CtcLexicon(["ab c"], {"a": 1, "b": 2, "c": 3, " ": 4})
    ids, lens, sc = A.ctc_beam_decode(lp[:0], 8, 2, lexicon=grid_lex)
    assert ids.shape == (0, 2, 75) and lens.shape == sc.shape == (0, 2)


class _Grid:
    def __init__(self):
        from avsync_b200.dataset import create_vocab
        self.char_to_idx, self.idx_to_char = create_vocab()


def test_decode_batch_and_evaluate_model_with_a_beam(A, grid, grid_lex, capsys):
    c2i, i2c, _ = grid
    sentences = R.grid_sentences(6, seed=8)
    lp = torch.from_numpy(R.grid_sentence_logp(sentences, c2i, seed=9)).cuda()
    ids, lens, _ = A.ctc_beam_decode(lp, 16, 1, lexicon=grid_lex)
    want = ["".join(i2c[i] for i in ids[b, 0, :lens[b, 0]].tolist()) for b in range(6)]
    assert want == sentences
    assert A.decode_batch(lp, _Grid(), beam_width=16, lexicon=grid_lex) == want
    free_ids, free_lens, _ = A.ctc_beam_decode(lp, 16, 1)
    assert A.decode_batch(lp, _Grid(), beam_width=16) == [
        "".join(i2c.get(i, "") for i in free_ids[b, 0, :free_lens[b, 0]].tolist()) for b in range(6)]
    g_ids, g_lens = A.ctc_greedy_decode(lp)
    assert A.decode_batch(lp, _Grid()) == [
        "".join(i2c.get(i, "") for i in g_ids[b, :g_lens[b]].tolist()) for b in range(6)]

    labels = torch.zeros((6, 40), dtype=torch.int64)
    label_lens = torch.tensor([len(s) for s in sentences])
    for b, s in enumerate(sentences):
        labels[b, :len(s)] = torch.tensor([c2i[ch] for ch in s])
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(lp.cpu(), labels, label_lens), batch_size=4)
    res = A.evaluate_model(torch.nn.Identity(), loader, _Grid(), torch.device("cuda"), num_samples=6, beam_width=16,
                           lexicon=grid_lex)
    assert [r[1] for r in res] == want and all(r[2] == 100.0 for r in res)
    assert capsys.readouterr().out.count("Character accuracy: 100.00%") == 6

    m = A.decode_metrics(ids[:, 0], lens[:, 0], labels.cuda().to(torch.int32), label_lens.cuda())
    assert (m["cer"] == 0).all() and (m["wer"] == 0).all()
