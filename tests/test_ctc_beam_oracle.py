"""CTC prefix beam search (K5b) without a device: the float64 oracle against brute-force enumeration and torch's CTC
loss, its invariants, and the argument checks of avs_ctc_lexicon_create / avs_ctc_beam (include/avsync.h), which run
before any CUDA call."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ctc_beam_ref as R

I32 = ctypes.POINTER(ctypes.c_int32)
FAKE = ctypes.c_void_p(256)     # never dereferenced: every call below fails its argument checks first


def tiny_logp(rng, T, V):
    x = rng.normal(size=(T, V)) * 2.0
    return x - np.logaddexp.reduce(x, axis=1, keepdims=True)


# blank 0, labels 1 and 2, space 3; words "1", "21", "112"
TINY_LEX = R.Lexicon([[1], [2, 1], [1, 1, 2]], vocab=4, blank=0, space_id=3)


@pytest.mark.parametrize("seed", range(40))
def test_oracle_top1_is_the_exact_best_labeling(seed):
    rng = np.random.default_rng(seed)
    T, V = int(rng.integers(1, 8)), int(rng.integers(2, 5))
    blank = int(rng.integers(V))
    lp = tiny_logp(rng, T, V)
    want, want_lp = R.exact_best(lp, blank)
    (got, got_lp), = R.beam_search(lp, 10 ** 6, 1, blank)[0]
    assert got == want
    assert abs(got_lp - want_lp) <= 1e-12


@pytest.mark.parametrize("seed", range(40))
def test_oracle_top1_with_a_lexicon_is_the_exact_best_text(seed):
    rng = np.random.default_rng(100 + seed)
    lp = tiny_logp(rng, int(rng.integers(1, 8)), 4)
    want, want_lp = R.exact_best(lp, 0, TINY_LEX)
    (got, got_lp), = R.beam_search(lp, 10 ** 6, 1, 0, TINY_LEX)[0]
    assert got == want and TINY_LEX.is_text(got)
    assert abs(got_lp - want_lp) <= 1e-12


@pytest.mark.parametrize("seed", range(10))
def test_exact_best_agrees_with_torch_ctc_loss(seed):
    rng = np.random.default_rng(200 + seed)
    T, V = int(rng.integers(2, 8)), int(rng.integers(2, 5))
    lp = tiny_logp(rng, T, V)
    y, y_lp = R.exact_best(lp, 0)
    assert len(y) > 0
    loss = torch.nn.functional.ctc_loss(torch.from_numpy(lp)[:, None], torch.tensor([y]), torch.tensor([T]),
                                        torch.tensor([len(y)]), blank=0, reduction="none")
    assert abs(-float(loss[0]) - y_lp) <= 1e-10
    for _ in range(5):   # any labeling, not only the best
        z = tuple(int(c) for c in rng.integers(1, V, int(rng.integers(1, (T + 1) // 2 + 1))))
        loss = torch.nn.functional.ctc_loss(torch.from_numpy(lp)[:, None], torch.tensor([z]), torch.tensor([T]),
                                            torch.tensor([len(z)]), blank=0, reduction="none")
        assert abs(-float(loss[0]) - R.ctc_log_prob(lp, z, 0)) <= 1e-10


@pytest.mark.parametrize("lexicon", [False, True])
def test_oracle_beams_never_hold_a_prefix_twice(lexicon):
    from avsync_b200.dataset import GRID_WORDS, create_vocab
    lex = R.Lexicon.from_words(GRID_WORDS, create_vocab()[0]) if lexicon else None
    lp = R.peaked_logp(4, seed=7)
    for b in range(4):
        _, _, beams = R.beam_search(lp[b], 64, 1, 0, lex, trace=True)
        assert max(len(s) for s in beams) == 64
        for step in beams:
            assert len(set(step)) == len(step)


def test_grid_lexicon_outputs_are_grid_words_joined_by_single_spaces():
    from avsync_b200.dataset import GRID_WORDS, create_vocab
    assert len(GRID_WORDS) == len(set(GRID_WORDS)) == 51 and "w" not in GRID_WORDS
    c2i, i2c = create_vocab()
    lex = R.Lexicon.from_words(GRID_WORDS, c2i)
    lp = np.concatenate([R.peaked_logp(6, seed=3),
                         R.grid_sentence_logp(R.grid_sentences(6, seed=4), c2i, seed=5)])
    n_texts = 0
    for b in range(len(lp)):
        hyps, _, _ = R.beam_search(lp[b], 32, 32, 0, lex)
        for ids, score in hyps:
            if score == -np.inf:
                continue
            text = "".join(i2c[i] for i in ids)
            assert text == "" or all(w in GRID_WORDS for w in text.split(" ")), text
            n_texts += text != ""
    assert n_texts > 100


# ---------------------------------------------------------------- argument checks through ctypes, no device needed

@pytest.fixture(scope="module")
def native():
    import avsync_b200
    N = avsync_b200._native
    if not __import__("os").path.isfile(N.LIB_PATH):
        N.build()
    return N


def test_lexicon_create_rejects_bad_input_without_a_device(native):
    L = native.lib()
    h = ctypes.c_void_p()

    def create(words, vocab=39, blank=0, space_id=37, n_words=None, offsets=None):
        ids = np.asarray([c for w in words for c in w] or [0], np.int32)
        off = np.asarray(offsets if offsets is not None else np.cumsum([0] + [len(w) for w in words]), np.int32)
        n = len(words) if n_words is None else n_words
        rc = L.avs_ctc_lexicon_create(ids.ctypes.data_as(I32), off.ctypes.data_as(I32), n, vocab, blank, space_id, None,
                                      ctypes.byref(h))
        return rc, L.avs_last_error_string().decode()

    ok = [[2, 9, 14]]
    rc, msg = create(ok, n_words=0)
    assert rc == -1 and "at least one word" in msg
    for kw, text in (({"vocab": 1}, "vocab must be in [2, 64]"), ({"vocab": 65}, "vocab must be in [2, 64]"),
                     ({"blank": -1}, "blank"), ({"blank": 39}, "blank"), ({"space_id": 39}, "space_id"),
                     ({"space_id": 0}, "space_id")):
        rc, msg = create(ok, **kw)
        assert rc == -1 and text in msg, (kw, msg)
    for words, text in (([[2, 9], []], "word 1 is empty"), ([[2, 0]], "blank"), ([[2, 37]], "space_id"),
                        ([[2, 39]], "< vocab"), ([[2, -3]], "< vocab")):
        rc, msg = create(words)
        assert rc == -1 and text in msg, (words, msg)
    rc, msg = create([[2, 9]], offsets=[1, 2])
    assert rc == -1 and "word_offsets[0]" in msg
    assert L.avs_ctc_lexicon_create(None, None, 1, 39, 0, 37, None, ctypes.byref(h)) == -1
    assert not h.value


def test_beam_rejects_bad_arguments_without_a_device(native):
    L = native.lib()

    def beam(n_clips=4, n_steps=75, vocab=39, blank=0, beam_width=8, top_n=1, ws_bytes=1 << 40, out=FAKE):
        rc = L.avs_ctc_beam(FAKE, n_clips, n_steps, vocab, blank, beam_width, top_n, None, out, out, out, FAKE,
                            ws_bytes, None)
        return rc, L.avs_last_error_string().decode()

    for kw, text in (({"beam_width": 0}, "beam_width must be in [1, 128]"),
                     ({"beam_width": 129}, "beam_width must be in [1, 128]"),
                     ({"top_n": 0}, "top_n must be in [1, beam_width]"),
                     ({"top_n": 9}, "top_n must be in [1, beam_width]"),
                     ({"vocab": 1}, "vocab must be in [2, 64]"), ({"vocab": 65}, "vocab must be in [2, 64]"),
                     ({"blank": -1}, "blank must be in [0, vocab)"), ({"blank": 39}, "blank must be in [0, vocab)"),
                     ({"n_steps": 0}, "n_steps must be in [1, 1024]"),
                     ({"n_steps": 1025}, "n_steps must be in [1, 1024]"),
                     ({"n_clips": -1}, "n_clips"), ({"out": None}, "null argument")):
        rc, msg = beam(**kw)
        assert rc == -1 and text in msg, (kw, msg)
    rc, msg = beam(ws_bytes=1024)
    assert rc == -4 and "workspace too small" in msg
    assert beam(n_clips=0, out=None)[0] == 0          # an empty batch needs no buffers and launches nothing


def test_beam_workspace_bytes(native):
    L = native.lib()
    per_clip = L.avs_ctc_beam_workspace_bytes(1, 75, 128)
    assert per_clip > 0 and L.avs_ctc_beam_workspace_bytes(4096, 75, 128) == 4096 * per_clip
    # the prefix trie holds at most n_steps * beam_width + 1 nodes, in a table at most half full
    assert per_clip >= 3 * 4 * (75 * 128 + 1)
    for args in ((0, 75, 8), (1, 0, 8), (1, 1025, 8), (1, 75, 0), (1, 75, 129)):
        assert L.avs_ctc_beam_workspace_bytes(*args) == 0
