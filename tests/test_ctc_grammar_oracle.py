"""Exact CTC decoding under a word-slot grammar (K5d) without a device: the float64 restatement against brute-force
enumeration of the grammar's sentences and against torch's CTC loss; the tie rule and statuses; GRID_SLOTS; the
argument checks of avs_ctc_grammar_create / avs_ctc_grammar_decode (include/avsync.h), which run before any CUDA call."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import ctc_align_ref
from oracle import ctc_grammar_ref as R

FAKE = ctypes.c_void_p(256)     # never dereferenced: every call below fails its argument checks first
BLANK, SPACE = 0, 1


def rand_logp(rng, T, V, scale=2.0):
    x = rng.normal(size=(T, V)) * scale
    return x - np.logaddexp.reduce(x, axis=1, keepdims=True)


def random_grammar(rng, V=6):
    """1-4 slots of 1-6 distinct words over labels 2..V-1, with repeated letters, a word and its prefix ("a" / "ab"),
    the same word in two slots and single-label words thrown in."""
    G = int(rng.integers(1, 5))
    slots = []
    for _ in range(G):
        ws = []
        for _ in range(int(rng.integers(1, 7))):
            r = rng.random()
            if r < 0.2:
                c = int(rng.integers(2, V))
                w = [c, c] + list(rng.integers(2, V, int(rng.integers(0, 2))))      # repeated letter
            elif r < 0.35 and ws:
                w = list(ws[int(rng.integers(len(ws)))]) + [int(rng.integers(2, V))]   # extends a word of the slot
            elif r < 0.5 and slots:
                w = list(slots[-1][0])                                                 # a word of the previous slot
            elif r < 0.7:
                w = [int(rng.integers(2, V))]                                          # a single label
            else:
                w = list(rng.integers(2, V, int(rng.integers(1, 4))))
            w = [int(c) for c in w]
            if w not in ws:
                ws.append(w)
        slots.append(ws)
    return slots


@pytest.mark.parametrize("seed", range(60))
def test_restatement_equals_brute_force(seed):
    rng = np.random.default_rng(3000 + seed)
    slots = random_grammar(rng)
    T = int(rng.integers(1, 24))
    n = int(rng.integers(0, T + 1)) if rng.random() < 0.3 else T
    lp = rand_logp(rng, T, 6).astype(np.float32)
    lat = R.lattice(slots, BLANK, SPACE)
    d, b = R.decode(lp, lat, n), R.brute_force(lp, slots, n, BLANK, SPACE)
    if b.loglik == -np.inf:
        assert d.path_score == d.loglik == -np.inf and (d.words == -1).all() and np.isnan(d.posterior).all()
        return
    assert d.path_score == b.path_score                         # the same adds in the same order
    assert abs(d.loglik - b.loglik) <= 1e-12 * max(1.0, abs(b.loglik))
    np.testing.assert_allclose(d.posterior, b.posterior, rtol=0, atol=1e-12)
    for a, e in zip(lat.slot_off[:-1], lat.slot_off[1:]):       # posteriors of each slot sum to 1
        assert abs(d.posterior[a:e].sum() - 1.0) <= 1e-12
    # the decoded sentence is a best one: its own K5c path score is path_score
    y = sum((([SPACE] if g else []) + slots[g][i] for g, i in enumerate(d.words)), [])
    r = ctc_align_ref.align(lp, y, n, BLANK)
    assert r.path_score == d.path_score
    # its spans are K5c's: from the word's first label frame to its last label frame
    k = 0
    for g, i in enumerate(d.words):
        k += 1 if g else 0
        L = len(slots[g][i])
        assert (d.span[g] == [r.span[k, 0], r.span[k + L - 1, 1]]).all()
        k += L
    p32 = d.posterior.astype(np.float32)
    assert [int(np.argmax(p32[a:e])) for a, e in zip(lat.slot_off[:-1], lat.slot_off[1:])] == d.mbr_words.tolist()


@pytest.mark.parametrize("seed", range(10))
def test_loglik_equals_log_sum_exp_of_torch_ctc_loss(seed):
    rng = np.random.default_rng(4000 + seed)
    slots = random_grammar(rng)
    T = int(rng.integers(8, 30))
    lp = rand_logp(rng, T, 6)
    ys = [y for _, y in R.sentences(slots, SPACE)]
    tg = torch.zeros((len(ys), max(map(len, ys))), dtype=torch.long)
    for i, y in enumerate(ys):
        tg[i, :len(y)] = torch.tensor(y)
    loss = torch.nn.functional.ctc_loss(torch.from_numpy(lp)[:, None].expand(T, len(ys), 6), tg,
                                        torch.full((len(ys),), T), torch.tensor([len(y) for y in ys]), blank=BLANK,
                                        reduction="none", zero_infinity=False)
    want = float(torch.logsumexp(-loss, 0))
    got = R.decode(lp, R.lattice(slots, BLANK, SPACE)).loglik
    assert (want == got == -np.inf) or abs(got - want) <= 1e-10 * max(1.0, abs(want)), (got, want)


def test_tie_rule():
    """Uniform rows: every path ties.  At SP and at the end the lowest word index wins; in a chain the stay."""
    lp = np.full((8, 6), np.log(1 / 6))
    d = R.decode(lp, R.lattice([[[2, 3], [4, 5]], [[2], [3]]], BLANK, SPACE))
    assert d.words.tolist() == [0, 0] and d.span.tolist() == [[0, 2], [3, 4]]
    d = R.decode(lp[:3], R.lattice([[[2], [3], [4]]], BLANK, SPACE))
    assert d.words.tolist() == [0] and d.span.tolist() == [[0, 1]] and d.mbr_words.tolist() == [0]
    np.testing.assert_allclose(d.posterior, [1 / 3] * 3, rtol=1e-12)
    d = R.decode(lp[:9], R.lattice([[[3], [2]], [[4], [5]], [[2]]], BLANK, SPACE))
    assert d.words.tolist() == [0, 0, 0] and d.span.tolist() == [[0, 1], [2, 3], [4, 5]]


def test_statuses():
    lat = R.lattice([[[2, 3]], [[4], [5]]], BLANK, SPACE)
    lp = rand_logp(np.random.default_rng(5), 10, 6)
    for n in (-1, 11):
        d = R.decode(lp, lat, n)
        assert np.isnan(d.path_score) and np.isnan(d.loglik) and (d.words == -1).all() and (d.span == -1).all()
        assert (d.mbr_words == -1).all() and np.isnan(d.posterior).all()
    for n in (0, 3):                    # "ab c" needs 4 frames
        d = R.decode(lp, lat, n)
        assert d.path_score == d.loglik == -np.inf and (d.words == -1).all() and np.isnan(d.posterior).all()
    assert np.isfinite(R.decode(lp, lat, 4).path_score)
    holes = lp.copy()
    holes[4, :] = np.nan
    assert R.decode(holes, lat).loglik == -np.inf
    holes = lp.copy()
    holes[4, 3] = np.nan
    a, b = R.decode(holes, lat), R.decode(np.where(np.isnan(holes), -np.inf, holes), lat)
    assert a.path_score == b.path_score and (a.words == b.words).all()


def test_grid_slots():
    from avsync_b200.dataset import GRID_SLOTS, GRID_WORDS
    assert GRID_WORDS == sum(GRID_SLOTS, [])
    assert [len(s) for s in GRID_SLOTS] == [4, 4, 4, 25, 10, 4] and len(GRID_WORDS) == 51
    from avsync_b200.dataset import create_vocab
    lat = R.lattice(R.slots_to_ids(GRID_SLOTS, create_vocab()[0]), 0, 37)
    assert len(lat.lab) == 304 and lat.n_chain == 299


# ---------------------------------------------------------------- argument checks through ctypes, no device needed

@pytest.fixture(scope="module")
def native():
    import avsync_b200
    N = avsync_b200._native
    if not os.path.isfile(N.LIB_PATH):
        N.build()
    return N


def create(L, slots, vocab=8, blank=0, space=1, n_slots=None):
    ids, w_off, s_off = [], [0], [0]
    for ws in slots:
        for w in ws:
            ids += w
            w_off.append(len(ids))
        s_off.append(len(w_off) - 1)
    arr = [(ctypes.c_int32 * max(len(a), 1))(*a) for a in (ids, w_off, s_off)]
    out = ctypes.c_void_p()
    rc = L.avs_ctc_grammar_create(arr[0], arr[1], arr[2], len(slots) if n_slots is None else n_slots, vocab, blank,
                                  space, None, ctypes.byref(out))
    return rc, L.avs_last_error_string().decode()


def test_grammar_create_rejects_bad_grammars_without_a_device(native):
    L = native.lib()
    ok = [[[2, 3]], [[4]]]
    long_word = [2] * 65
    for kw, text in (
            ({"slots": ok, "n_slots": 0}, "n_slots must be in [1, 16]"),
            ({"slots": [[[2]]] * 17}, "n_slots must be in [1, 16]"),
            ({"slots": ok, "vocab": 1}, "vocab must be in [2, 64]"),
            ({"slots": ok, "vocab": 65}, "vocab must be in [2, 64]"),
            ({"slots": ok, "blank": 8}, "blank must be in [0, vocab)"),
            ({"slots": ok, "space": 0}, "space must be in [0, vocab) and not the blank"),
            ({"slots": ok, "space": 8}, "space must be in [0, vocab) and not the blank"),
            ({"slots": [[[2]], []]}, "slot 1 has 0 words"),
            ({"slots": [[[2 + i % 6, 2 + i // 6 % 6, 2 + i // 36] for i in range(256)]]}, "slot 0 has 256 words"),
            ({"slots": [[[2], []]]}, "word 1 of slot 0 has 0 ids"),
            ({"slots": [[long_word]]}, "word 0 of slot 0 has 65 ids"),
            ({"slots": [[[2]], [[3, 8]]]}, "word 0 of slot 1 has id 8"),
            ({"slots": [[[2, 0]]]}, "has id 0"),
            ({"slots": [[[1]]]}, "has id 1"),
            ({"slots": [[[-1]]]}, "has id -1"),
            ({"slots": [[[2, 3], [4], [2, 3]]]}, "word 2 of slot 0 appears twice"),
            ({"slots": [[[2] * 64] * 1 + [[3] * 64] * 1] * 8 + [[[4]]]}, "2048")):
        rc, msg = create(L, **kw)
        assert rc == -1 and text in msg, (kw if len(str(kw)) < 200 else text, msg)
    # the state limit counts every chain (2 len + 1) and the G - 1 space states: 2 048 is allowed, 2 049 is not
    words = [[2 + i % 6] * 64 for i in range(6)]                          # 6 x 129 = 774 states per slot
    rc, msg = create(L, [words, words, [[2] * 64, [3] * 64, [4] * 64, [5] * 27, [6] * 28]])
    assert rc == -1 and "2049" in msg, msg


def test_grammar_decode_rejects_bad_arguments_without_a_device(native):
    L = native.lib()

    def call(grammar=FAKE, n_clips=4, n_steps=75):
        rc = L.avs_ctc_grammar_decode(grammar, FAKE, n_clips, n_steps, 39, None, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE,
                                      FAKE, 1 << 40, None)
        return rc, L.avs_last_error_string().decode()

    for kw, text in (({"grammar": None}, "null grammar"), ({"n_clips": -1}, "n_clips must be >= 0"),
                     ({"n_steps": 0}, "n_steps must be in [1, 1024]"), ({"n_steps": 1025}, "n_steps must be in [1, 1024]")):
        rc, msg = call(**kw)
        assert rc == -1 and text in msg, (kw, msg)
    assert L.avs_ctc_grammar_workspace_bytes(None, 4, 75) == 0
    L.avs_ctc_grammar_destroy(None)
