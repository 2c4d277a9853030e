"""float64 numpy restatement of K5b, the CTC prefix beam search of ``csrc/ctc_beam.cu``, and a brute-force check of it.

TEST INFRASTRUCTURE (oracle).  ``beam_search`` follows the kernel step for step: the same candidates in the same index
order ((r, c): r = rank of the source beam, c = -1 for the stay, then the non-blank labels in increasing order), the
same exact merge of an extension into the stay of the beam that already is its prefix (at the smaller index), the same
tie rule (score descending, index ascending), the same drop of candidates of score -inf, NaN read as -inf, and the same
lexicon.  It also reports how close each clip came to a different result: the smallest gap between the scores ranked
beam_width and beam_width + 1 over all steps, and between adjacent final ranks.  ``exact_best`` does not search at all:
it enumerates every labeling of a tiny problem and scores it with the CTC forward algorithm.
"""
from __future__ import annotations

import itertools
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

NEG_INF = -np.inf


class Lexicon:
    """Character trie of words given as label ids: ``table[state, c]`` is the state after label c or -1; the space
    column is 0 (back to the root) exactly at word ends.  The same table ``avs_ctc_lexicon_create`` builds."""

    def __init__(self, words: Sequence[Sequence[int]], vocab: int, blank: int, space_id: int):
        rows = [[-1] * vocab]
        for w in words:
            assert len(w) > 0 and all(0 <= c < vocab and c not in (blank, space_id) for c in w), w
            s = 0
            for c in w:
                if rows[s][c] < 0:
                    rows[s][c] = len(rows)
                    rows.append([-1] * vocab)
                s = rows[s][c]
            rows[s][space_id] = 0
        self.table = np.asarray(rows, dtype=np.int64)
        self.words = {tuple(int(c) for c in w) for w in words}
        self.vocab, self.blank, self.space_id = vocab, blank, space_id

    @classmethod
    def from_words(cls, words: Sequence[str], char_to_idx: Dict[str, int], space: str = " ", vocab: Optional[int] = None,
                   blank: int = 0) -> "Lexicon":
        vocab = max(char_to_idx.values()) + 1 if vocab is None else vocab
        return cls([[char_to_idx[ch] for ch in w] for w in words], vocab, blank, char_to_idx[space])

    def is_text(self, ids: Sequence[int]) -> bool:
        """ids are words of the lexicon joined by single spaces (or empty)."""
        if len(ids) == 0:
            return True
        words, cur = [], []
        for c in ids:
            if c == self.space_id:
                words.append(tuple(cur))
                cur = []
            else:
                cur.append(int(c))
        words.append(tuple(cur))
        return all(w in self.words for w in words)


def beam_search(logp: np.ndarray, beam_width: int, top_n: int = 1, blank: int = 0, lexicon: Optional[Lexicon] = None,
                trace: bool = False):
    """One clip: logp [T, V].  Returns (hyps, margin, beams): hyps = top_n pairs (ids tuple, score), best first, padded
    with ((), -inf); margin = the smallest pruning or final-rank gap (inf if nothing was ever cut or ranked); beams = the
    prefixes of every step's beam (as tuples) when ``trace``, else None."""
    lp = np.where(np.isnan(logp), NEG_INF, np.asarray(logp, dtype=np.float64))
    T, V = lp.shape
    labels = np.array([c for c in range(V) if c != blank], dtype=np.int64)
    slot_of = {int(c): j + 1 for j, c in enumerate(labels)}
    trie: Dict[Tuple[int, int], int] = {}
    node_prefix: List[Tuple[int, ...]] = [()]
    # beams in rank order
    node = np.array([0]); pnode = np.array([-1]); lex = np.array([0]); last = np.array([-1]); length = np.array([0])
    lpb = np.array([0.0]); lpnb = np.array([NEG_INF]); prank = np.array([-1])
    margin = np.inf
    beams = [] if trace else None
    with np.errstate(invalid="ignore"):
        for t in range(T):
            nb = len(node)
            if nb == 0:
                break
            row = lp[t]
            sc = np.logaddexp(lpb, lpnb)
            stay_b = sc + row[blank]
            stay_nb = np.where(length > 0, lpnb + row[np.maximum(last, 0)], NEG_INF)
            ext = np.where(labels[None, :] == last[:, None], lpb[:, None], sc[:, None]) + row[labels][None, :]
            if lexicon is not None:
                ext = np.where(lexicon.table[lex][:, labels] >= 0, ext, NEG_INF)
            c_b = np.concatenate([stay_b[:, None], np.full((nb, V - 1), NEG_INF)], axis=1).ravel()
            c_nb = np.concatenate([stay_nb[:, None], ext], axis=1).ravel()
            owner = np.full(nb * V, -1)          # the existing beam a merged candidate is
            owner[np.arange(nb) * V] = np.arange(nb)
            for s in np.nonzero(prank >= 0)[0]:
                e_slot, s_slot = prank[s] * V + slot_of[int(last[s])], s * V
                lo, hi = min(e_slot, s_slot), max(e_slot, s_slot)
                mb, mnb = stay_b[s], np.logaddexp(stay_nb[s], ext[prank[s], slot_of[int(last[s])] - 1])
                c_b[lo], c_nb[lo], owner[lo] = mb, mnb, s
                c_b[hi], c_nb[hi] = NEG_INF, NEG_INF
            score = np.logaddexp(c_b, c_nb)
            valid = np.nonzero(score > NEG_INF)[0]
            order = valid[np.lexsort((valid, -score[valid]))]
            if len(order) > beam_width:
                margin = min(margin, score[order[beam_width - 1]] - score[order[beam_width]])
            order = order[:beam_width]
            n2 = len(order)
            nn, npn, nlex, nlast, nlen = (np.empty(n2, np.int64) for _ in range(5))
            for k, i in enumerate(order):
                r, j = divmod(int(i), V)
                s = owner[i]
                if s >= 0:
                    nn[k], npn[k], nlex[k], nlast[k], nlen[k] = node[s], pnode[s], lex[s], last[s], length[s]
                else:
                    c = int(labels[j - 1])
                    key = (int(node[r]), c)
                    if key not in trie:
                        trie[key] = len(node_prefix)
                        node_prefix.append(node_prefix[node[r]] + (c,))
                    nn[k], npn[k], nlast[k], nlen[k] = trie[key], node[r], c, length[r] + 1
                    nlex[k] = lexicon.table[lex[r], c] if lexicon is not None else 0
            pos = {int(n): k for k, n in enumerate(nn)}
            prank = np.array([pos.get(int(p), -1) if ln > 0 else -1 for p, ln in zip(npn, nlen)], dtype=np.int64)
            node, pnode, lex, last, length = nn, npn, nlex, nlast, nlen
            lpb, lpnb = c_b[order], c_nb[order]
            if trace:
                beams.append([node_prefix[n] for n in node])
    final = np.logaddexp(lpb, lpnb)
    done = [k for k in range(len(node))
            if lexicon is None or length[k] == 0 or lexicon.table[lex[k], lexicon.space_id] >= 0]
    ranked = [final[k] for k in done[:top_n + 1]]
    for a, b in zip(ranked, ranked[1:]):
        margin = min(margin, a - b)
    hyps = [(node_prefix[node[k]], float(final[k])) for k in done[:top_n]]
    hyps += [((), NEG_INF)] * (top_n - len(hyps))
    return hyps, margin, beams


def beam_search_batch(logp: np.ndarray, beam_width: int, top_n: int = 1, blank: int = 0,
                      lexicon: Optional[Lexicon] = None):
    """logp [B, T, V] -> (ids int32 [B, top_n, T] padded with -1, lens [B, top_n], scores float64 [B, top_n],
    margins [B]): the layout of ``ctc_beam_decode``."""
    B, T, _ = logp.shape
    ids = np.full((B, top_n, T), -1, np.int32)
    lens = np.zeros((B, top_n), np.int32)
    scores = np.full((B, top_n), NEG_INF)
    margins = np.empty(B)
    for b in range(B):
        hyps, margins[b], _ = beam_search(logp[b], beam_width, top_n, blank, lexicon)
        for o, (h, s) in enumerate(hyps):
            ids[b, o, :len(h)] = h
            lens[b, o] = len(h)
            scores[b, o] = s
    return ids, lens, scores, margins


def ctc_log_prob(logp: np.ndarray, labels: Sequence[int], blank: int = 0) -> float:
    """log p(labels | logp) by the CTC forward algorithm, float64."""
    lp = np.where(np.isnan(logp), NEG_INF, np.asarray(logp, dtype=np.float64))
    T = lp.shape[0]
    ext = [blank]
    for c in labels:
        ext += [int(c), blank]
    S = len(ext)
    alpha = np.full(S, NEG_INF)
    alpha[0] = lp[0, blank]
    if S > 1:
        alpha[1] = lp[0, ext[1]]
    for t in range(1, T):
        new = np.full(S, NEG_INF)
        for s in range(S):
            a = alpha[s]
            if s >= 1:
                a = np.logaddexp(a, alpha[s - 1])
            if s >= 2 and ext[s] != blank and ext[s] != ext[s - 2]:
                a = np.logaddexp(a, alpha[s - 2])
            new[s] = a + lp[t, ext[s]]
        alpha = new
    return float(np.logaddexp(alpha[-1], alpha[-2]) if S > 1 else alpha[-1])


def exact_best(logp: np.ndarray, blank: int = 0, lexicon: Optional[Lexicon] = None) -> Tuple[Tuple[int, ...], float]:
    """The most probable labeling of a tiny problem (T <= 7, V <= 4) by enumeration, restricted to the texts of
    ``lexicon`` when given: (ids, log-probability).  Ties go to the shorter, then lexicographically smaller labeling."""
    T, V = logp.shape
    assert T <= 7 and V <= 4, "exact_best enumerates every labeling: keep it tiny"
    labels = [c for c in range(V) if c != blank]
    best, best_lp = (), NEG_INF
    for n in range(T + 1):
        for y in itertools.product(labels, repeat=n):
            if lexicon is not None and not lexicon.is_text(y):
                continue
            v = ctc_log_prob(logp, y, blank)
            if v > best_lp:
                best, best_lp = y, v
    return best, best_lp


def peaked_logp(n_clips: int, n_steps: int = 75, vocab: int = 39, seed: int = 0) -> np.ndarray:
    """Seeded synthetic float32 log-probs [n_clips, n_steps, vocab] shaped like a trained CTC head's: per step one label
    (the blank half of the time) near probability 1, two confusers at -0.5 .. -6 and the rest at -12 .. -40."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-40.0, -12.0, size=(n_clips, n_steps, vocab))
    for _ in range(2):
        c = rng.integers(0, vocab, (n_clips, n_steps, 1))
        np.put_along_axis(x, c, rng.uniform(-6.0, -0.5, size=(n_clips, n_steps, 1)), 2)
    top = np.where(rng.random((n_clips, n_steps)) < 0.5, 0, rng.integers(1, vocab, (n_clips, n_steps)))
    np.put_along_axis(x, top[..., None], 0.0, 2)
    return (x - np.logaddexp.reduce(x, axis=2, keepdims=True)).astype(np.float32)


def grid_sentence_logp(sentences: Sequence[str], char_to_idx: Dict[str, int], n_steps: int = 75, vocab: int = 39,
                       flip: float = 0.1, seed: int = 0) -> np.ndarray:
    """Seeded float32 log-probs [len(sentences), n_steps, vocab] of spoken sentences: each character holds for two steps
    (the second a blank when the next character is the same), the rest is blank, with the target's logit 8 above
    unit Gaussian noise.  With probability ``flip`` per character one of its steps has a wrong non-blank label 0.5 to 2
    above the target, so that the per-step arg-max (greedy decoding) spells non-words."""
    rng = np.random.default_rng(seed)
    out = np.empty((len(sentences), n_steps, vocab), np.float32)
    for b, s in enumerate(sentences):
        path = []
        for i, ch in enumerate(s):
            path += [char_to_idx[ch], 0 if s[i + 1:i + 2] == ch else char_to_idx[ch]]
        assert len(path) <= n_steps, s
        x = rng.normal(0.0, 1.0, size=(n_steps, vocab))
        x[np.arange(len(path)), path] += 8.0
        x[len(path):, 0] += 8.0
        for i in range(len(s)):
            if rng.random() < flip:
                t = 2 * i + int(rng.integers(2))
                wrong = int(rng.choice([c for c in range(1, vocab) if c != path[t]]))
                x[t, wrong] = x[t, path[t]] + rng.uniform(0.5, 2.0)
        out[b] = x - np.logaddexp.reduce(x, axis=1, keepdims=True)
    return out


def grid_sentences(n: int, seed: int = 0) -> List[str]:
    """n seeded sentences of the GRID grammar: command colour preposition letter digit adverb."""
    rng = np.random.default_rng(seed)
    cats = [["bin", "lay", "place", "set"], ["blue", "green", "red", "white"], ["at", "by", "in", "with"],
            list("abcdefghijklmnopqrstuvxyz"),
            ["zero", "one", "two", "three", "four", "five", "six", "seven", "eight", "nine"],
            ["again", "now", "please", "soon"]]
    return [" ".join(c[rng.integers(len(c))] for c in cats) for _ in range(n)]
