"""float64 numpy restatement of K5d, the word-slot grammar decoder of ``csrc/ctc_grammar.cu``, and a brute-force check.

TEST INFRASTRUCTURE (oracle).  ``decode`` builds the same lattice (one chain lb, c0, blank, ..., c_last, tb per word of
each slot, one space state SP_g per slot boundary) and runs the same three recurrences: the backward (log-sum-exp) that
keeps bh[t][SP_g], the forward (log-sum-exp) that gives the log-likelihood and accumulates the word posteriors as paths
leave each word into SP_g, and the Viterbi (max-plus) with the same tie rules (in a chain the stay, then s-1, then s-2;
at SP_g and at the end the stay, then the lowest word index, tb before c_last), NaN read as -inf and the same per-clip
statuses.  The Viterbi adds are the kernel's adds in the kernel's order, so words, spans, path scores and (through the
f32 posteriors) MBR words come out identical.  ``brute_force`` does not use the merged lattice: it enumerates every
sentence of the grammar and scores each with ``ctc_align_ref.align`` (K5c's restatement).
"""
from __future__ import annotations

import itertools
from typing import Dict, List, NamedTuple, Optional, Sequence

import numpy as np

from oracle import ctc_align_ref

NEG_INF = -np.inf


class Lattice(NamedTuple):
    lab: np.ndarray       # [S] label per state; chain states first (words in grammar order), then SP_0 .. SP_{G-2}
    p1: np.ndarray        # [Sc] second Viterbi choice (s-1, or SP_{g-1} for lb), -1 none
    p2: np.ndarray        # [Sc] third choice (s-2 between different labels, or SP_{g-1} for c0), -1 none
    succ1: np.ndarray     # [Sc] s+1 is a successor
    succ2: np.ndarray     # [Sc] s+2 is a successor
    exit: np.ndarray      # [Sc] the SP state tb/c_last of a non-last word leads to, -1 none
    start: np.ndarray     # [Sc] bool
    final: np.ndarray     # [Sc] bool
    word: np.ndarray      # [Sc] word index (grammar order)
    slot: np.ndarray      # [Sc]
    is_label: np.ndarray  # [Sc] bool: a character state
    word_lb: np.ndarray   # [W]
    word_tb: np.ndarray   # [W]
    slot_off: np.ndarray  # [G + 1]
    n_chain: int


def lattice(slots: Sequence[Sequence[Sequence[int]]], blank: int = 0, space: int = 1) -> Lattice:
    """slots[g] lists the words (label id sequences) of slot g."""
    G = len(slots)
    Sc = sum(2 * len(w) + 1 for ws in slots for w in ws)
    lab, p1, p2, start, final, exit_, word, slot, is_label, lb, tb = ([] for _ in range(11))
    w_idx, s, slot_off = 0, 0, [0]
    for g, ws in enumerate(slots):
        sp_in = Sc + g - 1 if g > 0 else -1
        for y in ws:
            n = len(y)
            lb.append(s)
            tb.append(s + 2 * n)
            for k in range(2 * n + 1):
                lab.append(y[k >> 1] if k & 1 else blank)
                p1.append(sp_in if k == 0 else s + k - 1)
                p2.append(sp_in if k == 1 else s + k - 2 if k > 1 and k & 1 and y[k >> 1] != y[(k >> 1) - 1] else -1)
                start.append(k <= 1 and g == 0)
                final.append(k >= 2 * n - 1 and g == G - 1)
                exit_.append(Sc + g if k >= 2 * n - 1 and g < G - 1 else -1)
                word.append(w_idx)
                slot.append(g)
                is_label.append(bool(k & 1))
            s += 2 * n + 1
            w_idx += 1
        slot_off.append(w_idx)
    lab += [space] * (G - 1)
    p1, p2 = np.array(p1, np.int64), np.array(p2, np.int64)
    idx = np.arange(Sc)
    succ1 = np.zeros(Sc, bool)
    succ2 = np.zeros(Sc, bool)
    succ1[:-1] = p1[1:] == idx[:-1]
    succ2[:-2] = p2[2:] == idx[:-2]
    return Lattice(np.array(lab, np.int64), p1, p2, succ1, succ2, np.array(exit_, np.int64), np.array(start, bool),
                   np.array(final, bool), np.array(word, np.int64), np.array(slot, np.int64), np.array(is_label, bool),
                   np.array(lb, np.int64), np.array(tb, np.int64), np.array(slot_off, np.int64), Sc)


class Decode(NamedTuple):
    words: np.ndarray       # int32 [G], -1 without a decode
    span: np.ndarray        # int32 [G, 2]
    path_score: float
    loglik: float
    posterior: np.ndarray   # float64 [W], NaN without a decode
    mbr_words: np.ndarray   # int32 [G]: arg-max of the f32-rounded posteriors per slot, the lowest index on a tie


def _undecoded(G: int, W: int, score: float) -> Decode:
    return Decode(np.full(G, -1, np.int32), np.full((G, 2), -1, np.int32), score, score, np.full(W, np.nan),
                  np.full(G, -1, np.int32))


def _at(x: np.ndarray, idx: np.ndarray) -> np.ndarray:   # x[idx], -inf where idx < 0
    return np.where(idx >= 0, x[np.maximum(idx, 0)], NEG_INF)


def decode(logp: np.ndarray, lat: Lattice, input_len: Optional[int] = None) -> Decode:
    """One clip: logp [T, V] float32 or float64 over the lattice of ``lattice``."""
    lp = np.where(np.isnan(logp), NEG_INF, np.asarray(logp, dtype=np.float64))
    T = lp.shape[0]
    Sc, S = lat.n_chain, len(lat.lab)
    G, W = len(lat.slot_off) - 1, len(lat.word_lb)
    G1 = G - 1
    space = int(lat.lab[Sc]) if G1 else 0
    n = T if input_len is None else int(input_len)
    if not 0 <= n <= T:
        return _undecoded(G, W, np.nan)
    if n == 0:
        return _undecoded(G, W, NEG_INF)
    lab = lat.lab[:Sc]
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        # backward
        bh = np.full(S, NEG_INF)
        bh[:Sc] = np.where(lat.final, lp[n - 1, lab], NEG_INF)
        bsp = np.full((n, G1), NEG_INF)
        for t in range(n - 2, -1, -1):
            nb = np.full(S, NEG_INF)
            terms = np.stack([bh[:Sc], np.where(lat.succ1, np.append(bh[1:Sc], NEG_INF), NEG_INF),
                              np.where(lat.succ2, np.append(bh[2:Sc], [NEG_INF, NEG_INF]), NEG_INF),
                              _at(bh, lat.exit)])
            nb[:Sc] = np.logaddexp.reduce(terms, axis=0) + lp[t, lab]
            for g in range(G1):
                lbs = lat.word_lb[lat.slot_off[g + 1]:lat.slot_off[g + 2]]
                vals = np.concatenate([[bh[Sc + g]], bh[lbs], bh[lbs + 1]])
                nb[Sc + g] = bsp[t, g] = np.logaddexp.reduce(vals) + lp[t, space]
            bh = nb
        starts = np.nonzero(lat.start)[0]
        Z = float(np.logaddexp.reduce(bh[starts]))
        track = Z > NEG_INF

        # forward and Viterbi
        a = np.full(S, NEG_INF)
        a[:Sc] = np.where(lat.start, lp[0, lab], NEG_INF)
        v = a.copy()
        post = np.zeros(W)
        bpc = np.zeros((n, Sc), np.int8)
        bpsp = np.zeros((n, G1), np.int64)
        for t in range(1, n):
            x = lp[t, lab]
            na, nv = np.full(S, NEG_INF), np.full(S, NEG_INF)
            v1, v2 = _at(v, lat.p1), _at(v, lat.p2)
            best, b = v[:Sc].copy(), np.zeros(Sc, np.int8)
            m = v1 > best
            best[m], b[m] = v1[m], 1
            m = v2 > best
            best[m], b[m] = v2[m], 2
            nv[:Sc] = best + x
            bpc[t] = b
            na[:Sc] = np.logaddexp(np.logaddexp(a[:Sc], _at(a, lat.p1)), _at(a, lat.p2)) + x
            xs = lp[t, space]
            for g in range(G1):
                sp, w0, w1 = Sc + g, lat.slot_off[g], lat.slot_off[g + 1]
                tb = lat.word_tb[w0:w1]
                vi = np.stack([v[tb], v[tb - 1]], axis=1).ravel()     # tb(w0), c_last(w0), tb(w1), ...
                k = int(np.argmax(vi))
                if vi[k] > v[sp]:
                    nv[sp], bpsp[t, g] = vi[k] + xs, k + 1
                else:
                    nv[sp] = v[sp] + xs
                ew = np.logaddexp(a[tb], a[tb - 1])
                na[sp] = np.logaddexp(a[sp], np.logaddexp.reduce(ew)) + xs
                if track:
                    post[w0:w1] += np.exp(ew + bsp[t, g] - Z)
            a, v = na, nv
        w0, w1 = lat.slot_off[G - 1], lat.slot_off[G]
        tb = lat.word_tb[w0:w1]
        vi = np.stack([v[tb], v[tb - 1]], axis=1).ravel()
        k = int(np.argmax(vi))
        if not vi[k] > NEG_INF:
            return _undecoded(G, W, NEG_INF)
        end = int(tb[k // 2] - (k & 1))
        path_score = float(vi[k])
        loglik = float(np.logaddexp.reduce(np.concatenate([a[tb], a[tb - 1]])))
        post[w0:w1] = np.exp(np.logaddexp(a[tb], a[tb - 1]) - Z) if track else 0.0
    words = np.full(G, -1, np.int32)
    span = np.full((G, 2), -1, np.int32)
    s = end
    for t in range(n - 1, -1, -1):
        if s < Sc:
            g = lat.slot[s]
            words[g] = lat.word[s] - lat.slot_off[g]
            if lat.is_label[s]:
                if span[g, 1] < 0:
                    span[g, 1] = t + 1
                span[g, 0] = t
            if t > 0:
                s = {0: s, 1: lat.p1[s], 2: lat.p2[s]}[int(bpc[t, s])]
        elif t > 0 and bpsp[t, s - Sc]:
            k = int(bpsp[t, s - Sc]) - 1
            s = int(lat.word_tb[lat.slot_off[s - Sc] + k // 2] - (k & 1))
    p32 = post.astype(np.float32)
    mbr = np.array([int(np.argmax(p32[lat.slot_off[g]:lat.slot_off[g + 1]])) for g in range(G)], np.int32)
    return Decode(words, span, path_score, loglik, post, mbr)


def decode_batch(logp: np.ndarray, lat: Lattice, input_lens: Optional[Sequence[int]] = None):
    """The layout of ``ctc_grammar_decode``: logp [B, T, V] -> (words int32 [B, G], span int32 [B, G, 2], path_score
    float64 [B], loglik float64 [B], posterior float64 [B, W], mbr_words int32 [B, G])."""
    rs = [decode(logp[b], lat, None if input_lens is None else int(input_lens[b])) for b in range(logp.shape[0])]
    return (np.stack([r.words for r in rs]), np.stack([r.span for r in rs]), np.array([r.path_score for r in rs]),
            np.array([r.loglik for r in rs]), np.stack([r.posterior for r in rs]), np.stack([r.mbr_words for r in rs]))


class BruteForce(NamedTuple):
    path_score: float        # the largest K5c path score over the sentences
    loglik: float            # log-sum-exp of the sentences' log-likelihoods
    posterior: np.ndarray    # [W] summed probability of the sentences that hold each word, over the total
    best: List[int]          # word indices (per slot) of the first sentence, in enumeration order, with the best path


def sentences(slots: Sequence[Sequence[Sequence[int]]], space: int):
    """Every sentence of the grammar, slot 0 varying slowest: (word index per slot, label ids)."""
    for choice in itertools.product(*[range(len(ws)) for ws in slots]):
        y = []
        for g, i in enumerate(choice):
            y += ([space] if g else []) + list(slots[g][i])
        yield list(choice), y


def brute_force(logp: np.ndarray, slots: Sequence[Sequence[Sequence[int]]], input_len: Optional[int] = None,
                blank: int = 0, space: int = 1) -> BruteForce:
    off = np.cumsum([0] + [len(ws) for ws in slots])
    lls, pss, choices = [], [], []
    for choice, y in sentences(slots, space):
        r = ctc_align_ref.align(logp, y, input_len, blank)
        lls.append(r.loglik)
        pss.append(r.path_score)
        choices.append(choice)
    lls, pss = np.array(lls), np.array(pss)
    with np.errstate(invalid="ignore", divide="ignore"):
        Z = float(np.logaddexp.reduce(lls))
        post = np.zeros(off[-1])
        for c, ll in zip(choices, lls):
            for g, i in enumerate(c):
                post[off[g] + i] += np.exp(ll - Z)
    i = int(np.argmax(pss))
    return BruteForce(float(pss[i]), Z, post, choices[i])


def slots_to_ids(slots: Sequence[Sequence[str]], char_to_idx: Dict[str, int]) -> List[List[List[int]]]:
    return [[[char_to_idx[ch] for ch in w] for w in ws] for ws in slots]
