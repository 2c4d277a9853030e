"""float64 numpy restatement of K5c, the CTC forced aligner of ``csrc/ctc_align.cu``, and a brute-force check of it.

TEST INFRASTRUCTURE (oracle).  ``align`` runs the same two recurrences over the extended target (blank, y0, blank, y1,
..., blank): the forward (log-sum-exp) for the log-likelihood and the Viterbi (max-plus) for the best path, with the
same skip rule (s-2 only into a non-blank state whose label differs from that of s-2), the same tie rule (stay, then
s-1, then s-2; the trailing blank wins a tie at the end), NaN read as -inf, the same per-clip statuses, spans and token
probabilities.  The Viterbi adds are the kernel's adds in the kernel's order, so path scores and decisions are
bit-identical to the kernel's fp64 state.  ``brute_force`` does not use the lattice: it enumerates every frame labelling
of a tiny problem that collapses to the target.
"""
from __future__ import annotations

import itertools
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import numpy as np

from oracle import ctc_beam_ref

NEG_INF = -np.inf


class Alignment(NamedTuple):
    loglik: float
    path_score: float
    frame_token: np.ndarray   # int32 [T]: target position, -1 blank, -2 at or past input_len (all -2 without alignment)
    span: np.ndarray          # int32 [L, 2]
    token_prob: np.ndarray    # float64 [L]


def _unaligned(T: int, L: int, score: float) -> Alignment:
    return Alignment(score, score, np.full(T, -2, np.int32), np.full((L, 2), -1, np.int32), np.full(L, np.nan))


def _shift(x: np.ndarray, k: int) -> np.ndarray:   # x[s - k], -inf where s < k
    out = np.full_like(x, NEG_INF)
    out[k:] = x[:max(len(x) - k, 0)]
    return out


def align(logp: np.ndarray, y: Sequence[int], input_len: Optional[int] = None, blank: int = 0) -> Alignment:
    """One clip: logp [T, V] float32 or float64, target y (L ids).  The statuses of K5c: an invalid target or length
    gives NaN scores, a target without an alignment of non-zero probability gives -inf scores."""
    lp = np.where(np.isnan(logp), NEG_INF, np.asarray(logp, dtype=np.float64))
    T, V = lp.shape
    y = np.asarray(y, dtype=np.int64)
    L = len(y)
    n = T if input_len is None else int(input_len)
    if not 0 <= n <= T or ((y < 0) | (y >= V) | (y == blank)).any():
        return _unaligned(T, L, np.nan)
    if n == 0:
        return Alignment(0.0, 0.0, np.full(T, -2, np.int32), np.full((L, 2), -1, np.int32), np.full(L, np.nan)) \
            if L == 0 else _unaligned(T, L, NEG_INF)
    S = 2 * L + 1
    lab = np.full(S, blank, np.int64)
    lab[1::2] = y
    skip = np.zeros(S, bool)
    skip[3::2] = y[1:] != y[:-1]
    a = np.full(S, NEG_INF)
    a[:min(S, 2)] = lp[0, lab[:2]]
    v = a.copy()
    bp = np.zeros((n, S), np.int8)
    with np.errstate(invalid="ignore"):
        for t in range(1, n):
            x = lp[t, lab]
            v1, v2 = _shift(v, 1), np.where(skip, _shift(v, 2), NEG_INF)
            best, b = v.copy(), np.zeros(S, np.int8)
            m = v1 > best
            best[m], b[m] = v1[m], 1
            m = v2 > best
            best[m], b[m] = v2[m], 2
            a = np.logaddexp(np.logaddexp(a, _shift(a, 1)), np.where(skip, _shift(a, 2), NEG_INF)) + x
            v = best + x
            bp[t] = b
    end = S - 2 if S > 1 and v[S - 2] > v[S - 1] else S - 1
    if v[end] == NEG_INF:
        return _unaligned(T, L, NEG_INF)
    loglik = float(np.logaddexp(a[S - 1], a[S - 2]) if S > 1 else a[0])
    ft = np.full(T, -2, np.int32)
    s = end
    for t in range(n - 1, -1, -1):
        ft[t] = s // 2 if s & 1 else -1
        s -= int(bp[t, s])
    span = np.full((L, 2), -1, np.int32)
    prob = np.full(L, np.nan)
    for k in range(L):
        f = np.nonzero(ft == k)[0]
        span[k] = f[0], f[-1] + 1
        assert len(f) == f[-1] + 1 - f[0]
        prob[k] = np.exp(lp[f, y[k]]).mean()
    return Alignment(loglik, float(v[end]), ft, span, prob)


def align_batch(logp: np.ndarray, targets: np.ndarray, target_lens: Sequence[int],
                input_lens: Optional[Sequence[int]] = None, blank: int = 0):
    """The layout of ``ctc_forced_align``: logp [B, T, V], targets [B, Lmax] -> (loglik [B], path_score [B] float64,
    frame_token int32 [B, T], span int32 [B, Lmax, 2], token_prob float64 [B, Lmax])."""
    B, T, _ = logp.shape
    Lmax = targets.shape[1]
    ll, ps = np.empty(B), np.empty(B)
    ft = np.empty((B, T), np.int32)
    span = np.full((B, Lmax, 2), -1, np.int32)
    prob = np.full((B, Lmax), np.nan)
    for b in range(B):
        L = int(target_lens[b])
        n = None if input_lens is None else int(input_lens[b])
        if not 0 <= L <= Lmax:
            r = _unaligned(T, 0, np.nan)
        else:
            r = align(logp[b], targets[b, :L], n, blank)
        ll[b], ps[b], ft[b] = r.loglik, r.path_score, r.frame_token
        span[b, :len(r.span)], prob[b, :len(r.span)] = r.span, r.token_prob
    return ll, ps, ft, span, prob


def collapse(labels: Sequence[int], blank: int = 0) -> Tuple[int, ...]:
    out, prev = [], None
    for c in labels:
        if c != prev and c != blank:
            out.append(int(c))
        prev = c
    return tuple(out)


def brute_force(logp: np.ndarray, y: Sequence[int], blank: int = 0) -> Tuple[float, float, np.ndarray]:
    """Every frame labelling of a tiny problem (T <= 8, V <= 4) that collapses to y: (log-likelihood, best path
    log-probability, the best labelling's target position per frame, -1 blank).  Assumes no exact tie for the best."""
    T, V = logp.shape
    assert T <= 8 and V <= 4, "brute_force enumerates every frame labelling: keep it tiny"
    lp = np.asarray(logp, dtype=np.float64)
    y = tuple(int(c) for c in y)
    scores, paths = [], []
    for path in itertools.product(range(V), repeat=T):
        if collapse(path, blank) == y:
            scores.append(sum(lp[t, c] for t, c in enumerate(path)))
            paths.append(path)
    if not scores:
        return NEG_INF, NEG_INF, np.full(T, -2, np.int32)
    i = int(np.argmax(scores))
    ft, k, prev = np.empty(T, np.int32), -1, blank
    for t, c in enumerate(paths[i]):
        if c != blank and c != prev:
            k += 1
        ft[t] = k if c != blank else -1
        prev = c
    return float(np.logaddexp.reduce(scores)), float(scores[i]), ft


def grid_targets(n: int, char_to_idx: Dict[str, int], seed: int = 0, lmax: Optional[int] = None
                 ) -> Tuple[List[str], np.ndarray, np.ndarray]:
    """n seeded GRID sentences (``ctc_beam_ref.grid_sentences``: command colour preposition letter digit adverb) as
    padded targets in the GRID ``collate_fn`` layout: (sentences, targets int32 [n, lmax] zero-padded, lengths [n])."""
    sentences = ctc_beam_ref.grid_sentences(n, seed)
    lens = np.array([len(s) for s in sentences], np.int32)
    lmax = int(lens.max()) if lmax is None else lmax
    targets = np.zeros((n, lmax), np.int32)
    for b, s in enumerate(sentences):
        targets[b, :len(s)] = [char_to_idx[ch] for ch in s]
    return sentences, targets, lens
