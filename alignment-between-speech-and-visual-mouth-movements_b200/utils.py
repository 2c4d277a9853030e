"""`utils.decode_prediction` drop-in (reference: utils.py:8-36) + the batched decode it is built on, exact decoding
under a word-slot grammar, and CTC forced alignment of known transcripts."""
from __future__ import annotations

import ctypes
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N


def ctc_greedy_decode(logp: torch.Tensor, blank_index: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """Batched greedy CTC decode (K5).  logp [B,T,V] CUDA f32 -> (ids int32 [B,T] padded with -1,
    lengths int32 [B]).  One launch and no host sync, instead of the reference's per-sample
    ``.cpu().numpy()`` + Python loop (utils.py:20-30)."""
    N.require_cuda(logp, "logp")
    if logp.dim() != 3:
        raise ValueError("logp must be [B, T, V]")
    logp = N.f32c(logp)
    B, T, V = logp.shape
    ids = torch.empty((B, T), dtype=torch.int32, device=logp.device)
    lens = torch.empty((B,), dtype=torch.int32, device=logp.device)
    if B:
        N.check(N.lib().avs_ctc_greedy(N.ptr(logp), B, T, V, int(blank_index), N.ptr(ids), N.ptr(lens),
                                       N.stream_ptr()), "ctc_greedy")
    return ids, lens


def ids_to_text(ids: List[int], dataset) -> str:
    """utils.py:33-34 — id -> char through ``dataset.idx_to_char`` (id 38 renders as '<pad>')."""
    table = dataset.idx_to_char
    return "".join(table.get(i, "") for i in ids if i in table)


def decode_prediction(outputs: torch.Tensor, dataset, blank_index: int = 0) -> str:
    """Same contract as the reference: ``outputs`` [T, V] log-probs of ONE sample -> text."""
    ids, lens = ctc_greedy_decode(outputs.unsqueeze(0), blank_index)
    n = int(lens[0].item())
    return ids_to_text(ids[0, :n].tolist(), dataset)


class CtcLexicon:
    """A word lexicon for ``ctc_beam_decode`` (K5b): the words' character trie, built once and kept on the current CUDA
    device.  ``words`` are strings over the keys of ``char_to_idx``; ``space`` separates words.  ``vocab`` defaults to
    the largest id of ``char_to_idx`` plus one; ``blank_index`` must be the blank the log-probs are decoded with."""

    def __init__(self, words: Sequence[str], char_to_idx: Dict[str, int], space: str = " ",
                 vocab: Optional[int] = None, blank_index: int = 0):
        ids, offsets = [], [0]
        for w in words:
            for ch in w:
                if ch not in char_to_idx:
                    raise ValueError(f"lexicon word {w!r} has a character {ch!r} outside char_to_idx")
                ids.append(char_to_idx[ch])
            offsets.append(len(ids))
        self.words = list(words)
        self.vocab = int(vocab) if vocab is not None else max(char_to_idx.values()) + 1
        self.blank = int(blank_index)
        self.space_id = char_to_idx[space]
        self.device = torch.device("cuda", torch.cuda.current_device())
        N.device_check()
        w_ids = np.asarray(ids if ids else [0], dtype=np.int32)
        w_off = np.asarray(offsets, dtype=np.int32)
        h = ctypes.c_void_p()
        N.check(N.lib().avs_ctc_lexicon_create(w_ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                               w_off.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), len(self.words),
                                               self.vocab, self.blank, self.space_id, N.stream_ptr(), ctypes.byref(h)),
                "ctc_lexicon_create")
        self._handle = N.Handle(h, N.lib().avs_ctc_lexicon_destroy)

    @property
    def handle(self) -> ctypes.c_void_p:
        return self._handle.h


def ctc_beam_decode(logp: torch.Tensor, beam_width: int, top_n: int = 1, blank_index: int = 0,
                    lexicon: Optional[CtcLexicon] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Batched CTC prefix beam search (K5b), optionally constrained to a ``CtcLexicon``.  logp [B,T,V] CUDA log-probs
    (NaN counts as -inf) -> (ids int32 [B, top_n, T] padded with -1, lengths int32 [B, top_n], scores f32 [B, top_n]),
    best first, on the device.  A score is the log-probability of its label sequence summed over the alignments the
    search kept.  With a lexicon only complete texts (words of the lexicon joined by single spaces, or the empty text)
    are returned; a slot with no hypothesis has score -inf and length 0.  One launch, no host sync.
    Limits: 1 <= beam_width <= 128, 1 <= top_n <= beam_width, 2 <= V <= 64, 1 <= T <= 1024."""
    N.require_cuda(logp, "logp")
    if logp.dim() != 3:
        raise ValueError("logp must be [B, T, V]")
    logp = N.f32c(logp)
    B, T, V = logp.shape
    if lexicon is not None and lexicon.device != logp.device:
        raise ValueError(f"the lexicon lives on {lexicon.device}, logp on {logp.device}")
    ids = torch.empty((B, top_n, T), dtype=torch.int32, device=logp.device)
    lens = torch.empty((B, top_n), dtype=torch.int32, device=logp.device)
    scores = torch.empty((B, top_n), dtype=torch.float32, device=logp.device)
    L = N.lib()
    ws = N.workspace(L.avs_ctc_beam_workspace_bytes(B, T, int(beam_width)), logp.device)
    N.check(L.avs_ctc_beam(N.ptr(logp), B, T, V, int(blank_index), int(beam_width), int(top_n),
                           lexicon.handle if lexicon is not None else None, N.ptr(ids), N.ptr(lens), N.ptr(scores),
                           N.ptr(ws), ws.numel(), N.stream_ptr()), "ctc_beam")
    return ids, lens, scores


class CtcAlignment(NamedTuple):
    """``ctc_forced_align`` outputs, on the device.  Per clip b, along the best (Viterbi) alignment:
    loglik f32 [B] log p(target | logp) over all alignments (= -ctc_loss); path_score f32 [B] the best alignment's
    log-probability; frame_token i32 [B, T] the target position each frame emits (-1 blank, -2 at or past input_len);
    span i32 [B, Lmax, 2] each token's first frame and end frame (exclusive), -1 past the target; token_prob f32
    [B, Lmax] the mean of exp(logp[t, token]) over the token's frames, NaN past the target.  An invalid clip (an id
    outside [0, V) or equal to the blank, a length out of range) has NaN scores; a clip without an alignment of
    non-zero probability has -inf scores; both have frame_token -2, span -1 and token_prob NaN."""
    loglik: torch.Tensor
    path_score: torch.Tensor
    frame_token: torch.Tensor
    span: torch.Tensor
    token_prob: torch.Tensor


def _i32_on(t: torch.Tensor, device) -> torch.Tensor:
    return t.to(device=device, dtype=torch.int32).contiguous()


def ctc_forced_align(logp: torch.Tensor, targets: torch.Tensor, target_lens: torch.Tensor,
                     input_lens: Optional[torch.Tensor] = None, blank_index: int = 0) -> CtcAlignment:
    """Batched CTC forced alignment (K5c) of known targets.  logp [B,T,V] CUDA log-probs (NaN counts as -inf);
    targets [B, Lmax] padded label ids and target_lens [B], the layout ``ctc_loss`` and the GRID ``collate_fn`` use;
    input_lens [B] valid frames per clip (default T).  Returns a ``CtcAlignment`` of device tensors.  One launch and no
    host sync when the index tensors are int32 on logp's device (others are converted first).
    Limits: 1 <= T <= 1024, 2 <= V <= 64, 0 <= Lmax <= 512."""
    N.require_cuda(logp, "logp")
    if logp.dim() != 3:
        raise ValueError("logp must be [B, T, V]")
    logp = N.f32c(logp)
    B, T, V = logp.shape
    dev = logp.device
    if targets.dim() != 2 or targets.shape[0] != B:
        raise ValueError(f"targets must be [B={B}, Lmax], got {tuple(targets.shape)}")
    if tuple(target_lens.shape) != (B,) or (input_lens is not None and tuple(input_lens.shape) != (B,)):
        raise ValueError(f"target_lens and input_lens must be [B={B}]")
    Lmax = targets.shape[1]
    targets, target_lens = _i32_on(targets, dev), _i32_on(target_lens, dev)
    input_lens = _i32_on(input_lens, dev) if input_lens is not None else None
    out = CtcAlignment(torch.empty((B,), dtype=torch.float32, device=dev),
                       torch.empty((B,), dtype=torch.float32, device=dev),
                       torch.empty((B, T), dtype=torch.int32, device=dev),
                       torch.empty((B, Lmax, 2), dtype=torch.int32, device=dev),
                       torch.empty((B, Lmax), dtype=torch.float32, device=dev))
    L = N.lib()
    ws = N.workspace(L.avs_ctc_align_workspace_bytes(B, T, Lmax), dev)
    N.check(L.avs_ctc_align(N.ptr(logp), B, T, V, int(blank_index), N.ptr(input_lens), N.ptr(targets), Lmax,
                            N.ptr(target_lens), *(N.ptr(t) for t in out), N.ptr(ws), ws.numel(), N.stream_ptr()),
            "ctc_align")
    return out


class _CtcLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, log_probs, targets, input_lengths, target_lengths, blank, reduction, zero_infinity):
        B, T, V = log_probs.shape
        L = N.lib()
        nll = torch.empty((B,), dtype=torch.float32, device=log_probs.device)
        ws = N.workspace(L.avs_ctc_loss_workspace_bytes(B, T, targets.shape[1]), log_probs.device)
        N.check(L.avs_ctc_loss(N.ptr(log_probs), B, T, V, blank, N.ptr(input_lengths), N.ptr(targets), targets.shape[1],
                               N.ptr(target_lengths), None, int(zero_infinity), N.ptr(nll), None, N.ptr(ws), ws.numel(),
                               N.stream_ptr()), "ctc_loss")
        ctx.save_for_backward(log_probs, targets, input_lengths, target_lengths)
        ctx.blank, ctx.reduction, ctx.zero_infinity = blank, reduction, zero_infinity
        if reduction == "none":
            return nll
        if reduction == "sum":
            return nll.sum()
        return (nll / target_lengths.clamp(min=1)).mean()

    @staticmethod
    def backward(ctx, grad_out):
        log_probs, targets, input_lengths, target_lengths = ctx.saved_tensors
        B, T, V = log_probs.shape
        if ctx.reduction == "none":
            scale = grad_out
        elif ctx.reduction == "sum":
            scale = grad_out.expand(B)
        else:
            scale = grad_out / (target_lengths.clamp(min=1) * B)
        scale = scale.to(torch.float32).contiguous()
        L = N.lib()
        nll = torch.empty((B,), dtype=torch.float32, device=log_probs.device)
        grad = torch.empty_like(log_probs)
        ws = N.workspace(L.avs_ctc_loss_workspace_bytes(B, T, targets.shape[1]), log_probs.device)
        N.check(L.avs_ctc_loss(N.ptr(log_probs), B, T, V, ctx.blank, N.ptr(input_lengths), N.ptr(targets),
                               targets.shape[1], N.ptr(target_lengths), N.ptr(scale), int(ctx.zero_infinity), N.ptr(nll),
                               N.ptr(grad), N.ptr(ws), ws.numel(), N.stream_ptr()), "ctc_loss")
        return grad, None, None, None, None, None, None


def ctc_loss(log_probs: torch.Tensor, targets: torch.Tensor, input_lengths, target_lengths, blank: int = 0,
             reduction: str = "mean", zero_infinity: bool = False) -> torch.Tensor:
    """CTC loss (K5e) with its gradient, differentiable with respect to ``log_probs``.  Unlike
    ``torch.nn.functional.ctc_loss``, log_probs are batch-first [B, T, V] like LipNet's output (and ``ctc_forced_align``'s
    input), and targets are padded [B, Lmax].  ``reduction`` follows ``F.ctc_loss``: "none" gives the per-clip losses,
    "sum" their sum, "mean" the batch mean of each loss divided by ``target_length.clamp(min=1)``.  ``zero_infinity``
    turns the loss of a clip without an alignment of non-zero probability (+inf, NaN gradient) into 0 with gradient 0.
    An invalid clip (an id outside [0, V) or equal to the blank, a length out of range) and a NaN log-prob inside
    input_length give NaN.  The loss is the float64 forward of K5c, so ``ctc_loss(..., reduction="none")`` equals
    ``-ctc_forced_align(...).loglik`` bit for bit on NaN-free log-probs.  One launch forward, one backward, no host sync.
    Limits: 1 <= T <= 1024, 2 <= V <= 64, 0 <= Lmax <= 512."""
    N.require_cuda(log_probs, "log_probs")
    if log_probs.dim() != 3:
        raise ValueError("log_probs must be [B, T, V] (batch first)")
    if reduction not in ("none", "mean", "sum"):
        raise ValueError(f"reduction must be 'none', 'mean' or 'sum', got {reduction!r}")
    B = log_probs.shape[0]
    dev = log_probs.device
    targets = torch.as_tensor(targets)
    if targets.dim() != 2 or targets.shape[0] != B:
        raise ValueError(f"targets must be padded [B={B}, Lmax], got {tuple(targets.shape)}")
    input_lengths, target_lengths = torch.as_tensor(input_lengths), torch.as_tensor(target_lengths)
    if tuple(input_lengths.shape) != (B,) or tuple(target_lengths.shape) != (B,):
        raise ValueError(f"input_lengths and target_lengths must be [B={B}]")
    lp = log_probs.to(torch.float32).contiguous()
    return _CtcLoss.apply(lp, _i32_on(targets, dev), _i32_on(input_lengths, dev), _i32_on(target_lengths, dev),
                          int(blank), reduction, bool(zero_infinity))


def align_words(logp: torch.Tensor, texts: Sequence[str], char_to_idx: Optional[Dict[str, int]] = None,
                fps: float = 25.0, space: str = " ", blank_index: int = 0, input_lens: Optional[torch.Tensor] = None
                ) -> List[Tuple[List[Tuple[str, float, float, float]], float]]:
    """Word timings of known transcripts in LipNet log-probs [B,T,V]: ``texts[b]`` is aligned to clip b with
    ``ctc_forced_align`` (one upload of the targets, one copy of the results back).  Returns per clip
    ``(words, loglik)``; ``words`` lists ``(word, start_s, end_s, score)`` for every maximal run of non-space
    characters: from its first character's first frame to its last character's end frame, over ``fps``, scored by the
    mean ``token_prob`` of its characters.  A clip without an alignment (loglik -inf, or NaN for an invalid clip)
    keeps its words with NaN times and scores.  ``char_to_idx`` defaults to the GRID vocabulary (``create_vocab``); a
    character outside it raises ``ValueError``."""
    if char_to_idx is None:
        from .dataset import create_vocab
        char_to_idx = create_vocab()[0]
    if len(texts) != logp.shape[0]:
        raise ValueError(f"{len(texts)} texts for {logp.shape[0]} clips")
    B = len(texts)
    for s in texts:
        for ch in s:
            if ch not in char_to_idx:
                raise ValueError(f"character {ch!r} of {s!r} is outside char_to_idx")
    Lmax = max((len(s) for s in texts), default=0)
    host = np.zeros(B * Lmax + B, dtype=np.int32)      # targets [B, Lmax], then target_lens [B]: one upload
    for b, s in enumerate(texts):
        host[b * Lmax:b * Lmax + len(s)] = [char_to_idx[ch] for ch in s]
        host[B * Lmax + b] = len(s)
    dev = torch.from_numpy(host).to(logp.device)
    al = ctc_forced_align(logp, dev[:B * Lmax].view(B, Lmax), dev[B * Lmax:], input_lens, blank_index)
    packed = torch.cat([al.span.view(B, 2 * Lmax), al.token_prob.view(torch.int32),
                        al.loglik.view(torch.int32).view(B, 1)], dim=1).cpu().numpy()   # one copy back
    span = packed[:, :2 * Lmax].reshape(B, Lmax, 2)
    prob = packed[:, 2 * Lmax:3 * Lmax].view(np.float32)
    loglik = packed[:, 3 * Lmax].view(np.float32)
    out = []
    for b, s in enumerate(texts):
        ok = np.isfinite(loglik[b])
        words, k = [], 0
        for w in s.split(space):
            if w:
                a, e = k, k + len(w)
                if ok:
                    words.append((w, float(span[b, a, 0]) / fps, float(span[b, e - 1, 1]) / fps,
                                  float(prob[b, a:e].astype(np.float64).mean())))
                else:
                    words.append((w, float("nan"), float("nan"), float("nan")))
            k += len(w) + len(space)
        out.append((words, float(loglik[b])))
    return out


class CtcGrammar:
    """A word-slot grammar for ``ctc_grammar_decode`` (K5d): ``slots[g]`` lists the words of slot g, and a sentence is
    one word of each slot, in slot order, joined by single spaces.  Its lattice tables are built once and kept on the
    current CUDA device.  Words are strings over the keys of ``char_to_idx`` (a character outside raises
    ``ValueError``); ``space`` separates words.  ``vocab`` defaults to the largest id of ``char_to_idx`` plus one;
    ``blank_index`` must be the blank the log-probs are decoded with.  Limits (checked natively): 1-16 slots, 1-255
    distinct words per slot, 1-64 characters per word, at most 2 048 lattice states (the sum of 2·len + 1 over the words,
    plus one per slot boundary)."""

    def __init__(self, slots: Sequence[Sequence[str]], char_to_idx: Dict[str, int], space: str = " ",
                 vocab: Optional[int] = None, blank_index: int = 0):
        ids, w_off, s_off = [], [0], [0]
        for words in slots:
            for w in words:
                for ch in w:
                    if ch not in char_to_idx:
                        raise ValueError(f"grammar word {w!r} has a character {ch!r} outside char_to_idx")
                    ids.append(char_to_idx[ch])
                w_off.append(len(ids))
            s_off.append(len(w_off) - 1)
        self.slots = [list(words) for words in slots]
        self.space = space
        self.vocab = int(vocab) if vocab is not None else max(char_to_idx.values()) + 1
        self.blank = int(blank_index)
        self.space_id = char_to_idx[space]
        self.device = torch.device("cuda", torch.cuda.current_device())
        N.device_check()
        arrs = [np.asarray(a if a else [0], dtype=np.int32) for a in (ids, w_off, s_off)]
        p = [a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)) for a in arrs]
        h = ctypes.c_void_p()
        N.check(N.lib().avs_ctc_grammar_create(p[0], p[1], p[2], len(self.slots), self.vocab, self.blank,
                                               self.space_id, N.stream_ptr(), ctypes.byref(h)), "ctc_grammar_create")
        self._handle = N.Handle(h, N.lib().avs_ctc_grammar_destroy)

    @property
    def handle(self) -> ctypes.c_void_p:
        return self._handle.h

    @property
    def n_words(self) -> int:
        return sum(len(words) for words in self.slots)

    def texts(self, words) -> List[str]:
        """Word indices [B, G] (``CtcGrammarResult.words`` or ``mbr_words``, a tensor or an array) -> one sentence per
        clip; a clip without a decode (indices -1) gives the empty string."""
        rows = words.tolist() if hasattr(words, "tolist") else list(words)
        return ["" if any(i < 0 for i in row) else self.space.join(s[i] for s, i in zip(self.slots, row))
                for row in rows]


class CtcGrammarResult(NamedTuple):
    """``ctc_grammar_decode`` outputs, on the device.  Per clip b: words i32 [B, G] the word index within each slot along
    the best path; span i32 [B, G, 2] each of those words' first frame and end frame (exclusive), from its first to its
    last character frame; path_score f32 [B] the best path's log-probability; loglik f32 [B] log of the summed
    probability of every sentence of the grammar; posterior f32 [B, W] P(slot g = w) for every word, in grammar order;
    mbr_words i32 [B, G] the per-slot arg-max of posterior (the lowest index on a tie), the decode that minimises the
    expected number of word errors.  A clip whose input length is out of range has NaN scores; one without a path of
    non-zero probability has -inf scores; both have words, span and mbr_words -1 and posterior NaN."""
    words: torch.Tensor
    span: torch.Tensor
    path_score: torch.Tensor
    loglik: torch.Tensor
    posterior: torch.Tensor
    mbr_words: torch.Tensor


def ctc_grammar_decode(logp: torch.Tensor, grammar: CtcGrammar, input_lens: Optional[torch.Tensor] = None,
                       blank_index: int = 0) -> CtcGrammarResult:
    """Exact CTC decoding (K5d) of log-probs [B,T,V] (CUDA; NaN counts as -inf) over every sentence of a ``CtcGrammar``:
    the best sentence (Viterbi) with its word spans, the grammar's log-likelihood and every word's posterior.
    input_lens [B] valid frames per clip (default T).  One launch and no host sync when input_lens is int32 on logp's
    device (otherwise it is converted first).  Limits: 1 <= T <= 1024, V equal to the grammar's vocab."""
    N.require_cuda(logp, "logp")
    if logp.dim() != 3:
        raise ValueError("logp must be [B, T, V]")
    if int(blank_index) != grammar.blank:
        raise ValueError(f"the grammar was built for blank {grammar.blank}, not {blank_index}")
    logp = N.f32c(logp)
    B, T, V = logp.shape
    dev = logp.device
    if grammar.device != dev:
        raise ValueError(f"the grammar lives on {grammar.device}, logp on {dev}")
    if input_lens is not None:
        if tuple(input_lens.shape) != (B,):
            raise ValueError(f"input_lens must be [B={B}]")
        input_lens = _i32_on(input_lens, dev)
    G, W = len(grammar.slots), grammar.n_words
    out = CtcGrammarResult(torch.empty((B, G), dtype=torch.int32, device=dev),
                           torch.empty((B, G, 2), dtype=torch.int32, device=dev),
                           torch.empty((B,), dtype=torch.float32, device=dev),
                           torch.empty((B,), dtype=torch.float32, device=dev),
                           torch.empty((B, W), dtype=torch.float32, device=dev),
                           torch.empty((B, G), dtype=torch.int32, device=dev))
    L = N.lib()
    ws = N.workspace(L.avs_ctc_grammar_workspace_bytes(grammar.handle, B, T), dev)
    N.check(L.avs_ctc_grammar_decode(grammar.handle, N.ptr(logp), B, T, V, N.ptr(input_lens), *(N.ptr(t) for t in out),
                                     N.ptr(ws), ws.numel(), N.stream_ptr()), "ctc_grammar_decode")
    return out


def _check_decoder(beam_width, lexicon, grammar) -> None:
    if grammar is not None and (beam_width is not None or lexicon is not None):
        raise ValueError("grammar decodes exactly: it cannot be combined with beam_width or lexicon")


def decode_batch(outputs: torch.Tensor, dataset, blank_index: int = 0, beam_width: Optional[int] = None,
                 lexicon: Optional[CtcLexicon] = None, grammar: Optional[CtcGrammar] = None) -> List[str]:
    """Decode a whole batch [B,T,V] with one kernel launch and one device->host copy: greedy (K5) by default, the top
    hypothesis of ``ctc_beam_decode`` (K5b) when ``beam_width`` is given, the best sentence of ``grammar`` by
    ``ctc_grammar_decode`` (K5d) when a grammar is given (the empty string for a clip without one)."""
    _check_decoder(beam_width, lexicon, grammar)
    if grammar is not None:
        return grammar.texts(ctc_grammar_decode(outputs, grammar, blank_index=blank_index).words.cpu())
    if beam_width is None:
        ids, lens = ctc_greedy_decode(outputs, blank_index)
    else:
        ids, lens, _ = ctc_beam_decode(outputs, beam_width, 1, blank_index, lexicon)
        ids, lens = ids[:, 0], lens[:, 0]
    ids_h, lens_h = ids.cpu().tolist(), lens.cpu().tolist()
    return [ids_to_text(row[:n], dataset) for row, n in zip(ids_h, lens_h)]


def evaluate_model(model, test_loader, dataset, device, num_samples=5, verbose=True, beam_width=None, lexicon=None,
                   grammar=None):
    """Reference utils.py:38-86 — forward, decode, naive positional character accuracy for the first
    ``num_samples`` items.  One batched decode (K5) per batch instead of one device sync per sample; with
    ``beam_width`` the decode is ``ctc_beam_decode`` (K5b, optionally with ``lexicon``), with ``grammar`` the best
    sentence of that ``CtcGrammar`` (K5d).
    Prints the reference's lines when ``verbose`` and returns [(true_text, predicted_text, accuracy %)]."""
    _check_decoder(beam_width, lexicon, grammar)
    model.eval()
    model.to(device)
    results = []
    if verbose:
        print("\nModel Evaluation:")
        print("-" * 50)
    with torch.no_grad():
        for i, (videos, labels, label_lengths) in enumerate(test_loader):
            if i >= num_samples:
                break
            outputs = model(videos.to(device))
            texts = decode_batch(outputs, dataset, beam_width=beam_width, lexicon=lexicon, grammar=grammar)
            for j in range(videos.size(0)):
                n = i * test_loader.batch_size + j
                if n >= num_samples:
                    break
                true_label = labels[j][:label_lengths[j]]
                true_text = "".join(dataset.idx_to_char.get(int(t), "") for t in true_label if int(t) != 0)
                correct = sum(1 for a, b in zip(true_text, texts[j]) if a == b)
                acc = correct / max(len(true_text), 1) * 100
                results.append((true_text, texts[j], acc))
                if verbose:
                    print(f"\nSample {n + 1}:")
                    print(f"True text: {true_text}")
                    print(f"Predicted text: {texts[j]}")
                    print(f"Character accuracy: {acc:.2f}%")
    return results


def decode_metrics(pred_ids: torch.Tensor, pred_lens: torch.Tensor, target_ids: torch.Tensor, target_lens: torch.Tensor,
                   space_id: int = 37, pad_id: int = 38):
    """Batched CER / WER / positional character accuracy on DEVICE id sequences (SURVEY 8f-3), with the text
    semantics of the reference: ``calculate_cer`` / ``calculate_wer`` (train.py:945-993) on the strings the ids
    render to (id 38 renders as the 5 characters '<pad>'), and ``evaluate_model``'s accuracy (utils.py:83-86).
    Returns a dict of CPU float tensors [B]: cer, wer, char_accuracy (percent), plus the raw int table."""
    for t, n in ((pred_ids, "pred_ids"), (pred_lens, "pred_lens"), (target_ids, "target_ids"), (target_lens, "target_lens")):
        N.require_cuda(t, n)
    pred_ids, target_ids = pred_ids.to(torch.int32).contiguous(), target_ids.to(torch.int32).contiguous()
    pred_lens, target_lens = pred_lens.to(torch.int32).contiguous(), target_lens.to(torch.int32).contiguous()
    B = pred_ids.shape[0]
    out = torch.empty((B, 6), dtype=torch.int32, device=pred_ids.device)
    if B:
        N.check(N.lib().avs_edit_metrics(N.ptr(pred_ids), N.ptr(pred_lens), pred_ids.shape[1], N.ptr(target_ids),
                                         N.ptr(target_lens), target_ids.shape[1], B, space_id, pad_id, 16, 1, 4,
                                         N.ptr(out), N.stream_ptr()), "edit_metrics")
    r = out.cpu().to(torch.float64)
    pred_n, tgt_n, tgt_w = r[:, 5], r[:, 1], r[:, 3]
    cer = torch.where(tgt_n > 0, r[:, 0] / tgt_n.clamp(min=1), (pred_n > 0).to(torch.float64))
    pred_w_nonzero = (r[:, 2] > 0) | (tgt_w > 0)          # target empty: WER = 1 if the prediction has any word
    wer = torch.where(tgt_w > 0, r[:, 2] / tgt_w.clamp(min=1), ((r[:, 2] > 0) & pred_w_nonzero).to(torch.float64))
    acc = r[:, 4] / tgt_n.clamp(min=1) * 100.0
    return {"cer": cer, "wer": wer, "char_accuracy": acc, "raw": out.cpu()}
