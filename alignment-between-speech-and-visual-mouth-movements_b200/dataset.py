"""GPU pre-processing prologue for the path (SURVEY.md section 8f-2): the per-frame arithmetic of the
reference's ``GridDataset.process_video`` (dataset.py:176-256) — gray, mouth crop, bilinear resize to
100x50, /255, pad/truncate to 75 frames — as one kernel, bit-exact with OpenCV's 8-bit paths.
Directory discovery, ``.align`` parsing (``read_grid_align``) and video DECODING stay on the host (file / codec IO)."""
from __future__ import annotations

import ctypes
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N

VOCAB_CHARS = "abcdefghijklmnopqrstuvwxyz0123456789 "


def create_vocab():
    """(char_to_idx, idx_to_char) of GridDataset._create_vocab (dataset.py:38-46): 37 characters -> 1..37,
    '<blank>' = 0, '<pad>' = 38."""
    char_to_idx = {c: i + 1 for i, c in enumerate(VOCAB_CHARS)}
    char_to_idx["<blank>"] = 0
    char_to_idx["<pad>"] = len(VOCAB_CHARS) + 1
    return char_to_idx, {i: c for c, i in char_to_idx.items()}


# The GRID corpus grammar (Cooke et al., 2006): command, colour, preposition, letter (no "w"), digit, adverb.
GRID_SLOTS = [["bin", "lay", "place", "set"], ["blue", "green", "red", "white"], ["at", "by", "in", "with"],
              [c for c in "abcdefghijklmnopqrstuvxyz"],
              ["zero", "one", "two", "three", "four", "five", "six", "seven", "eight", "nine"],
              ["again", "now", "please", "soon"]]
GRID_WORDS = sum(GRID_SLOTS, [])


def grid_lexicon():
    """The 51 GRID words as a ``CtcLexicon`` over ``create_vocab()`` (blank 0, space 37, 39 ids), on the current
    CUDA device, for ``ctc_beam_decode`` / ``decode_batch`` / ``evaluate_model``."""
    from .utils import CtcLexicon
    return CtcLexicon(GRID_WORDS, create_vocab()[0], space=" ")


def grid_grammar():
    """The GRID grammar, six slots of ``GRID_SLOTS`` (64 000 sentences), as a ``CtcGrammar`` over ``create_vocab()``
    (blank 0, space 37, 39 ids), on the current CUDA device, for ``ctc_grammar_decode`` / ``decode_batch`` /
    ``evaluate_model``."""
    from .utils import CtcGrammar
    return CtcGrammar(GRID_SLOTS, create_vocab()[0], space=" ")


def read_grid_align(path: str) -> Tuple[str, List[Tuple[str, float, float]]]:
    """A GRID ``.align`` file -> (text, [(word, start_frame, end_frame)]).  Each line is ``start end word`` with times in
    units of 1/25 000 s, i.e. 1 000 per video frame at 25 fps; frames are those times / 1000, as LipNet's reader divides
    them (GRID boundaries need not fall on frame boundaries).  The silence markers ``sil`` and ``sp`` are dropped;
    ``text`` is the remaining words joined by single spaces, the transcript ``align_words`` takes."""
    words = []
    with open(path) as f:
        for line in f:
            parts = line.split()
            if not parts:
                continue
            if len(parts) != 3:
                raise ValueError(f"{path}: expected 'start end word', got {line.strip()!r}")
            start, end, word = parts
            if word not in ("sil", "sp"):
                words.append((word, int(start) / 1000.0, int(end) / 1000.0))
    return " ".join(w for w, _, _ in words), words


class GridPreprocessor:
    """Decoded uint8 frames -> float32 [B, 1, 75, 50, 100] on the GPU."""

    def __init__(self):
        self._plans: Dict[tuple, N.Handle] = {}
        self.vocab, self.idx_to_char = create_vocab()

    def _plan(self, h: int, w: int, c: int) -> N.Handle:
        key = (torch.cuda.current_device(), h, w, c)
        p = self._plans.get(key)
        if p is None:
            N.device_check()
            hnd = N.c_void_p()
            N.check(N.lib().avs_preproc_create(h, w, c, ctypes.byref(hnd)), "preproc_create")
            p = self._plans[key] = N.Handle(hnd, N.lib().avs_preproc_destroy)
        return p

    def crop_box(self, h: int, w: int, channels: int = 3):
        y0, x0, ch, cw = (ctypes.c_int() for _ in range(4))
        N.check(N.lib().avs_preproc_crop(self._plan(h, w, channels).h, *(ctypes.byref(v) for v in (y0, x0, ch, cw))))
        return y0.value, x0.value, ch.value, cw.value

    def process_batch(self, frames: torch.Tensor, lengths: Optional[torch.Tensor] = None) -> torch.Tensor:
        """frames: CUDA uint8 [B, n, h, w, 3] (BGR) or [B, n, h, w] (gray); lengths: valid frames per clip."""
        N.require_cuda(frames, "frames")
        if frames.dtype != torch.uint8 or frames.dim() not in (4, 5):
            raise RuntimeError("frames must be uint8 [B, n, h, w, 3] or [B, n, h, w]")
        frames = frames.contiguous()
        B, n, h, w = frames.shape[:4]
        c = frames.shape[4] if frames.dim() == 5 else 1
        out = torch.empty((B, 1, 75, 50, 100), dtype=torch.float32, device=frames.device)
        if n == 0:
            return out.zero_()
        ln = None
        if lengths is not None:
            ln = lengths.to(device=frames.device, dtype=torch.int32).contiguous()
        N.check(N.lib().avs_preproc_run(self._plan(h, w, c).h, N.ptr(frames), B, n, N.ptr(ln), N.ptr(out),
                                        N.stream_ptr()), "preproc_run")
        return out

    def process_frames(self, frames: np.ndarray) -> torch.Tensor:
        """One clip of decoded frames (numpy uint8 [n, h, w, 3] or [n, h, w]) -> CUDA float32 [1, 75, 50, 100],
        the tensor ``GridDataset.process_video`` returns for that clip."""
        f = torch.from_numpy(np.ascontiguousarray(frames[:75])).cuda()
        return self.process_batch(f.unsqueeze(0))[0]

    def process_video(self, video_path: str) -> torch.Tensor:
        """Reference entry point (dataset.py:176): ``.npy`` clips of the right shape are normalised and padded
        on the host exactly as the reference does; video files are decoded with cv2 on the host and processed on
        the GPU.  Returns a CPU tensor like the reference."""
        if video_path.endswith(".npy"):
            frames = np.load(video_path)
            if frames.max() > 1.0:
                frames = frames / 255.0
            if frames.shape[1:] != (50, 100):
                raise RuntimeError("pre-processed .npy clips must already be 50 x 100 (float resize is host-side only)")
            frames = frames[:75]
            if len(frames) < 75:
                frames = np.concatenate([frames, np.zeros((75 - len(frames), 50, 100))], axis=0)
            return torch.FloatTensor(frames).unsqueeze(0)
        import cv2
        cap = cv2.VideoCapture(video_path)
        decoded = []
        while len(decoded) < 75:
            ret, frame = cap.read()
            if not ret:
                break
            decoded.append(frame)
        cap.release()
        if not decoded:
            print(f"Warning: No frames extracted from {video_path}")
            return torch.zeros((1, 75, 50, 100))
        return self.process_frames(np.stack(decoded)).cpu()
