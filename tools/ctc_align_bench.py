"""CTC forced alignment (K5c, ctc_forced_align) on one GPU: 256 and 4 096 GRID-shaped clips per call (T = 75, V = 39,
seeded GRID-sentence targets padded to 40, log-probs of those sentences being spoken, device-resident), timed with CUDA
events.  For scale, on the same input: torch's CUDA ctc_loss (likelihood only, no alignment), and
torchaudio.functional.forced_align on the GPU called once per clip (its kernels take a batch of one; recorded as absent
when this torchaudio has no CUDA kernel for it).  In the same run: the largest loglik / token_prob error against the
float64 oracle and whether frame tokens, spans and path scores equal it.  Reads the card's name and power limit in the
same call.

    python tools/ctc_align_bench.py [--reps 50] [--torchaudio-clips 64] [--out profiles/r06_ctc_align_bench.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import avsync_b200 as A  # noqa: E402
from oracle import ctc_align_ref as R  # noqa: E402
from oracle import ctc_beam_ref  # noqa: E402
from tools.ctc_beam_bench import time_ms  # noqa: E402
from tools.ragged_bench import card  # noqa: E402


def torchaudio_per_clip(lp, targets, lens, n_clips):
    """clips/s of torchaudio.functional.forced_align on the GPU, one call per clip, or the reason it cannot run."""
    try:
        import torchaudio.functional as F
        F.forced_align(lp[:1], targets[:1, :lens[0]], torch.tensor([lp.shape[1]], device=lp.device),
                       lens[:1], blank=0)
    except Exception as e:  # noqa: BLE001
        return {"available": False, "reason": f"{type(e).__name__}: {e}"[:300]}
    T = torch.tensor([lp.shape[1]], device=lp.device)
    lens_h = lens.cpu().tolist()

    def run():
        for b in range(n_clips):
            F.forced_align(lp[b:b + 1], targets[b:b + 1, :lens_h[b]], T, lens[b:b + 1], blank=0)
    run()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run()
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    return {"available": True, "clips": n_clips, "clips_per_s": round(n_clips / s, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--torchaudio-clips", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    A._native.device_check()
    torch.cuda.set_device(0)
    from avsync_b200.dataset import create_vocab
    c2i = create_vocab()[0]
    res = {"card": card(), "T": 75, "V": 39, "Lmax": 40, "reps": args.reps, "cases": []}
    for n in (256, 4096):
        sentences, tg_h, lens_h = R.grid_targets(n, c2i, seed=n, lmax=40)
        lp_h = ctc_beam_ref.grid_sentence_logp(sentences, c2i, seed=n + 1)
        lp = torch.from_numpy(lp_h).cuda()
        tg, lens = torch.from_numpy(tg_h).cuda(), torch.from_numpy(lens_h).cuda()
        inl = torch.full((n,), 75, dtype=torch.int32, device="cuda")
        ms = time_ms(lambda: A.ctc_forced_align(lp, tg, lens), args.reps)
        lp_tb = lp.transpose(0, 1)
        tg64, lens64, inl64 = tg.long(), lens.long(), inl.long()
        ms_loss = time_ms(lambda: torch.nn.functional.ctc_loss(lp_tb, tg64, inl64, lens64, reduction="none"), args.reps)
        row = {"clips": n, "ctc_forced_align_ms": round(ms, 4), "ctc_forced_align_clips_per_s": round(n / ms * 1e3),
               "torch_ctc_loss_cuda_ms": round(ms_loss, 4), "torch_ctc_loss_cuda_clips_per_s": round(n / ms_loss * 1e3)}
        if n == 256:
            row["torchaudio_forced_align_gpu_per_clip"] = torchaudio_per_clip(lp, tg, lens, args.torchaudio_clips)
            got = [t.cpu().numpy() for t in A.ctc_forced_align(lp, tg, lens)]
            want = R.align_batch(lp_h, tg_h, lens_h)
            fin = np.isfinite(want[4])
            row.update({
                "oracle_clips": n,
                "frame_token_span_path_score_equal": bool(np.array_equal(got[2], want[2])
                                                          and np.array_equal(got[3], want[3])
                                                          and np.array_equal(got[1], want[1].astype(np.float32))),
                "max_rel_loglik_err": float(np.max(np.abs(got[0] - want[0]) / np.maximum(np.abs(want[0]), 1.0))),
                "max_rel_token_prob_err": float(np.max(np.abs(got[4][fin] - want[4][fin]) / want[4][fin])),
                "loglik_range": [float(want[0].min()), float(want[0].max())]})
        res["cases"].append(row)
        print(json.dumps(row), flush=True)
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
