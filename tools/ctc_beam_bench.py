"""CTC prefix beam search (K5b, ctc_beam_decode) on one GPU: 256 and 4 096 clips of seeded peaked log-probs at T = 75,
V = 39 (oracle.ctc_beam_ref.peaked_logp, device-resident), beam widths 8, 32 and 128, with and without the GRID
lexicon, timed with CUDA events; greedy K5 on the same input for scale.  In the same run: the largest |score - float64
oracle| over the first clips of every case, and the oracle itself (oracle/ctc_beam_ref.py) on the host cores — an
unoptimised Python/numpy port kept as the tests' reference, not a CPU decoder baseline.  Reads the card's name and power
limit in the same call.

    python tools/ctc_beam_bench.py [--reps 20] [--oracle-clips 32] [--out profiles/r05_ctc_beam_bench.json]
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
from oracle import ctc_beam_ref as R  # noqa: E402
from tools.ragged_bench import card  # noqa: E402


def time_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--oracle-clips", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    A._native.device_check()
    torch.cuda.set_device(0)
    from avsync_b200.dataset import GRID_WORDS, create_vocab
    lex_g = A.grid_lexicon()
    lex_o = R.Lexicon.from_words(GRID_WORDS, create_vocab()[0])
    res = {"card": card(), "T": 75, "V": 39, "reps": args.reps, "cases": []}
    for n in (256, 4096):
        lp_h = R.peaked_logp(n, 75, 39, seed=n)
        lp = torch.from_numpy(lp_h).cuda()
        g_ms = time_ms(lambda: A.ctc_greedy_decode(lp), args.reps)
        res["cases"].append({"clips": n, "decoder": "greedy K5", "ms": round(g_ms, 4), "clips_per_s": round(n / g_ms * 1e3)})
        for bw in (8, 32, 128):
            for lex in (False, True):
                g, o = (lex_g, lex_o) if lex else (None, None)
                ms = time_ms(lambda: A.ctc_beam_decode(lp, bw, 1, 0, g), args.reps)
                row = {"clips": n, "decoder": "beam K5b", "beam_width": bw, "lexicon": "grid" if lex else None,
                       "ms": round(ms, 4), "clips_per_s": round(n / ms * 1e3)}
                if n == 256:
                    k = args.oracle_clips
                    ids, lens, sc = A.ctc_beam_decode(lp[:k], bw, bw, 0, g)
                    t0 = time.perf_counter()
                    o_ids, o_lens, o_sc, margin = R.beam_search_batch(lp_h[:k], bw, bw, 0, o)
                    host_s = time.perf_counter() - t0
                    ok = margin > 1e-9
                    got = sc.cpu().numpy().astype(np.float64)
                    fin = np.isfinite(o_sc) & ok[:, None]
                    err = np.abs(got[fin] - o_sc[fin])
                    row.update({
                        "oracle_clips": k, "oracle_clips_compared": int(ok.sum()),
                        "ids_equal_on_compared": bool(np.array_equal(ids.cpu().numpy()[ok], o_ids[ok])
                                                      and np.array_equal(lens.cpu().numpy()[ok], o_lens[ok])),
                        "max_abs_score_err": float(err.max()) if err.size else 0.0,
                        "max_rel_score_err": float((err / np.maximum(np.abs(o_sc[fin]), 1.0)).max()) if err.size else 0.0,
                        "python_oracle_port_clips_per_s_host": round(k / host_s, 1)})
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
