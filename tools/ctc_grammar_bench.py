"""Exact GRID-grammar decoding (K5d, ctc_grammar_decode) on one GPU: 256 and 4 096 GRID-shaped clips per call (T = 75,
V = 39, log-probs of seeded GRID sentences being spoken, device-resident), timed with CUDA events.  In the same process
and on the same input: the lexicon beam search (K5b, ctc_beam_decode with grid_lexicon()) at beam widths 8 and 128,
and the brute force the grammar decode replaces, all 64 000 GRID sentences aligned with K5c (ctc_forced_align) per
clip, on a few clips.  Also in the same run: equality of words, spans, MBR words and path scores with the float64
restatement on 256 clips and the largest loglik / posterior errors, and how many clips' beam texts break the grammar.
Reads the card's name and power limit in the same call.

    python tools/ctc_grammar_bench.py [--reps 50] [--brute-clips 4] [--out profiles/r07_ctc_grammar_bench.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import avsync_b200 as A  # noqa: E402
from oracle import ctc_beam_ref  # noqa: E402
from oracle import ctc_grammar_ref as R  # noqa: E402
from tools.ctc_beam_bench import time_ms  # noqa: E402
from tools.ragged_bench import card  # noqa: E402


def brute_force_targets(c2i):
    slots = R.slots_to_ids(A.GRID_SLOTS, c2i)
    ys = [y for _, y in R.sentences(slots, c2i[" "])]
    lens = np.array([len(y) for y in ys], np.int32)
    tg = np.zeros((len(ys), lens.max()), np.int32)
    for i, y in enumerate(ys):
        tg[i, :len(y)] = y
    return torch.from_numpy(tg).cuda(), torch.from_numpy(lens).cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--brute-clips", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    A._native.device_check()
    torch.cuda.set_device(0)
    from avsync_b200.dataset import create_vocab
    c2i, i2c = create_vocab()
    grammar, lexicon = A.grid_grammar(), A.grid_lexicon()
    lat = R.lattice(R.slots_to_ids(A.GRID_SLOTS, c2i), 0, c2i[" "])
    res = {"card": card(), "T": 75, "V": 39, "sentences": 64000, "reps": args.reps, "cases": []}
    for n in (256, 4096):
        sentences = ctc_beam_ref.grid_sentences(n, seed=n)
        lp_h = ctc_beam_ref.grid_sentence_logp(sentences, c2i, seed=n + 1)
        lp = torch.from_numpy(lp_h).cuda()
        ms = time_ms(lambda: A.ctc_grammar_decode(lp, grammar), args.reps)
        row = {"clips": n, "ctc_grammar_decode_ms": round(ms, 4), "ctc_grammar_decode_clips_per_s": round(n / ms * 1e3)}
        for bw in (8, 128):
            ms_b = time_ms(lambda: A.ctc_beam_decode(lp, bw, 1, lexicon=lexicon), args.reps)
            row[f"beam{bw}_grid_lexicon_ms"] = round(ms_b, 4)
            row[f"beam{bw}_grid_lexicon_clips_per_s"] = round(n / ms_b * 1e3)
        if n == 256:
            got = [t.cpu().numpy() for t in A.ctc_grammar_decode(lp, grammar)]
            want = R.decode_batch(lp_h, lat)
            fin = np.isfinite(want[4])
            row.update({
                "oracle_clips": n,
                "words_span_mbr_path_score_equal": bool(np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
                                                        and np.array_equal(got[5], want[5])
                                                        and np.array_equal(got[2], want[2].astype(np.float32))),
                "max_rel_loglik_err": float(np.max(np.abs(got[3] - want[3]) / np.maximum(np.abs(want[3]), 1.0))),
                "max_abs_posterior_err": float(np.max(np.abs(got[4][fin] - want[4][fin]))),
                "loglik_range": [float(want[3].min()), float(want[3].max())],
                "viterbi_sentence_is_the_spoken_one": int(sum(t == s for t, s in zip(grammar.texts(got[0]), sentences))),
                "mbr_sentence_is_the_spoken_one": int(sum(t == s for t, s in zip(grammar.texts(got[5]), sentences)))})
            for bw in (8, 128):
                ids, lens, _ = A.ctc_beam_decode(lp, bw, 1, lexicon=lexicon)
                texts = ["".join(i2c[i] for i in ids[b, 0, :lens[b, 0]].tolist()) for b in range(n)]
                row[f"beam{bw}_text_is_the_spoken_one"] = int(sum(t == s for t, s in zip(texts, sentences)))
            tg, tl = brute_force_targets(c2i)
            k = args.brute_clips
            x = lp[:1].expand(tg.shape[0], 75, 39)
            ms_bf = time_ms(lambda: A.ctc_forced_align(x, tg, tl), max(1, args.reps // 10))
            same = 0
            for b in range(k):
                al = A.ctc_forced_align(lp[b:b + 1].expand(tg.shape[0], 75, 39), tg, tl)
                same += float(al.path_score.max()) == float(got[2][b])
            row["k5c_brute_force"] = {"alignments_per_clip": int(tg.shape[0]), "ms_per_clip": round(ms_bf, 3),
                                      "clips_per_s": round(1e3 / ms_bf, 1), "clips_checked": k,
                                      "max_path_score_equals_k5d": same}
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
