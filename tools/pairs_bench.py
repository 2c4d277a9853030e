"""Cross-pair scores (K4x, SyncSweeper.run_pairs / sweep_score_pairs) on one GPU, bf16 STCNN, device-resident u8 frames.

  * 1 024 videos x 1 024 tracks: the time of run_pairs (CUDA events), and the kernel times of the pair kernel, the ha
    kernel and the arg-max pass (torch.profiler, in a run of their own on cached statistics).  The pair kernel's element
    rate (Bv * Ba * K * H per second) is set beside its issue bound, computed from instruction counts (two issue slots
    per element: FADD2 + FFMA2 per two elements, two FMNMX), not measured.
  * 1 x 1 024 and 64 x 64: run_pairs against run on the expanded pairs (every pair cut into one clip), alternated in one
    process; the largest score difference and the best-shift agreement where run's top-2 margin exceeds twice it.
  * The largest error of sweep_score_pairs against float64 (oracle/f64_ref) on the 64 x 64 statistics.
Reads the card's name and power limit in the same call.

    python tools/pairs_bench.py [--reps 5] [--out profiles/r08_pairs_bench.json]
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
from oracle import f64_ref, lipnet_ref, sweep_ref  # noqa: E402
from tools.ctc_beam_bench import time_ms  # noqa: E402
from tools.ragged_bench import card  # noqa: E402

S, H = 20, 512


def kernel_ms(fn, reps):
    """Mean device time per call of each pair kernel, from torch.profiler's CUDA activities."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for k in ("pair_score_kernel", "pair_ha_kernel", "pair_argmax_kernel", "sgemm", "splitk"):
            if k in e.key:
                out[k] = out.get(k, 0.0) + e.device_time_total / 1e3 / reps
    return {k: round(v, 4) for k, v in out.items()}


def compare(ps, pb, rs, rb):
    """run_pairs [n_pairs, K] against run on the cut pairs: largest |difference|, and best-shift equality where run's
    top-2 margin exceeds twice it."""
    err = float((ps - rs).abs().max())
    srt = rs.sort(dim=1).values
    clear = (srt[:, -1] - srt[:, -2]) > 2 * err
    return {"max_abs_diff_vs_run": err, "pairs_resolvable": int(clear.sum()), "pairs": int(rs.shape[0]),
            "best_equal_where_resolvable": bool(torch.equal(pb[clear], rb[clear])),
            "best_equal_all": int((pb == rb).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    A._native.device_check()
    torch.cuda.set_device(0)
    net = A.LipNet(39, precision="bf16")
    net.load_state_dict(lipnet_ref.init_lipnet_state(39, 256, seed=0))
    net = net.cuda().eval()
    det_sd = sweep_ref.init_detector_state(13864, H, seed=1)
    det = A.MisalignmentDetector(13864, H)
    det.load_state_dict(det_sd)
    det = det.cuda().eval()
    sw = A.SyncSweeper(net, det, S, chunk_clips=128)
    K = sw.K
    res = {"card": card(), "precision": "bf16", "K": K, "hidden": H, "chunk_clips": 128, "reps": args.reps}

    n = 1024
    g = torch.Generator().manual_seed(8)
    frames = torch.randint(0, 256, (n, 1, 75, 50, 100), generator=g, dtype=torch.uint8).cuda()
    audio = torch.from_numpy(sweep_ref.synth_audio(n, seed=8, kind="speechlike")).cuda()
    ms = time_ms(lambda: sw.run_pairs(frames, audio), args.reps)
    ms_run = time_ms(lambda: sw.run(frames, audio), args.reps)
    vst, ast = A.visual_stats(net, frames), A.audio_stats_sweep(audio, sw.shifts, 16000, 20)
    ms_score = time_ms(lambda: A.sweep_score_pairs(vst, ast, det), args.reps)
    kern = kernel_ms(lambda: A.sweep_score_pairs(vst, ast, det), args.reps)
    elems = n * n * K * H
    row = {"videos": n, "tracks": n, "run_pairs_ms": round(ms, 3),
           "run_ms_same_clips_own_audio_only": round(ms_run, 3),
           "sweep_score_pairs_ms_on_cached_stats": round(ms_score, 3), "kernel_ms": kern,
           "pair_elements": elems}
    if "pair_score_kernel" in kern:
        row["pair_kernel_elements_per_s"] = elems / (kern["pair_score_kernel"] / 1e3)
        row["pair_kernel_issue_bound_ms_computed_not_measured"] = {
            f"{mhz} MHz": round(elems * 2 / 32 / (148 * 4) / (mhz * 1e6) * 1e3, 3) for mhz in (1965, 1550)}
    res["1024x1024"] = row
    print(json.dumps(row), flush=True)

    for Bv, Ba in ((1, 1024), (64, 64)):
        fr, au = frames[:Bv], audio[:Ba]
        vi = torch.arange(Bv, device="cuda").repeat_interleave(Ba)
        ai = torch.arange(Ba, device="cuda").repeat(Bv)
        fe, ae = fr[vi].contiguous(), au[ai].contiguous()
        ms_p, ms_r = [], []
        for _ in range(2):                       # alternated
            ms_p.append(time_ms(lambda: sw.run_pairs(fr, au), args.reps))
            ms_r.append(time_ms(lambda: sw.run(fe, ae), args.reps))
        ps, pb = sw.run_pairs(fr, au)
        rs, rb = sw.run(fe, ae)
        row = {"videos": Bv, "tracks": Ba, "run_pairs_ms": [round(x, 3) for x in ms_p],
               "run_on_expanded_pairs_ms": [round(x, 3) for x in ms_r],
               **compare(ps.reshape(-1, K), pb.reshape(-1), rs, rb)}
        if Bv == 64:
            v64, a64 = A.visual_stats(net, fr), A.audio_stats_sweep(au, sw.shifts, 16000, 20)
            got = A.sweep_score_pairs(v64, a64, det)[0].cpu().numpy()
            w = [det_sd[k] for k in ("classifier.0.weight", "classifier.0.bias", "classifier.3.weight", "classifier.3.bias")]
            vd, ad = v64.double().cpu(), a64.double().cpu()
            want = np.concatenate([f64_ref.detector_scores_f64(*w, vd[i:i + 8].repeat_interleave(Ba, 0),
                                                               ad.repeat(vd[i:i + 8].shape[0], 1, 1)).reshape(-1, Ba, K)
                                   for i in range(0, Bv, 8)])
            row["sweep_score_pairs_max_abs_err_vs_f64"] = float(np.abs(got - want).max())
            row["score_range"] = [float(want.min()), float(want.max())]
        res[f"{Bv}x{Ba}"] = row
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
