"""Windowed sync sweep on one GPU: SyncSweeper.run_windows on a seeded 10-minute recording (15 000 u8 frames, 9.6 M
samples at 16 kHz, device-resident) at strides of 25 and 75 frames, read at 25 fps and at 29.97 fps.  In the same
process and alternated with each case, the do-it-yourself path: cut the windows by hand (a copy of every window's
frames and audio) and score them with SyncSweeper.run_ragged; the outputs of the two paths are compared for equality.
Reports windows/s of each, per-kernel times (avs_prof_*), the K1 unique frames per window of the windowed plan against
the cut clips', the plan times, and the card's name and power limit read in the same call.

    python tools/window_bench.py [--steps 5] [--rounds 3] [--out profiles/r04_window_bench.json]
"""
import argparse
import ctypes
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import avsync_b200 as A  # noqa: E402
from avsync_b200.misalignment_detection_train import mfcc_window_plan  # noqa: E402
from oracle import lipnet_ref, sweep_ref  # noqa: E402
from tools.ragged_bench import SLOTS, card  # noqa: E402


def unique_frames(T, n_audio, fps, stride, group, sr=16000, S=20):
    """K1 unique frames per window: the windowed plan (groups of `group` windows) against the cut clips' ragged plan."""
    L = A._native.lib()
    i32, i64 = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
    _, a0, a1 = A.window_bounds(T, n_audio, fps, sr, stride)
    W = len(a0)
    row = np.array([A.shift_samples(k, fps, sr) for k in range(-S, S + 1)], dtype=np.int32)
    a0 = np.ascontiguousarray(a0, np.int64)
    ln = np.ascontiguousarray(a1 - a0, np.int32)
    nf, gu = np.zeros(W, np.int32), np.zeros((W + group - 1) // group, np.int32)
    t0 = time.perf_counter()
    A._native.check(L.avs_mfcc_ragged_plan_describe_windows(W, n_audio, a0.ctypes.data_as(i64), ln.ctypes.data_as(i32), group, sr,
                                                            row.ctypes.data_as(i32), len(row), nf.ctypes.data_as(i32),
                                                            gu.ctypes.data_as(i32), None, None), "describe_windows")
    host_ms = (time.perf_counter() - t0) * 1e3
    rows = np.repeat(row[None], W, axis=0)
    off, nfr, nu = np.zeros(W + 1, np.int64), np.zeros(W, np.int32), np.zeros(W, np.int32)
    A._native.check(L.avs_mfcc_ragged_plan_describe(W, ln.ctypes.data_as(i32), sr, rows.ctypes.data_as(i32), rows.shape[1],
                                                    off.ctypes.data_as(i64), nfr.ctypes.data_as(i32), nu.ctypes.data_as(i32),
                                                    None, None), "describe")
    return {"windows": W, "windowed_unique_per_window": round(float(gu.sum()) / W, 1),
            "cut_clips_unique_per_window": round(float(nu.mean()), 1), "host_plan_ms": round(host_ms, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=15000)
    ap.add_argument("--samples", type=int, default=9_600_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=128)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    A._native.device_check()
    dev = torch.device("cuda", 0)
    S, T = 20, args.frames
    net = A.LipNet(39, precision=args.precision)
    net.load_state_dict(lipnet_ref.init_lipnet_state(39, 256, seed=0))
    net = net.to(dev).eval()
    det = A.MisalignmentDetector(13864, 512)
    det.load_state_dict(sweep_ref.init_detector_state(13864, 512, seed=1))
    det = det.to(dev).eval()
    g = torch.Generator().manual_seed(0)
    frames = torch.randint(0, 256, (T, 50, 100), generator=g, dtype=torch.uint8).to(dev)
    audio = torch.from_numpy(np.resize(sweep_ref.synth_audio(1, seed=0, n_samples=480000, kind="speechlike")[0],
                                       args.samples).astype(np.float32)).to(dev)
    sw = A.SyncSweeper(net, det, S, 48000, chunk_clips=args.chunk)

    def diy(fps, stride):
        t, a0, a1 = A.window_bounds(T, audio.numel(), fps, 16000, stride)
        cut = torch.stack([frames[int(x):int(x) + 75] for x in t])[:, None]
        return sw.run_ragged(cut, [audio[int(s):int(e)] for s, e in zip(a0, a1)], fps)

    cases = {}
    for fps in (25.0, 29.97):
        for stride in (25, 75):
            cases[f"windows_{fps}fps_stride{stride}"] = (lambda f=fps, s=stride: sw.run_windows(frames, audio, f, s)[:2])
            cases[f"diy_cut_ragged_{fps}fps_stride{stride}"] = (lambda f=fps, s=stride: diy(f, s))
    out = {"card": card(), "recording": {"frames": T, "samples": args.samples, "sample_rate": 16000},
           "shifts": 2 * S + 1, "precision": args.precision, "chunk_clips": args.chunk, "frames": "u8, device-resident"}
    plan_ms = {}
    for fps in (25.0, 29.97):
        for stride in (25, 75):
            row = [A.shift_samples(k, fps, 16000) for k in range(-S, S + 1)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mfcc_window_plan(T, audio.numel(), fps, stride, 16000, 20, row, args.chunk)
            torch.cuda.synchronize()
            plan_ms[f"{fps}fps_stride{stride}"] = round((time.perf_counter() - t0) * 1e3, 1)
    out["window_plan_create_ms_incl_upload"] = plan_ms
    out["k1_unique_frames"] = {f"{fps}fps_stride{stride}": unique_frames(T, args.samples, fps, stride, args.chunk)
                               for fps in (25.0, 29.97) for stride in (25, 75)}
    for fn in cases.values():                                         # warm-up: modules, plans, buffers
        fn()
        fn()
    torch.cuda.synchronize()
    n_win = {k: int(v()[0].shape[0]) for k, v in cases.items()}
    res = {k: [] for k in cases}
    outputs = {}
    for _ in range(args.rounds):                                      # every case once per round, windowed then DIY
        for name, fn in cases.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                outputs[name] = fn()
            torch.cuda.synchronize()
            res[name].append(n_win[name] * args.steps / (time.perf_counter() - t0))
    out["windows_per_s"] = {k: {"windows": n_win[k], "median": round(float(np.median(v)), 1), "all": [round(x, 1) for x in v]}
                            for k, v in res.items()}
    out["windowed_equals_diy"] = {}
    for k in cases:
        if k.startswith("windows_"):
            d = outputs["diy_cut_ragged_" + k[len("windows_"):]]
            out["windowed_equals_diy"][k] = bool(torch.equal(outputs[k][0], d[0]) and torch.equal(outputs[k][1], d[1]))
    L = A._native.lib()
    kernels = {}
    for name, fn in cases.items():                                    # a separate, profiled step per case
        L.avs_prof_enable(1)
        L.avs_prof_reset()
        fn()
        torch.cuda.synchronize()
        ms, cnt, row = ctypes.c_double(), ctypes.c_int(), {}
        for slot, sname in enumerate(SLOTS):
            if L.avs_prof_read(slot, ctypes.byref(ms), ctypes.byref(cnt)) == 0 and cnt.value:
                row[sname] = {"ms": round(ms.value, 3), "launches": cnt.value}
        L.avs_prof_enable(0)
        kernels[name] = row
    out["kernel_ms_per_step"] = kernels
    b = outputs["windows_25.0fps_stride25"][1]
    out["best_offset_histogram_25fps_stride25"] = np.bincount((b + S).cpu().numpy(), minlength=2 * S + 1).tolist()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")
    if not all(out["windowed_equals_diy"].values()):
        raise SystemExit("windowed outputs differ from the cut-and-run_ragged outputs")


if __name__ == "__main__":
    main()
