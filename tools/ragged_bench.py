"""Ragged sync sweep on one GPU: SyncSweeper.run_ragged on 1024 device-resident clips whose audio lengths are seeded in
[46000, 50000] samples, all at 25 fps and as a 25 / 29.97 fps mix, alternated with SyncSweeper.run on uniform
48000-sample clips in the same process.  Reports clips/s of each, per-kernel times (avs_prof_*), the host plan time and
the card's name and power limit read in the same call.

    python tools/ragged_bench.py [--steps 5] [--rounds 3] [--out profiles/r03_ragged_bench.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import avsync_b200 as A  # noqa: E402
from oracle import lipnet_ref, sweep_ref  # noqa: E402

SLOTS = ["pack", "conv1", "conv2", "conv3", "vstats", "mfcc_logmel", "mfcc_stats", "score_gemm", "score"]


def card():
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        smi = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "name_power_limit_max_sm_clock": smi}


def plan_host_us(lengths, fps, sr=16000, S=20, reps=3):
    """Single-threaded host plan time per clip (avs_mfcc_ragged_plan_describe: the same plan builder as create)."""
    L = A._native.lib()
    i32, i64 = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
    rows = np.array([[A.shift_samples(k, f, sr) for k in range(-S, S + 1)] for f in fps], dtype=np.int32)
    ln = np.asarray(lengths, dtype=np.int32)
    B = len(lengths)
    off, nf, nu = np.zeros(B + 1, np.int64), np.zeros(B, np.int32), np.zeros(B, np.int32)
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        A._native.check(L.avs_mfcc_ragged_plan_describe(B, ln.ctypes.data_as(i32), sr, rows.ctypes.data_as(i32), rows.shape[1],
                                                        off.ctypes.data_as(i64), nf.ctypes.data_as(i32),
                                                        nu.ctypes.data_as(i32), None, None), "describe")
        best = min(best, time.perf_counter() - t0)
    return {"us_per_clip": best / B * 1e6, "unique_frames_per_clip": float(nu.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=128)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    A._native.device_check()
    dev = torch.device("cuda", 0)
    n, S = args.clips, 20
    net = A.LipNet(39, precision=args.precision)
    net.load_state_dict(lipnet_ref.init_lipnet_state(39, 256, seed=0))
    net = net.to(dev).eval()
    det = A.MisalignmentDetector(13864, 512)
    det.load_state_dict(sweep_ref.init_detector_state(13864, 512, seed=1))
    det = det.to(dev).eval()
    g = torch.Generator().manual_seed(0)
    frames = torch.randint(0, 256, (n, 1, 75, 50, 100), generator=g, dtype=torch.uint8).to(dev)
    rng = np.random.default_rng(0)
    lengths = rng.integers(46000, 50001, n)
    audio = [torch.from_numpy(rng.normal(0, 0.1, int(m)).astype(np.float32)).to(dev) for m in lengths]
    audio_uniform = torch.from_numpy(rng.normal(0, 0.1, (n, 48000)).astype(np.float32)).to(dev)
    fps25 = [25.0] * n
    fps_mix = [25.0 if i % 2 == 0 else 29.97 for i in range(n)]
    sw = A.SyncSweeper(net, det, S, 48000, chunk_clips=args.chunk)
    cases = {
        "uniform_run": lambda: sw.run(frames, audio_uniform),
        "ragged_25fps": lambda: sw.run_ragged(frames, audio, fps25),
        "ragged_25_29.97fps": lambda: sw.run_ragged(frames, audio, fps_mix),
    }
    out = {"card": card(), "clips": n, "shifts": 2 * S + 1, "precision": args.precision, "chunk_clips": args.chunk,
           "frames": "u8, device-resident", "lengths": [int(lengths.min()), int(lengths.max())]}
    plan_ms = {}
    for name, fps in (("ragged_25fps", fps25), ("ragged_25_29.97fps", fps_mix)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        A.misalignment_detection_train.mfcc_ragged_plan([int(m) for m in lengths], 16000, 20,
                                                        np.array([[A.shift_samples(k, f, 16000) for k in range(-S, S + 1)]
                                                                  for f in fps], dtype=np.int32))
        torch.cuda.synchronize()
        plan_ms[name] = (time.perf_counter() - t0) * 1e3
    out["plan_create_ms_incl_upload"] = plan_ms
    out["plan_host_25fps"] = plan_host_us(lengths, fps25)
    out["plan_host_25_29.97fps"] = plan_host_us(lengths, fps_mix)
    out["plan_host_29.97fps"] = plan_host_us(lengths, [29.97] * n)
    for fn in cases.values():                                         # warm-up: modules, plans, buffers
        fn()
        fn()
    torch.cuda.synchronize()
    res = {k: [] for k in cases}
    outputs = {}
    for _ in range(args.rounds):                                      # A/B/C alternated
        for name, fn in cases.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                outputs[name] = fn()
            torch.cuda.synchronize()
            res[name].append(n * args.steps / (time.perf_counter() - t0))
    out["clips_per_s"] = {k: {"median": float(np.median(v)), "all": [round(x, 1) for x in v]} for k, v in res.items()}
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
    b_r = outputs["ragged_25fps"][1]
    out["checksums"] = {k: float(v[0].double().sum()) for k, v in outputs.items()}
    out["best_offset_histogram_ragged_25fps"] = np.bincount((b_r + S).cpu().numpy(), minlength=2 * S + 1).tolist()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
