#!/usr/bin/env python
"""bench.py — clips/s of the 41-offset (+-20 frame) AV sync sweep (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference]
                    [--precision bf16|bf16x3|fp32] [--clips-per-gpu C] [--chunk M] [--no-configs]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (K2 STCNN + visual stats | K1 MFCC stats for 41 shifts -> K4
scores + arg-max, plus the cross-rank score gather when N > 1) over one batch of synthetic clips:
C clips per GPU, fixed as N grows (weak scaling; N = 8, C = 1024 is BASELINE config 3's 8192 clips).
Prints ONE JSON line (rank 0).  --dump-outputs DIR also writes what the last timed step returned (see dump_outputs):
inputs and weights come from fixed seeds, so two builds run with the same arguments can be compared output for output.

  value      device-resident throughput (inputs already in HBM), CUDA events, max over ranks
  e2e        the same sweep through the host-buffer entry point: pinned host inputs, H2D / D2H inside the timed
             region.  Frames cross PCIe as the uint8 pixels GRID frames are made of (dataset.py:226-231:
             frames = float32(u8 / 255.0)); `e2e_f32_frames` is the same call fed with the f32 tensor instead.
  parity     bf16 (headline dtype) against the fp32-grade bf16x3 path on this very batch, outside the timed region
  configs    the other BASELINE configs (1, 2, 4, 5, the fp32-grade sweep, the drop-in per-shift loop), measured
             after the headline; config 5 (DDP detector step) runs on all N ranks
  roofline   the dominant kernel (conv2) against the measured sustained bf16 rate
  cpu_baseline  the reference's CPU path (oracle port) on this box's host cores, BASELINE.md section 2 protocol
"""
from __future__ import annotations

import os
import sys

if "reference" in sys.argv:
    # The reference arm uses every host core.  torchrun exports OMP_NUM_THREADS=1 to its workers, which would pin the
    # BLAS / OpenMP pools of numpy, scipy and torch to one thread before they initialise (round 1: 3.7 vs 7.4 clips/s
    # between torchrun and plain launches): set the pools explicitly, before those libraries load.
    for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import argparse
import json
import subprocess
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

S_FRAMES = 20
N_SHIFTS = 2 * S_FRAMES + 1
N_SAMPLES = 48000
FRAME_ELEMS = 75 * 50 * 100
METRIC = "clips/sec for 41-offset AV sync sweep"
# algorithmic work per clip (SURVEY.md section 8d): MACs of the three conv layers
CONV_FLOP = {1: 2 * 0.900e9, 2: 2 * 14.400e9, 3: 2 * 3.73248e9}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def conv2_traffic(clips_per_launch: int, precision: str):
    """DRAM bytes per launch of the layer-2 conv kernel: a CONSTANT taken from the committed `ncu --set full` capture
    (profiles/r02_conv2_ncu_full.txt: dram__bytes_read.sum + dram__bytes_write.sum = 746.1 MB for a 64-clip bf16
    launch = 11.66 MB per clip; algorithmic: 8.6 MB padded input + 2.9 MB pooled output), scaled to the clips one
    bench launch processes — not measured by this run."""
    if precision != "bf16":
        return None
    return 11.66e6 * clips_per_launch


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,power.draw.instant,enforced.power.limit")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def count(self):
        """Samples written so far."""
        try:
            return sum(1 for r in open(self.f.name) if r.count(",") >= 8)
        except Exception:
            return 0

    def stop(self, first: int = 0):
        """Stops nvidia-smi and summarises the samples from index `first` on."""
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8][first:]
        os.unlink(self.f.name)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any("Active" == r[5 + j].strip() for r in rows)]
        out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "samples": len(rows),
               "power_w_max": max(float(r[3]) for r in rows), "reasons": reasons}
        try:   # power.draw is nvidia-smi's one-second average and lags a short timed region; the instantaneous reading and
            # the enforced limit show how close to the cap the step runs (profiles/r02_power_trace.txt: 986 of 1000 W)
            out["power_w_instant_max"] = max(float(r[9]) for r in rows)
            out["power_limit_w"] = float(rows[0][10])
        except (ValueError, IndexError):
            pass
        return out


def synth_inputs(n: int, seed: int, pin: bool = True):
    """Host tensors (pinned when a GPU is present): frames u8 [n,1,75,50,100] uniform over 0..255 — the 8-bit mouth crops
    GRID frames are made of; the reference's f32 tensor is float32(u8 / 255.0) (dataset.py:226-231), see frames_f32() —
    and audio [n,48000] ~ N(0,0.1^2) clipped, with a per-clip random amplitude envelope so shifted versions differ
    (SURVEY.md section 8d)."""
    g = torch.Generator().manual_seed(seed)
    pin = pin and torch.cuda.is_available()
    frames = torch.empty((n, 1, 75, 50, 100), dtype=torch.uint8)
    audio = torch.empty((n, N_SAMPLES), dtype=torch.float32)
    if pin:
        frames, audio = frames.pin_memory(), audio.pin_memory()
    for i in range(0, n, 64):
        m = min(64, n - i)
        frames[i:i + m] = torch.randint(0, 256, (m, 1, 75, 50, 100), generator=g, dtype=torch.uint8)
        env = torch.nn.functional.interpolate(torch.rand((m, 1, 13), generator=g), size=N_SAMPLES, mode="linear",
                                              align_corners=True)[:, 0]
        audio[i:i + m] = (torch.randn((m, N_SAMPLES), generator=g) * 0.1).clamp_(-1, 1) * env * env
    return frames, audio


def frames_f32(frames_u8: torch.Tensor, pin: bool = True) -> torch.Tensor:
    """The reference's frames tensor for these pixels: u8 / 255.0 in float64, stored as float32."""
    out = torch.empty(frames_u8.shape, dtype=torch.float32)
    if pin and torch.cuda.is_available():
        out = out.pin_memory()
    for i in range(0, frames_u8.shape[0], 64):
        out[i:i + 64] = (frames_u8[i:i + 64].to(torch.float64) / 255.0).to(torch.float32)
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, scores: np.ndarray, best: np.ndarray):
    """Writes the sweep's results as out_dir/scores.npy (float32 [clips, 41], sigmoid score of every offset) and
    out_dir/best.npy (float64 [clips], best offset in frames).  Should they exceed 64 MB, a fixed seeded sample of
    clips is written instead, with the sampled clip indices in out_dir/clips.npy."""
    os.makedirs(out_dir, exist_ok=True)
    n, k = scores.shape
    row_bytes = 4 * k + 8
    if n * row_bytes > DUMP_BYTES - 4096:                  # 4096: room for the .npy headers
        keep = np.sort(np.random.default_rng(0).choice(n, (DUMP_BYTES - 4096) // (row_bytes + 8), replace=False))
        scores, best = scores[keep], best[keep]
        np.save(os.path.join(out_dir, "clips.npy"), keep.astype(np.float64))
    np.save(os.path.join(out_dir, "scores.npy"), scores.astype(np.float32))
    np.save(os.path.join(out_dir, "best.npy"), best.astype(np.float64))


def parity_stats(scores, best, scores_ref, best_ref):
    """Headline-dtype scores / best offsets against the fp32-grade path on the same clips.  A clip is *resolvable*
    when the reference's top-2 score margin exceeds 10x the largest score difference seen; on those the best offset
    must be identical (north_star: arg-max bit-exact)."""
    scores, scores_ref = np.asarray(scores, dtype=np.float64), np.asarray(scores_ref, dtype=np.float64)
    d = float(np.abs(scores - scores_ref).max())
    srt = np.sort(scores_ref, axis=1)
    margin = srt[:, -1] - srt[:, -2]
    res = margin > 10 * d
    agree = np.asarray(best) == np.asarray(best_ref)
    return {"clips": int(scores.shape[0]), "max_abs_dscore": d, "argmax_agree": float(agree.mean()),
            "resolvable_frac": float(res.mean()),
            "argmax_agree_resolvable": float(agree[res].mean()) if res.any() else None,
            "unresolvable_disagreements": int((~agree & ~res).sum()),
            "median_top2_margin": float(np.median(margin))}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_clip_times(n_clips: int, warm: int, batched: bool, S: int = S_FRAMES):
    """Per-clip wall times of the reference's CPU path (oracle port: B=1 STCNN once per clip, then per shift
    shift_audio -> MFCC stats -> cat -> sigmoid(detector); batched=True is the "best-effort CPU" variant with one
    detector call for all shifts) on this box's host cores."""
    from oracle import lipnet_ref, sweep_ref
    torch.set_num_threads(os.cpu_count() or 1)
    sd = lipnet_ref.init_lipnet_state(39, 256, seed=0)
    det = sweep_ref.init_detector_state(13864, 512, seed=1)
    frames = sweep_ref.synth_frames(n_clips + warm, seed=4321)
    audio = sweep_ref.synth_audio(n_clips + warm, seed=4321, kind="speechlike")
    shifts = list(range(-S, S + 1))
    times = []
    for i in range(warm + n_clips):
        t0 = time.perf_counter()
        sweep_ref.sweep_clip(sd, det, frames[i], audio[i], shifts, batched=batched)
        if i >= warm:
            times.append(time.perf_counter() - t0)
    return times


def cpu_stage_split(n_clips: int = 3):
    """Seconds per clip of the three stages of the reference-style loop (STCNN B=1, 41 MFCC-stats calls, 41 detector calls)."""
    from oracle import lipnet_ref, sweep_ref
    torch.set_num_threads(os.cpu_count() or 1)
    sd = lipnet_ref.init_lipnet_state(39, 256, seed=0)
    det = sweep_ref.init_detector_state(13864, 512, seed=1)
    frames = sweep_ref.synth_frames(n_clips, seed=99)
    audio = sweep_ref.synth_audio(n_clips, seed=99, kind="speechlike")
    t = {"stcnn_b1": 0.0, "mfcc_x41": 0.0, "detector_x41": 0.0}
    with torch.no_grad():
        for i in range(n_clips):
            t0 = time.perf_counter()
            v = sweep_ref.visual_stats(lipnet_ref.stcnn(sd, frames[i].unsqueeze(0))[0])
            t1 = time.perf_counter()
            a = [sweep_ref.compute_audio_stats(sweep_ref.shift_audio(audio[i], k, 25.0, 16000), 16000, 20)
                 for k in range(-S_FRAMES, S_FRAMES + 1)]
            t2 = time.perf_counter()
            for ak in a:
                torch.sigmoid(sweep_ref.detector_logits(det, torch.cat([v, ak]).unsqueeze(0)))
            t3 = time.perf_counter()
            t["stcnn_b1"] += (t1 - t0) / n_clips
            t["mfcc_x41"] += (t2 - t1) / n_clips
            t["detector_x41"] += (t3 - t2) / n_clips
    return t


def run_reference(args, rank: int):
    """--impl reference: the reference's CPU implementation (oracle port; /root/reference is Python and does not exist
    on the GPU box) timed on the host cores with all the threads it can use.  Rank 0 only.  Protocol of BASELINE.md
    section 2: warm-up clips, then >= 16 timed clips (steps x ref-clips), median s/clip -> clips/s; the best-effort
    (batched detector) variant and a per-stage split are reported beside it."""
    if rank != 0:
        return
    per_step = args.ref_clips
    n_timed = max(16, args.steps * per_step)
    t0 = time.perf_counter()
    times = cpu_clip_times(n_timed, warm=max(2, args.warmup), batched=False)
    wall = time.perf_counter() - t0
    med = float(np.median(times))
    v = 1.0 / med
    best_effort = cpu_clip_times(16, warm=2, batched=True)
    s15 = cpu_clip_times(8, warm=1, batched=False, S=15)
    cores = os.cpu_count() or 1
    cpu = {"value": v, "unit": "clips/s", "cores": cores, "kind": "port",
           "sample": f"{n_timed} timed clips after {max(2, args.warmup)} warm-up clips, median s/clip, reference-style loop "
                     f"(oracle port), torch {torch.get_num_threads()} threads, OMP_NUM_THREADS={os.environ.get('OMP_NUM_THREADS')}",
           "mean_value": len(times) / sum(times), "median_s_per_clip": med,
           "best_effort_value": 1.0 / float(np.median(best_effort)),
           "best_effort": "same loop with one batched detector call for the 41 shifts (16 clips, median)",
           "s15_value": 1.0 / float(np.median(s15)),
           "stage_s_per_clip": cpu_stage_split(3)}
    line = {
        "metric": METRIC, "value": v, "unit": "clips/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * med * per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": f"+-{S_FRAMES}-frame (41-offset) sync sweep, reference-style CPU loop, "
                               f"{per_step} clips per step (bounded sample of the 1024-clip step)", "l2": "n/a (CPU)",
                   "wall_s": wall},
        "cpu_baseline": cpu,
        "e2e": {"value": v, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


def cpu_baseline_subprocess(n_clips: int):
    """The cpu_baseline leg of the native arm runs the reference arm in a fresh process (same code, same thread pools:
    this process may have been started with OMP_NUM_THREADS=1) and returns its cpu_baseline object."""
    steps = max(1, (n_clips + 3) // 4)
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", "2"],
                       capture_output=True, text=True, env=env, timeout=900)
    for ln in reversed(r.stdout.strip().splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)["cpu_baseline"]
    return {"value": None, "error": r.stderr[-400:]}


# ------------------------------------------------------------------------------------------------ other configs
def cuda_time(fn, iters: int, warm: int = 2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def other_configs(A, dev, det, frames_u8_h, audio_h, world: int):
    """BASELINE configs 1, 2, 4 and the fp32-grade sweep on this GPU (rank 0, N = 1), device-resident, CUDA events."""
    out = {}
    f32_64 = frames_f32(frames_u8_h[:256], pin=False).to(dev)
    au = audio_h[:256].to(dev)
    nets = {}
    for prec in ("bf16x3", "bf16"):
        torch.manual_seed(0)
        nets[prec] = A.LipNet(39, precision=prec).to(dev).eval()
    # config 1: ONE clip end to end (STCNN + Bi-GRU head + greedy decode + +-15 sweep), fp32-grade
    sw1 = A.SyncSweeper(nets["bf16x3"], det, 15, N_SAMPLES, chunk_clips=1)

    def cfg1():
        lp = nets["bf16x3"](f32_64[:1])
        A.ctc_greedy_decode(lp)
        sw1.run(f32_64[:1], au[:1])
    out["config1_one_clip_ms"] = {"value": cuda_time(cfg1, 20), "unit": "ms/clip", "precision": "bf16x3",
                                  "what": "1 clip: LipNet forward + greedy CTC + +-15 sweep, device-resident"}
    # config 2: 64 clips, +-15, fp32-grade (and bf16 beside it)
    for prec in ("bf16x3", "bf16"):
        sw = A.SyncSweeper(nets[prec], det, 15, N_SAMPLES, chunk_clips=64)
        ms = cuda_time(lambda: sw.run(f32_64[:64], au[:64]), 10)
        out[f"config2_batch64_s15_{prec}"] = {"value": 64 / (ms / 1e3), "unit": "clips/s", "ms_per_step": ms}
    # config 4: 256 clips LipNet.forward + greedy decode
    for prec in ("bf16x3", "bf16"):
        def cfg4(p=prec):
            A.ctc_greedy_decode(nets[p](f32_64))
        ms = cuda_time(cfg4, 5)
        out[f"config4_batch256_decode_{prec}"] = {"value": 256 / (ms / 1e3), "unit": "clips/s", "ms_per_step": ms}
    del f32_64
    return out, nets


def dropin_loop(A, dev, det, net, frames_u8_h, audio_h, n_clips: int = 6):
    """What INTEGRATION.md's two-line import swap buys a maintainer who keeps the reference's per-(clip, shift) loop:
    FeatureExtractor.build_feature(path, k) + sigmoid(detector(feature[None])) for every k (B = 1 STCNN once per clip,
    one K1 launch + one H2D + one D2H per shift), wall clock."""
    class Grid:
        def process_video(self, path):
            return frames_f32(frames_u8_h[int(path):int(path) + 1], pin=False)[0]

    def loader(path):
        return audio_h[int(path)].numpy(), 16000
    fx = A.FeatureExtractor(Grid(), net, dev, A.DetectorConfig(max_shift_frames=S_FRAMES), audio_loader=loader)

    def clip(i):
        with torch.no_grad():
            sc = [float(torch.sigmoid(det(fx.build_feature(str(i), k)[0].to(dev).unsqueeze(0)))[0])
                  for k in range(-S_FRAMES, S_FRAMES + 1)]
        return int(np.argmax(sc))
    clip(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(1, 1 + n_clips):
        clip(i)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"value": n_clips / dt, "unit": "clips/s", "clips": n_clips, "precision": net.precision,
            "what": "per-(clip, shift) loop through the reference-named shims (build_feature + detector), wall clock"}


def ddp_config5(A, dev, world: int, rank: int, steps: int = 20):
    """Config 5: one data-parallel training step of the detector (hidden 512, batch 64 per rank, BCE-with-logits,
    Adam lr 1e-3 / L2 1e-5; run_train_misalignment.sh:32-42, misalignment_detection_train.py:260-266) with ONE
    all-reduce of the flat 28.4 MB gradient bucket; CUDA events, max over ranks.  Also times the bare all-reduce of the
    same bucket to report its share of the step."""
    import torch.distributed as dist
    torch.manual_seed(1)
    det = A.MisalignmentDetector(13864, 512).to(dev)
    opt = torch.optim.Adam(det.parameters(), lr=1e-3, weight_decay=1e-5)
    g = torch.Generator().manual_seed(100 + rank)
    x = torch.randn((64, 13864), generator=g).to(dev)
    y = (torch.rand((64,), generator=g) > 0.5).float().to(dev)
    ms_step = cuda_time(lambda: A.distributed.ddp_detector_step(det, x, y, opt), steps, warm=3)
    n_grad = sum(p.numel() for p in det.parameters())
    ms_ar = 0.0
    if world > 1:
        flat = torch.zeros(n_grad, device=dev)
        ms_ar = cuda_time(lambda: dist.all_reduce(flat), steps, warm=3)
    t = torch.tensor([ms_step, ms_ar], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, ms_ar = float(t[0]), float(t[1])
    out = {"value": ms_step, "unit": "ms/step", "global_batch": 64 * world, "grad_floats": n_grad,
           "allreduce_ms": ms_ar, "allreduce_share": (ms_ar / ms_step) if ms_step else None,
           "allreduce_busbw_gbs": (2 * (world - 1) / world * n_grad * 4 / (ms_ar / 1e3) / 1e9) if ms_ar else None,
           "samples_per_s": 64 * world / (ms_step / 1e3)}
    return out, (det, opt, x, y, steps)



def ddp_config5_graph(A, dev, world: int, rank: int, ctx):
    """The config-5 step captured in one CUDA graph (forward, loss, backward, all-reduce, Adam): the eager step is ~30
    launch-bound torch kernels.  Every rank must take the same branch, so a failure on any rank disables it on all."""
    import torch.distributed as dist
    det, opt, x, y, steps = ctx
    stepper, err = None, ""
    try:
        stepper = A.distributed.GraphedDetectorStep(det, opt, 64)
    except Exception as e:                      # noqa: BLE001 - reported in the line
        err = f"{type(e).__name__}: {e}"[:200]
    ok = torch.tensor([1.0 if stepper is not None else 0.0], device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if float(ok) != 1.0:
        return {"unavailable": err or "capture failed on another rank"}
    ms_g = torch.tensor([cuda_time(lambda: stepper.step(x, y), steps, warm=3)], device=dev)
    flat_p = torch.cat([p.detach().reshape(-1) for p in det.parameters()])
    spread = torch.stack([flat_p.max(), -flat_p.min(), flat_p.double().sum().float()])
    lo = spread.clone()
    if world > 1:
        dist.all_reduce(ms_g, op=dist.ReduceOp.MAX)
        dist.all_reduce(spread, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    return {"value": float(ms_g), "unit": "ms/step", "samples_per_s": 64 * world / (float(ms_g) / 1e3),
            "ranks_in_sync": bool(torch.equal(spread, lo)),
            "what": "the same step as one CUDA graph replay (distributed.GraphedDetectorStep)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "bf16x3", "fp32"])
    ap.add_argument("--clips-per-gpu", type=int, default=1024)
    ap.add_argument("--chunk", type=int, default=128)
    ap.add_argument("--ref-clips", type=int, default=4, help="clips per step of the reference arm")
    ap.add_argument("--cpu-clips", type=int, default=16, help="timed clips of the cpu_baseline sample (0 = skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configs and the parity pass")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the scores and best offsets of the last timed step "
                                                           "to DIR/*.npy (native arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs --impl native")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    import avsync_b200 as A

    torch.cuda.set_device(local_rank)
    A._native.device_check()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    L = A._native.lib()

    # random-init weights of the reference architecture (PyTorch default initialisers, seeded); the
    # product package only — oracle/ is imported by the cpu_baseline leg alone
    torch.manual_seed(0)
    net = A.LipNet(39, precision=args.precision).to(dev).eval()
    torch.manual_seed(1)
    det = A.MisalignmentDetector(13864, 512).to(dev).eval()
    C = args.clips_per_gpu
    n_total = C * world
    sw = A.SyncSweeper(net, det, S_FRAMES, N_SAMPLES, chunk_clips=min(args.chunk, C))
    frames_h, audio_h = synth_inputs(C, seed=1000 + rank)         # u8 pixels + f32 audio, pinned
    frames_d, audio_d = frames_h.to(dev), audio_h.to(dev)

    def step_device():
        s, b = sw.run(frames_d, audio_d)
        return A.distributed.gather_scores(s, b, n_total)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput
    # nvidia-smi is started before the warm-up (it needs a few hundred ms to deliver its first sample); only samples
    # taken from the start of the timed region on are used
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(args.warmup):
        step_device()
    barrier()
    L.avs_prof_reset()
    L.avs_prof_enable(1)
    launches0 = L.avs_launch_count()
    first_sample = sampler.count() if sampler else 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        scores, best = step_device()
    ev1.record()
    barrier()
    L.avs_prof_enable(0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, scores.cpu().numpy(), best.cpu().numpy())
    # a timed region shorter than ~0.4 s may see fewer than three 100 ms samples: keep the GPU under the identical load
    # (untimed steps, all ranks) until three have been taken
    extra = torch.zeros(1, device=dev, dtype=torch.int32)
    t_extra = time.perf_counter()
    while True:
        extra[0] = 1 if (sampler is not None and sampler.count() - first_sample < 3 and time.perf_counter() - t_extra < 3.0) else 0
        if world > 1:
            dist.broadcast(extra, src=0)
        if int(extra.item()) == 0:
            break
        step_device()
        torch.cuda.synchronize()
    clocks = sampler.stop(first_sample) if sampler else None
    if clocks is not None:
        clocks["window"] = "samples every 100 ms from the start of the timed region; if it ends before three were taken, identical untimed steps keep the load up until they are"
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    launches = torch.tensor([L.avs_launch_count() - launches0], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(launches, op=dist.ReduceOp.SUM)
    ms_total = float(ms.item())
    value = n_total * args.steps / (ms_total / 1e3)

    # per-kernel times of rank 0 (CUDA events on the launching streams, inside the timed region)
    import ctypes
    prof = {}
    names = ["pack", "conv1", "conv2", "conv3", "vstats", "mfcc_logmel", "mfcc_stats", "score_gemm", "score"]
    for i, nme in enumerate(names):
        t, c = ctypes.c_double(), ctypes.c_int()
        L.avs_prof_read(i, ctypes.byref(t), ctypes.byref(c))
        prof[nme] = {"ms_total": t.value, "launches": c.value}

    # ---------------- the same step fed with the reference's f32 frames tensor (device-resident)
    f32_h = frames_f32(frames_h)
    f32_d = f32_h.to(dev)

    def step_device_f32():
        s, b = sw.run(f32_d, audio_d)
        return A.distributed.gather_scores(s, b, n_total)
    step_device_f32()
    barrier()
    ev0.record()
    for _ in range(max(2, args.steps // 2)):
        s32, b32 = step_device_f32()
    ev1.record()
    barrier()
    ms32 = torch.tensor([ev0.elapsed_time(ev1) / max(2, args.steps // 2)], device=dev)
    if world > 1:
        dist.all_reduce(ms32, op=dist.ReduceOp.MAX)
    value_f32 = n_total / (float(ms32.item()) / 1e3)
    f32_matches = bool(torch.equal(s32, scores) and torch.equal(b32, best))
    del f32_d

    # ---------------- end-to-end through the host-buffer entry points
    def time_host(fh, ah):
        def step_host():
            s, b = sw.run_host(fh, ah)
            if world > 1:
                return A.distributed.gather_scores(torch.from_numpy(s).to(dev), torch.from_numpy(b).to(dev), n_total)
            return s, b
        for _ in range(2):
            step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            s_h, b_h = step_host()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        same = np.array_equal(np.asarray(s_h if world == 1 else s_h.cpu().numpy()), scores.cpu().numpy())
        return n_total * args.steps / float(dt.item()), bool(same)

    e2e = e2e_f32 = None
    if not args.no_e2e:
        v, same = time_host(frames_h.numpy(), audio_h.numpy())
        e2e = {"value": v, "unit": "clips/s",
               "h2d_bytes_per_step": n_total * (FRAME_ELEMS * 1 + N_SAMPLES * 4),
               "d2h_bytes_per_step": n_total * (N_SHIFTS + 1) * 4, "frames": "uint8 pixels (avs_sweep_run_host_u8)",
               "timer": "host wall clock around the synchronous host-buffer call, barrier + cuda sync both sides, max over ranks",
               "matches_device_path": same}
        v, same = time_host(f32_h.numpy(), audio_h.numpy())
        e2e_f32 = {"value": v, "unit": "clips/s",
                   "h2d_bytes_per_step": n_total * (FRAME_ELEMS + N_SAMPLES) * 4,
                   "d2h_bytes_per_step": n_total * (N_SHIFTS + 1) * 4, "frames": "float32 tensor (avs_sweep_run_host)",
                   "matches_device_path": same}
        if world == 1:
            # the same call from ordinary (pageable) numpy arrays: every chunk is staged through the handle's pinned slots
            # by a host memcpy on the calling thread (csrc/sweep.cu, sweep_run_host: `direct == false`)
            fp, ap = np.array(frames_h.numpy(), copy=True), np.array(audio_h.numpy(), copy=True)
            v, same = time_host(fp, ap)
            e2e["pageable_host_buffers"] = {"value": v, "unit": "clips/s", "matches_device_path": same,
                                            "what": "uint8 frames + f32 audio in pageable memory, staged chunk by chunk"}
            del fp, ap
    del f32_h

    # ---------------- parity of the headline dtype on this batch, and the other BASELINE configs (outside the timed region)
    parity = None
    configs = {}
    if not args.no_configs:
        if rank == 0 and args.precision == "bf16":
            torch.manual_seed(0)
            net3 = A.LipNet(39, precision="bf16x3").to(dev).eval()
            sw3 = A.SyncSweeper(net3, det, S_FRAMES, N_SAMPLES, chunk_clips=min(args.chunk, C))
            s3, b3 = sw3.run(frames_d, audio_d)
            loc_s, loc_b = sw.run(frames_d, audio_d)
            parity = parity_stats(loc_s.cpu().numpy(), loc_b.cpu().numpy(), s3.cpu().numpy(), b3.cpu().numpy())
            parity["reference"] = "bf16x3 (fp32-grade) path of this library on the same clips; that path is pinned to the " \
                                  "reference's golden scores to 3.6e-7 in tests/test_gpu_parity.py"
            ms3 = cuda_time(lambda: sw3.run(frames_d, audio_d), 3, warm=1)
            configs["sweep_s20_bf16x3"] = {"value": C / (ms3 / 1e3), "unit": "clips/s", "ms_per_step": ms3,
                                           "what": f"the headline step ({C} clips, +-20) in fp32-grade arithmetic, 1 GPU"}
            del sw3, net3, s3, b3
        if world == 1:
            oc, nets = other_configs(A, dev, det, frames_h, audio_h, world)
            configs.update(oc)
            configs["dropin_per_shift_loop"] = dropin_loop(A, dev, det, nets["bf16x3"], frames_h, audio_h)
            del nets
        configs["config5_ddp_detector_step"], cfg5_ctx = ddp_config5(A, dev, world, rank)

    if rank == 0:
        pk, pk_src = peaks()
        conv2 = prof["conv2"]
        clips_per_launch = min(args.chunk, C)
        nl = max(conv2["launches"], 1)
        avg_ms = conv2["ms_total"] / nl
        mult = 3 if args.precision == "bf16x3" else 1
        achieved = (CONV_FLOP[2] * clips_per_launch / (avg_ms / 1e3) / 1e12) if avg_ms > 0 else 0.0
        tensor_peak = pk["bf16_tflops_sustained"]
        roof = {"kernel": "conv_l2_fused_kernel[layer 2: Conv3d 32->64, 3x5x5 + bias + ReLU + pool]" if args.precision != "fp32"
                else "conv_pool_ffma_kernel[layer 2]",
                "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                "frac": achieved / tensor_peak, "traffic": conv2_traffic(clips_per_launch, args.precision),
                "traffic_source": "constant from the committed ncu --set full capture (11.66 MB per clip) x clips per launch; "
                                  "not measured by this run",
                "peak_source": f"{pk_src} bf16_tflops_sustained (kernel timed inside a long step)",
                "algorithmic_flop_per_launch": CONV_FLOP[2] * clips_per_launch,
                "issued_mma_multiplier": mult, "avg_launch_ms": avg_ms, "launches_timed": conv2["launches"],
                "share_of_step": conv2["ms_total"] / ms_total if ms_total else None,
                # the sustained peak is a measured cuBLAS bf16 GEMM rate, not a hardware bound: a frac near (or a
                # little above) 1 says "as fast as cuBLAS keeps this GPU busy under its power cap"
                "frac_of_burst_peak": achieved / pk["bf16_tflops"] if pk.get("bf16_tflops") else None,
                "whole_step_tflops": sum(CONV_FLOP.values()) * n_total / world / (ms_total / args.steps / 1e3) / 1e12}
        cpu = None
        if args.cpu_clips > 0 and world == 1:
            cpu = cpu_baseline_subprocess(args.cpu_clips)
        line = {
            "metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": f"+-{S_FRAMES}-frame (41-offset) sync sweep, {C} clips per GPU per step "
                                   f"({n_total} clips/step), GRID-shaped 1x75x50x100 mouth crops as uint8 pixels "
                                   f"(the reference's f32 frames are float32(u8/255)) + 3 s 16 kHz f32 audio, "
                                   f"random-init LipNet STCNN + detector(hidden 512), chunks of {min(args.chunk, C)} clips",
                       "clips_per_gpu": C, "n_shifts": N_SHIFTS, "precision": args.precision,
                       "parallelism": f"clip-sharded x{world}, NCCL all_gather of [{n_total},41] scores" if world > 1 else "1 GPU",
                       "l2": f"inputs per step {C * (FRAME_ELEMS + N_SAMPLES * 4) / 1e6:.0f} MB per GPU and "
                             f"{C * 19.3:.0f} MB of inter-layer activations > 126 MB L2 (no flush needed)"},
            "e2e": e2e, "e2e_f32_frames": e2e_f32,
            "value_f32_frames": {"value": value_f32, "unit": "clips/s", "scores_identical_to_u8_path": f32_matches,
                                 "what": "device-resident step fed with the reference's f32 frames tensor"},
            "gpu_launches": int(launches.item()), "clocks": clocks, "roofline": roof, "parity": parity,
            "configs": configs, "cpu_baseline": cpu, "kernel_ms": prof,
        }
    else:
        line = None
    # Last leg, after every number of the line exists: config 5 as one CUDA graph (NCCL all-reduce captured when N > 1).
    # A capture that wedged would cost the whole line, so a timer prints the line without this leg and ends the process.
    if not args.no_configs and os.environ.get("AVS_BENCH_NO_GRAPH") != "1":
        import threading

        def give_up():
            if line is not None:
                line["configs"]["config5_ddp_detector_step"]["cuda_graph"] = {"unavailable": "timed out after 120 s"}
                print(json.dumps(line), file=_REAL_STDOUT, flush=True)
            os._exit(0)
        timer = threading.Timer(120.0, give_up)
        timer.daemon = True
        timer.start()
        g5 = ddp_config5_graph(A, dev, world, rank, cfg5_ctx)
        timer.cancel()
        if line is not None:
            line["configs"]["config5_ddp_detector_step"]["cuda_graph"] = g5
    if line is not None:
        print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def _json_only_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner at communicator
    creation): point fd 1 at stderr for the life of the process and keep the real stdout for the JSON line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


if __name__ == "__main__":
    _REAL_STDOUT = _json_only_stdout()
    main()
