"""One fine-tuning step of LipNet's Bi-GRU head on one GPU (B = 64 clips, T = 75, H = 256, in = 6912, V = 39, GRID
sentence targets, device-resident embeddings), each part timed on its own with CUDA events: the training forward
(LipNet.gru_head_train), the CTC loss with its gradient (ctc_loss forward + backward, K5e) and the head's backward
(K3b).  The backward's kernel times by name come from torch.profiler in a separate pass, next to the FLOPs of its
GEMMs computed from the shapes.  For context only: the same step with torch's nn.GRU, Linear and F.ctc_loss in fp32 on
the same GPU.  Reads the card's name and power limit in the same call.

    python tools/head_train_bench.py [--reps 20] [--precision bf16x3] [--out profiles/r09_head_train_bench.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import avsync_b200 as A  # noqa: E402
from oracle import ctc_align_ref, lipnet_ref  # noqa: E402
from oracle import ctc_loss_ref as R  # noqa: E402
from tools.ctc_beam_bench import time_ms  # noqa: E402
from tools.ragged_bench import card  # noqa: E402

B, T, H, IN, V = 64, 75, 256, 6912, 39


def backward_gemm_gflop():
    """FLOPs of the backward's sgemm_nt calls, from the shapes (2 * M * N * K, K = B * T rows)."""
    rows = B * T
    g = {"dW_ih layer 1": 2 * 6 * H * IN * rows, "dW_ih layer 2": 2 * 6 * H * 2 * H * rows,
         "dW_hh (2 layers x 2 directions)": 4 * 2 * 3 * H * H * rows, "dx layer 2": 2 * rows * 2 * H * 6 * H,
         "fc (dW_fc, dh2)": 2 * (2 * V * 2 * H * rows)}
    return {k: round(v / 1e9, 2) for k, v in g.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--precision", default="bf16x3")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    A._native.device_check()
    torch.cuda.set_device(0)
    c2i = A.dataset.create_vocab()[0]
    sd = lipnet_ref.init_lipnet_state(V, H, seed=0)
    net = A.LipNet(V, hidden_dim=H, precision=args.precision)
    net.load_state_dict(sd)
    net = net.cuda()
    gen = torch.Generator(device="cuda").manual_seed(0)
    emb = torch.randn((B, T, IN), device="cuda", generator=gen) * 0.05
    _, targets, lens = ctc_align_ref.grid_targets(B, c2i, seed=0)
    targets, lens = torch.from_numpy(targets).cuda(), torch.from_numpy(lens).cuda()
    il = torch.full((B,), T, dtype=torch.int32, device="cuda")
    head = [q for n, q in net.named_parameters() if n.startswith(("gru", "fc"))]
    res = {"card": card(), "shape": {"B": B, "T": T, "H": H, "in": IN, "V": V}, "precision": args.precision,
           "reps": args.reps}

    for p in (0.0, 0.5):
        lp = net.gru_head_train(emb, dropout=p)
        fwd = time_ms(lambda: net.gru_head_train(emb, dropout=p), args.reps)
        lpd = lp.detach().requires_grad_()

        def ctc():
            A.ctc_loss(lpd, targets, il, lens, zero_infinity=True).backward()
        ctc_ms = time_ms(ctc, args.reps)
        ctc()
        g = lpd.grad.detach().clone()

        def bwd():
            lp.backward(g, retain_graph=True)
        bwd_ms = time_ms(bwd, args.reps)

        def step():
            A.ctc_loss(net.gru_head_train(emb, dropout=p), targets, il, lens, zero_infinity=True).backward()
        step_ms = time_ms(step, args.reps)
        res[f"dropout_{p}"] = {"forward_ms": round(fwd, 3), "ctc_loss_fwd_bwd_ms": round(ctc_ms, 3),
                               "backward_ms": round(bwd_ms, 3), "whole_step_ms": round(step_ms, 3)}

    # backward kernels by name (torch.profiler, a separate pass)
    lp = net.gru_head_train(emb)
    g = torch.randn_like(lp) * 1e-3
    lp.backward(g, retain_graph=True)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            lp.backward(g, retain_graph=True)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA and e.count:
            name = e.key.split("(")[0].split("<")[0].replace("void ", "").split("::")[-1]
            t = getattr(e, "device_time_total", None) or e.cuda_time_total
            kern[name] = kern.get(name, 0.0) + t / 5 / 1000.0
    total = sum(kern.values())
    res["backward_kernels_ms_per_step"] = {k: round(v, 3) for k, v in sorted(kern.items(), key=lambda kv: -kv[1])}
    res["backward_kernel_total_ms"] = round(total, 3)
    res["backward_gemm_gflop"] = gemm = backward_gemm_gflop()
    sg = kern.get("sgemm_nt_kernel", 0.0)
    res["sgemm_nt_share_of_backward_kernel_time"] = round(sg / total, 3) if total else None
    res["sgemm_nt_rate_tflops"] = round(sum(gemm.values()) / 1e3 / (sg / 1e3), 2) if sg else None

    # the same step in torch, fp32, for context
    _, (g1, g2, fc) = R.head_reference(sd, emb, dtype=torch.float32)
    tparams = list(g1.parameters()) + list(g2.parameters()) + list(fc.parameters())

    def torch_step():
        x, _ = g1(emb)
        x, _ = g2(x)
        lp = torch.log_softmax(fc(x), -1)
        F.ctc_loss(lp.transpose(0, 1), targets.long(), il.long(), lens.long(), zero_infinity=True).backward()
    res["torch_fp32_step_ms"] = round(time_ms(torch_step, args.reps), 3)
    res["torch_cudnn_enabled"] = torch.backends.cudnn.enabled
    del tparams
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
