#!/usr/bin/env python
"""DinoLoss at wide prototype heads (8192 < K <= 65536: the cluster kernels of csrc/next_rows.cu), one GPU.

    python tools/bench_dino_wide.py [--reps 20] [--timeline]   -> a markdown report on stdout

For each shape: forward + backward through the public `DinoLoss`, timed with CUDA events over CUDA-graph replays with
the L2 flushed between repetitions (bench_losses.time_graph / l2_flush); algorithmic bytes (2 (2 + nv) + nv) bs K 4 as
in bench_losses' DINO rows (the forward reads teacher + student, the backward reads them again and writes the
gradient) and their fraction of the measured copy rate; the same loss written as eager torch fp32 ops, timed the same
way on the same GPU, and the parity of the two.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "self-supervised-vision_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import bench_losses as B  # noqa: E402

SHAPES = [(64, 12, 65536), (256, 12, 65536), (1024, 10, 16384)]   # (bs, nv, K): DINO's head, a larger batch, C = 2
TEMP_S, TEMP_T = 0.1, 0.04
COPY_GBS = 6547.8   # BASELINE.md: b.copy_(a) of 1 Gi bf16 on a B200, read + write bytes


def copy_rate():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json"
    return COPY_GBS, "BASELINE.md"


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info = q.stdout.strip() if q.returncode == 0 else f"nvidia-smi rc={q.returncode}"
    except (OSError, subprocess.SubprocessError) as e:
        info = f"nvidia-smi unavailable ({type(e).__name__})"
    return name, info


def torch_dino(teacher, student, temp_s, temp_t, center):
    """utils/losses.py:80-89 as eager fp32 torch ops: both teacher views' softmax summed, one log_softmax per student row."""
    tsum = torch.softmax((teacher - center) / temp_t, dim=-1).sum(1, keepdim=True)
    logp = torch.log_softmax(student / temp_s, dim=-1)
    return -(tsum * logp).sum(-1).mean()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--timeline", action="store_true", help="also print the kernel timeline of one graph replay per shape")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a B200"
    torch.cuda.set_device(0)
    import ssv_b200 as S
    dev = torch.device("cuda", 0)
    name, info = card()
    gbs, gbs_src = copy_rate()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    print(f"# DinoLoss, wide heads (cluster kernels): forward + backward on one GPU\n")
    print(f"GPU: {name}; power.limit, clocks.max.sm: {info}")
    print(f"Copy rate: {gbs:.1f} GB/s ({gbs_src}).  Times: median of {args.reps} CUDA-graph replays, L2 flushed before each "
          f"(256 MiB write + 256 MiB read).  temp_s {TEMP_S}, temp_t {TEMP_T}.\n")
    print("| bs x nv x K | cluster | bytes | ours ms | ours TB/s | of copy rate | torch fp32 ms | torch / ours | "
          "loss rel | grad rel-L2 |")
    print("|---|---|---|---|---|---|---|---|---|---|")
    timelines = []
    for bs, nv, k in SHAPES:
        g = torch.Generator().manual_seed(bs + k)
        t = torch.randn(bs, 2, k, generator=g).to(dev)
        c = (0.2 * torch.randn(k, generator=g)).to(dev)
        s_ours = torch.randn(bs, nv, k, generator=g).to(dev).requires_grad_(True)
        s_ref = s_ours.detach().clone().requires_grad_(True)
        fn = S.DinoLoss()
        ours = B.fwd_bwd(lambda: fn(t, s_ours, TEMP_S, TEMP_T, c), s_ours)
        ref = B.fwd_bwd(lambda: torch_dino(t, s_ref, TEMP_S, TEMP_T, c), s_ref)
        ms = B.time_graph(ours, args.reps, flush)
        if ms is None:
            raise RuntimeError("CUDA-graph capture of DinoLoss failed")
        ref_ms = B.time_graph(ref, max(5, args.reps // 2), flush)
        # parity on one fresh eager step of each
        ours()
        ref()
        l_ours = fn(t, s_ours.detach(), TEMP_S, TEMP_T, c).item()
        l_ref = torch_dino(t, s_ref.detach(), TEMP_S, TEMP_T, c).item()
        lrel = abs(l_ours - l_ref) / abs(l_ref)
        grel = ((s_ours.grad.double() - s_ref.grad.double()).norm() / s_ref.grad.double().norm()).item()
        nbytes = (2 * (2 + nv) + nv) * bs * k * 4
        tbs = nbytes / (ms * 1e-3) / 1e12
        ref_s = f"{ref_ms:.3f}" if ref_ms else "capture failed"
        ratio = f"{ref_ms / ms:.1f}x" if ref_ms else "-"
        print(f"| {bs} x {nv} x {k} | {-(-k // 8192)} CTAs | {nbytes / 1e6:.0f} MB | {ms:.4f} | {tbs:.2f} | "
              f"{tbs * 1e3 / gbs:.2f} | {ref_s} | {ratio} | {lrel:.1e} | {grel:.1e} |", flush=True)
        if args.timeline:
            import io
            buf = io.StringIO()
            B.graph_timeline(ours, flush, f"{bs} x {nv} x {k}, ours", buf)
            timelines.append(buf.getvalue())
        del t, c, s_ours, s_ref
        torch.cuda.empty_cache()
    print("\n(bytes: (2 (2 + nv) + nv) bs K 4 - the forward reads teacher + student, the backward reads them again and "
          "writes the gradient; parity: ours against the eager torch fp32 loss on the same inputs)")
    if timelines:
        print("\n## Kernel timeline of one graph replay (torch.profiler)\n\n```")
        for tl in timelines:
            print(tl, end="")
        print("```")


if __name__ == "__main__":
    main()
