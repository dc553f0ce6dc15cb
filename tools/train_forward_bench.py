"""Time the training-mode U-Net forward (network([x_t, t, ctx], training=True): batch-statistics BatchNorm, per-sample t)
against the inference forward at cfg-2 (conditional U-Net, B=8, 32^3 x 256) with CUDA events, alternating the two programs.

    python tools/train_forward_bench.py [--batch 8] [--iters 50] [--warmup 5]

Prints the card name and power limit beside the numbers.  Writes nothing.
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    import torch
    import b200dm
    from b200dm import _lib as L
    L.require_gpu()
    B, S, C, T = a.batch, 32, 256, 1000
    net = b200dm.build_model(S, C, [64, 128, 256], [False, False, True, True], context_dim=1)
    net.compile(B, T, per_sample_t=True)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(B, S, S, S, C, generator=g).cuda()
    t = torch.randint(0, T, (B,), generator=g)
    ctx = torch.arange(B) % 2
    net([x, t, ctx])
    net([x, t, ctx], training=True)
    tr = net.training_program()
    progs = {"inference": net.prog, "training": tr.prog}
    times = {k: [] for k in progs}
    for k, p in progs.items():
        for _ in range(a.warmup):
            p.run()
    torch.cuda.synchronize()
    for _ in range(a.iters):
        for k, p in progs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            p.run()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    assert L.debug_flag() == 0
    print(f"card: {card()}")
    print(f"cfg-2 U-Net forward, B={B}, {S}^3 x {C}, per-sample t, {a.iters} alternating runs (device events, eager program):")
    for k in progs:
        ts = sorted(times[k])
        print(f"  {k:9s} median {statistics.median(ts):.3f} ms  min {ts[0]:.3f}  max {ts[-1]:.3f}  launches {progs[k].num_launches}")
    print(f"  training / inference: {statistics.median(times['training']) / statistics.median(times['inference']):.3f}")


if __name__ == "__main__":
    main()
