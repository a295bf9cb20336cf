#!/usr/bin/env python
"""Gradient / loss error of BarlowLoss against the fp64 oracle for the shipped code path.  Prints one line per shape.
The fused-vs-unfused backward error comparison of DESIGN §4.2 needs the A/B switches that commit 3683d33 still has:
run this script at that commit to reproduce it."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "self-supervised-vision_b200")]
import ssv_b200 as S  # noqa: E402
from oracle import ssl_oracle as O  # noqa: E402


def inputs(n, d, corr=0.7):
    g = torch.Generator().manual_seed(7)
    sig = (torch.rand(d, generator=g) * 1.5 + 0.5).numpy()
    mu = torch.randn(d, generator=g).numpy()
    zi = torch.randn(n, d, generator=torch.Generator().manual_seed(0)).numpy() * sig + mu
    zj = corr * zi + (1 - corr) * (torch.randn(n, d, generator=torch.Generator().manual_seed(1)).numpy() * sig + mu)
    return zi.astype(np.float32), zj.astype(np.float32)


def rl2(x, y):
    return float(np.linalg.norm(x - y) / np.linalg.norm(y))


for n, d in ((512, 4096), (256, 1000), (200, 264)):
    zi, zj = inputs(n, d)
    a = torch.from_numpy(zi).cuda().requires_grad_(True)
    b = torch.from_numpy(zj).cuda().requires_grad_(True)
    loss = S.BarlowLoss(False, 0.005)(a, b)
    loss.backward()
    ref = O.barlow(zi, zj, False, 0.005)
    print(f"barlow n={n} d={d}: loss rel {abs(loss.item() - ref[0]) / abs(ref[0]):.2e}  "
          f"dzi rel-L2 {rl2(a.grad.cpu().numpy(), ref[1]):.2e}  dzj rel-L2 {rl2(b.grad.cpu().numpy(), ref[2]):.2e}")
