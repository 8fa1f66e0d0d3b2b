#!/usr/bin/env python
"""minimum_error_rate_loss forward + backward on the cfg2 shapes (64 and 16 384 utterances x 8
samples, T = 100): ms per call.  The call declares its references shared, so the fused
bit-vector kernel takes it without a probe."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "pydrobert-pytorch_b200")):
    sys.path.insert(0, p)
import torch

import b200lev.functional as F
import bench

dev = torch.device("cuda", 0)
wl = bench.Workload(2)
for utts in (64, 16384):
    r, h, cells = wl.make(utts * 8, 1)
    ref = torch.from_numpy(r[:, ::8].copy()).to(dev)
    hyp = torch.from_numpy(h).to(dev).view(h.shape[0], utts, 8)
    lp = torch.randn(utts, 8, device=dev, requires_grad=True)

    def f():
        loss = F.minimum_error_rate_loss(lp, ref, hyp, eos=0, warn=False)
        loss.backward()

    for _ in range(5):
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        f()
    e1.record()
    torch.cuda.synchronize()
    print(f"{utts} utterances x 8 samples: {e0.elapsed_time(e1) / 50:.4f} ms per forward + backward")
