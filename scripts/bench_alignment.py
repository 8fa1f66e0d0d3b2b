#!/usr/bin/env python
"""error_alignment against error_counts on the same inputs.

    python scripts/bench_alignment.py [--steps 50] [--warmup 10] [--out FILE]

Shapes as scripts/bench_counts.py: cfg4 (1 M word pairs, T = 31: the short form), cfg1 (65 536
character pairs, T = 51: the short form; the inputs fit in L2, so 8 batches rotate) and cfg3's
8 192 x 200 (the long form: K0, K1 with the trace, the walk).  Per shape error_alignment and
error_counts, both with (3, 3, 4) costs, alternate call by call, timed with CUDA events after a
warm-up.  At full size the op histogram of every pair is checked against error_counts on the
device.  Prints one JSON line with the GPU name and power limit.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "pydrobert-pytorch_b200"), os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

import b200lev.functional as F  # noqa: E402
from bench_counts import NIST, gpu_info, shape  # noqa: E402


def histogram_matches(ref, hyp, kw):
    ops = F.error_alignment(ref, hyp, warn=False, **kw, **NIST)
    cnt = F.error_counts(ref, hyp, warn=False, **kw, **NIST)
    hist = torch.stack([(ops == k).sum(0) for k in range(4)], 1)
    return bool(torch.equal(hist, cnt))


def time_calls(batches, kw, steps, warmup):
    calls = {
        "error_alignment_nist": lambda r, h: F.error_alignment(r, h, warn=False, **kw, **NIST),
        "error_counts_nist": lambda r, h: F.error_counts(r, h, warn=False, **kw, **NIST),
    }
    ms = {k: [] for k in calls}
    for it in range(warmup + steps):
        for name, fn in calls.items():  # alternate the calls
            r, h = batches[it % len(batches)]
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(r, h)
            b.record()
            b.synchronize()
            if it >= warmup:
                ms[name].append(a.elapsed_time(b))
    return {k: float(np.median(v)) for k, v in ms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_alignment.py needs a CUDA device"
    res = gpu_info()
    res["shapes"] = {}
    for name, cfg, pairs, rotate in (("cfg4", 4, 1_000_000, 1), ("cfg1", 1, 65536, 8), ("long_8192x200", 3, 8192, 1)):
        batches, kw = shape(cfg, pairs, rotate)
        t = time_calls(batches, kw, args.steps, args.warmup)
        R, H = batches[0][0].shape[0], batches[0][1].shape[0]
        row = {"pairs": pairs, "R": R, "H": H, "rotate": rotate, "ms_per_call": t,
               "ratio": t["error_alignment_nist"] / t["error_counts_nist"],
               "ops_bytes": (R + H) * pairs, "histogram_equals_counts": histogram_matches(*batches[0], kw)}
        res["shapes"][name] = row
        del batches
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
