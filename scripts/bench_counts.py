#!/usr/bin/env python
"""error_counts against error_rate(norm=False) on the same inputs.

    python scripts/bench_counts.py [--steps 50] [--warmup 10] [--out FILE]

Shapes: cfg4 (1 M word pairs, T = 31: the short form), cfg1 (65 536 character pairs, T = 51:
the short form, two-word rows; the inputs fit in L2, so several batches rotate) and cfg3's
8 192 x 200 (the long form: K0 + K1).  Per shape the three calls -- error_counts with (3, 3, 4)
costs, error_rate(norm=False) with unit costs and with (3, 3, 4) -- alternate call by call,
timed with CUDA events after a warm-up.  At full size every identity is checked on the device:
C + S + D = r, C + S + I = h, S + D + I = error_rate(norm=False), 3 I + 3 D + 4 S =
edit_distance(norm=False).  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "pydrobert-pytorch_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import b200lev.functional as F  # noqa: E402
from bench import Workload  # noqa: E402

NIST = dict(ins_cost=3.0, del_cost=3.0, sub_cost=4.0)


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def shape(cfg, pairs, rotate, seed=0):
    w = Workload(cfg)
    batches = []
    for k in range(rotate):
        ref, hyp, _ = w.make(pairs, seed + k)
        batches.append((torch.from_numpy(ref).cuda(), torch.from_numpy(hyp).cuda()))
    kw = dict(eos=w.eos, include_eos=w.include_eos)
    return batches, kw


def identities(ref, hyp, kw):
    cnt = F.error_counts(ref, hyp, warn=False, **kw, **NIST)
    C, S, D, I = cnt.unbind(1)
    out = {}
    for name, costs in (("unit", dict(ins_cost=1.0, del_cost=1.0, sub_cost=1.0)), ("nist", NIST)):
        c = F.error_counts(ref, hyp, warn=False, **kw, **costs)
        Cc, Sc, Dc, Ic = c.unbind(1)
        er = F.error_rate(ref, hyp, norm=False, warn=False, **kw, **costs)
        ed = F.edit_distance(ref, hyp, norm=False, warn=False, **kw, **costs)
        lin = costs["ins_cost"] * Ic + costs["del_cost"] * Dc + costs["sub_cost"] * Sc
        out[name] = bool(torch.equal((Sc + Dc + Ic).float(), er)) and bool(torch.equal(lin.float(), ed))
    # lengths from the eos of the call (these workloads always hold one)
    inc = 1 if kw["include_eos"] else 0
    rl = (ref == kw["eos"]).int().argmax(0).long() + inc
    hl = (hyp == kw["eos"]).int().argmax(0).long() + inc
    out["lengths"] = bool(torch.equal(C + S + D, rl)) and bool(torch.equal(C + S + I, hl))
    return out


def time_calls(batches, kw, steps, warmup):
    calls = {
        "error_counts_nist": lambda r, h: F.error_counts(r, h, warn=False, **kw, **NIST),
        "error_rate_unit": lambda r, h: F.error_rate(r, h, norm=False, warn=False, **kw),
        "error_rate_nist": lambda r, h: F.error_rate(r, h, norm=False, warn=False, **kw, **NIST),
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
    assert torch.cuda.is_available(), "bench_counts.py needs a CUDA device"
    res = gpu_info()
    res["shapes"] = {}
    for name, cfg, pairs, rotate in (("cfg4", 4, 1_000_000, 1), ("cfg1", 1, 65536, 8), ("long_8192x200", 3, 8192, 1)):
        batches, kw = shape(cfg, pairs, rotate)
        t = time_calls(batches, kw, args.steps, args.warmup)
        row = {"pairs": pairs, "T": batches[0][0].shape[0], "rotate": rotate,
               "ms_per_call": t, "pairs_per_s": {k: pairs / (v * 1e-3) for k, v in t.items()},
               "identities": identities(*batches[0], kw)}
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
