#!/usr/bin/env python
"""infix_edit_distance / infix_matches against the composition available without them.

    python scripts/bench_infix.py [--steps 20] [--warmup 3] [--out FILE]

The baseline is the only route to an infix distance the library had before: the minimum over
start offsets s of prefix_edit_distances(ref, hyp[s:]) -- H + 1 calls and about H / 2 times the
cells.  Shapes, on both sides of the route choice of the distance-only call:
  (a) 65 536 pairs, references of 2-16 tokens (ragged), hypotheses of 128, unit costs:
      infix_edit_distance on the short bit-vector kernel's infix kind;
  (b) (a) through infix_matches: the wavefront kernel with the start channel;
  (c) (a) with costs (3, 3, 4): the wavefront kernel;
  (d) 1 024 pairs, R = 300, H = 2 000, unit costs: the wavefront kernel over several strips; the
      new call alone (the baseline would take 2 001 calls), reported in GCUPS (P * R * H cells).
On (a)-(c) the new call and the baseline alternate call by call (CUDA events after a warm-up) and
the new call's distance is checked against the baseline's.  Prints one JSON line.
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

EOS = -1
SHAPES = {  # pairs, reference lengths (lo, hi), hypothesis length, costs, call
    "a": (65536, (2, 16), 128, (1.0, 1.0, 1.0), "distance"),
    "b": (65536, (2, 16), 128, (1.0, 1.0, 1.0), "matches"),
    "c": (65536, (2, 16), 128, (3.0, 3.0, 4.0), "distance"),
    "d": (1024, (300, 300), 2000, (1.0, 1.0, 1.0), "distance"),
}


def make(shape, dev, seed=0):
    """(ref, hyp, costs, eos): sequence-first int64 tensors on `dev`.  References are ragged
    (padded with eos); hypotheses hold no eos, so h = H, and a noisy copy of the reference is planted
    in every other one."""
    P, (lo, hi), H, costs, _ = SHAPES[shape]
    rng = np.random.default_rng(seed)
    V = 50
    ref = np.full((hi, P), EOS, np.int64)
    lens = rng.integers(lo, hi + 1, P)
    body = rng.integers(0, V, (hi, P))
    ref[np.arange(hi)[:, None] < lens[None]] = body[np.arange(hi)[:, None] < lens[None]]
    hyp = rng.integers(0, V, (H, P))
    at = rng.integers(0, H - hi, P)
    for n in range(0, P, 2):
        seg = ref[:lens[n], n].copy()
        noise = rng.random(lens[n]) < 0.15
        seg[noise] = rng.integers(0, V, int(noise.sum()))
        hyp[at[n]:at[n] + lens[n], n] = seg
    return torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev), costs, EOS


def shifted_prefix(ref, hyp, costs, eos):
    """min over s of prefix_edit_distances(ref, hyp[s:]), s = 0 .. H (the last: the empty suffix)."""
    c = dict(ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
    best = None
    for s in range(hyp.shape[0] + 1):
        p = F.prefix_edit_distances(ref, hyp[s:], eos=eos, include_eos=False, warn=False, **c)
        m = p.min(0).values
        best = m if best is None else torch.minimum(best, m)
    return best


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def _stats(ms):
    a = np.asarray(ms)
    return {"median_ms": float(np.median(a)), "p10_ms": float(np.percentile(a, 10)),
            "p90_ms": float(np.percentile(a, 90))}


def _time(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def run_shape(name, steps, warmup):
    dev = torch.device("cuda")
    ref, hyp, costs, eos = make(name, dev)
    P, _, H, _, call = SHAPES[name]
    c = dict(eos=eos, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2], warn=False)
    if call == "distance":
        new = lambda: F.infix_edit_distance(ref, hyp, **c)  # noqa: E731
    else:
        new = lambda: F.infix_matches(ref, hyp, **c)[0]  # noqa: E731
    out = {"shape": name, "pairs": P, "R": ref.shape[0], "H": H, "costs": list(costs), "call": call}
    dist = new()
    if name == "d":
        for _ in range(warmup):
            new()
        ms = [_time(new) for _ in range(steps)]
        out["new"] = _stats(ms)
        cells = float(P) * ref.shape[0] * H
        out["gcups"] = cells / (out["new"]["median_ms"] * 1e-3) / 1e9
        return out
    base = lambda: shifted_prefix(ref, hyp, costs, eos)  # noqa: E731
    out["dist_equal"] = bool(torch.equal(dist, base()))
    for _ in range(warmup):
        new()
        base()
    ms_new, ms_base = [], []
    for _ in range(steps):
        ms_new.append(_time(new))
        ms_base.append(_time(base))
    out["new"] = _stats(ms_new)
    out["baseline_shifted_prefix"] = _stats(ms_base)
    out["speedup"] = out["baseline_shifted_prefix"]["median_ms"] / out["new"]["median_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="abcd")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_infix.py measures the B200 kernels: no CUDA device")
    res = {"bench": "infix", **gpu_info(), "steps": a.steps,
           "shapes": [run_shape(s, a.steps, a.warmup) for s in a.shapes]}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
