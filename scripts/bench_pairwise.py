#!/usr/bin/env python
"""pairwise_error_rates and minimum_bayes_risk against what a user does without them.

    python scripts/bench_pairwise.py [--steps 50] [--warmup 10] [--out FILE]

Baseline: the cross product materialised with index_select (the hypotheses of every pair, the
references not repeated), then the body of error_rate with ref_group = B -- the private n-best form
(functional._string_matching) that minimum_error_rate_loss uses.  Through the public error_rate a
user would have to materialise the references too, so this baseline is at least as fast as what a
user can call.  Shapes (every group's hypotheses are word-level edits of one
another, vocabulary 10 000, eos -1):

  (a) MBR on word n-best lists: G = 4 096 groups of M = 16, T = 31, unit costs -- 1 M pairs, the
      short cross form; also timed on a batch-stride-2 view of the same tokens, which takes the
      gather path (gather, then the plain short-reference kernel);
  (b) G = 16 384, M = 8, T = 100 (cfg2's token shape), unit costs -- 1 M pairs, gather + the fused
      bit-vector kernel;
  (c) shape (a) with costs (3, 3, 4) -- gather + the wavefront kernels;
  (d) minimum_bayes_risk on (a) against the torch composition: materialise, error_rate, softmax,
      einsum, argmin.

Each call alternates with its baseline call by call, timed with CUDA events after a warm-up;
median, 10th and 90th percentile ms.  The inputs of (a), (c) and (d) (16 MB of tokens) stay in L2,
as a decoder's n-best lists would; the baseline's materialised pairs (268 MB) do not.  Outputs are
compared with the baseline at full size in the same run.  Prints one JSON line with the device
name and its power limit.
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

SHAPES = {"a": (4096, 16, 31, (1.0, 1.0, 1.0)), "b": (16384, 8, 100, (1.0, 1.0, 1.0)),
          "c": (4096, 16, 31, (3.0, 3.0, 4.0))}


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def nbest_words(G, M, T, V=10_000, seed=0):
    """(T, G, M) int64: per group one random word sequence, each hypothesis replacing 15 % of its
    words, lengths T // 3 .. T - 1, then eos -1."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, V, (T, G, 1))
    hyp = np.where(rng.random((T, G, M)) < 0.15, rng.integers(0, V, (T, G, M)), base)
    lens = rng.integers(T // 3, T, (G, M))
    return np.where(np.arange(T)[:, None, None] < lens, hyp, -1)


def materialised(h, costs, norm=True):
    """What a user does today: (T, G*M*M) hypotheses by index_select, then error_rate in the n-best
    form (reference column pair // M)."""
    T, G, M = h.shape
    flat = h.reshape(T, G * M)
    idx = torch.arange(G * M * M, device=h.device)
    hx = flat.index_select(1, idx // (M * M) * M + idx % M)
    return F._string_matching(flat, hx, -1, False, False, costs[0], costs[1], costs[2], False, norm, False,
                              False, 0, True, M)


def mbr_composition(lp, h):
    T, G, M = h.shape
    er = materialised(h, (1.0, 1.0, 1.0)).view(G, M, M)
    risk = torch.einsum("na,nai->ni", lp.softmax(1), er)
    return risk.argmin(1), risk


def time_pair(calls, steps, warmup):
    ms = {k: [] for k in calls}
    for it in range(warmup + steps):
        for name, fn in calls.items():  # alternate the calls
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            if it >= warmup:
                ms[name].append(a.elapsed_time(b))
    return {k: {"median": float(np.median(v)), "p10": float(np.percentile(v, 10)),
                "p90": float(np.percentile(v, 90))} for k, v in ms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_pairwise.py needs a CUDA device"
    res = gpu_info()
    res["shapes"] = {}
    for name, (G, M, T, costs) in SHAPES.items():
        h = torch.from_numpy(nbest_words(G, M, T)).cuda()
        kw = dict(eos=-1, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2], warn=False)
        calls = {"pairwise_error_rates": lambda: F.pairwise_error_rates(h, h, **kw),
                 "materialised_error_rate": lambda: materialised(h, costs)}
        if name == "a":
            # the same tokens as a view with batch stride 2: b200lev_final_cross takes the gather
            # path (then the plain short-reference kernel) -- the short cross form against the
            # gather path on one shape
            hs = torch.empty((T, G, 2 * M), dtype=h.dtype, device=h.device)[:, :, ::2]
            hs.copy_(h)
            calls["pairwise_error_rates_gather_path"] = lambda: F.pairwise_error_rates(hs, hs, **kw)
        t = time_pair(calls, args.steps, args.warmup)
        pairs = G * M * M
        row = {"G": G, "M": M, "T": T, "costs": costs, "pairs": pairs, "ms_per_call": t,
               "pairs_per_s": {k: pairs / (v["median"] * 1e-3) for k, v in t.items()},
               "speedup": t["materialised_error_rate"]["median"] / t["pairwise_error_rates"]["median"],
               "equal": bool(torch.equal(F.pairwise_error_rates(h, h, **kw).reshape(-1), materialised(h, costs)))}
        if name == "a":
            row["gather_path_equal"] = bool(torch.equal(F.pairwise_error_rates(hs, hs, **kw),
                                                        F.pairwise_error_rates(h, h, **kw)))
            del hs
        res["shapes"][name] = row
        del h
        torch.cuda.empty_cache()
    G, M, T, _ = SHAPES["a"]
    h = torch.from_numpy(nbest_words(G, M, T, seed=1)).cuda()
    lp = torch.randn(G, M, device="cuda").log_softmax(1)
    t = time_pair({"minimum_bayes_risk": lambda: F.minimum_bayes_risk(lp, h, eos=-1, include_eos=False, warn=False),
                   "torch_composition": lambda: mbr_composition(lp, h)}, args.steps, args.warmup)
    best, risk = F.minimum_bayes_risk(lp, h, eos=-1, include_eos=False, warn=False)
    cbest, crisk = mbr_composition(lp, h)
    srt = crisk.sort(1).values
    clear = srt[:, 1] - srt[:, 0] > 1e-5
    res["shapes"]["d"] = {
        "G": G, "M": M, "T": T, "pairs": G * M * M, "ms_per_call": t,
        "speedup": t["torch_composition"]["median"] / t["minimum_bayes_risk"]["median"],
        "risk_max_abs_diff": float((risk - crisk).abs().max()),
        "best_equal_fraction": float((best == cbest).float().mean()),
        "best_equal_where_gap_over_1e-5": bool(torch.equal(best[clear], cbest[clear])),
        "groups_with_gap_over_1e-5": int(clear.sum())}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
