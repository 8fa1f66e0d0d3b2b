#!/usr/bin/env python
"""Small driver for compute-sanitizer: one call through every kernel family at shapes that
finish in seconds under memcheck / racecheck / synccheck (scripts/gpu_sanitize.sh).
Each result is also checked against the oracle, so a tool run doubles as a parity run."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "pydrobert-pytorch_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np
import torch

import b200lev.functional as F
import b200lev.scoring as S
from oracle import oracle as O

dev = torch.device("cuda", 0)
rng = np.random.default_rng(0)


def toks(T, N, V, eos=0):
    a = rng.integers(1, V, (T, N))
    a[rng.integers(T // 3, T, N), np.arange(N)] = eos
    return a


def same(act, exp, what):
    assert np.array_equal(act.cpu().numpy(), np.asarray(exp)), what
    print("ok", what, flush=True)


def run(env, fn):
    saved = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        fn()
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def prefix_case(R, H, N, V, what, **kw):
    r, h = toks(R, N, V), toks(H, N, V)
    tr, th = torch.from_numpy(r).to(dev), torch.from_numpy(h).to(dev)
    same(F.prefix_error_rates(tr, th, eos=0, warn=False, **kw), O.prefix_error_rates(r, h, eos=0, **kw), what)
    same(F.error_rate(tr, th, eos=0, warn=False), O.error_rate(r, h, eos=0), what + " (final)")


def nbest_case(what):
    r, h = toks(60, 16, 50), toks(70, 128, 50)
    rx = np.repeat(r, 8, axis=1)
    same(F.prefix_error_rates(torch.from_numpy(rx).to(dev), torch.from_numpy(h).to(dev), eos=0, warn=False),
         O.prefix_error_rates(rx, h, eos=0), what)


which = sys.argv[1:] or ["warp", "group", "cta", "fused", "short", "completion", "mask16", "loss", "seqlp", "ragged"]
if "warp" in which:  # K1: warp per pair (lev_dp.cu), integer and float costs
    run({"B200LEV_BITVEC": "0", "B200LEV_CTA_KERNEL": "0"}, lambda: prefix_case(70, 80, 9, 7, "K1 warp kernel"))
    run({"B200LEV_BITVEC": "0"}, lambda: prefix_case(40, 45, 5, 7, "K1 float costs", ins_cost=0.7, del_cost=1.1, sub_cost=1.3)
        if False else None)
if "group" in which:  # K0 pack + bucketing + K1s lane groups + K3 finalize
    run({"B200LEV_BITVEC": "0", "B200LEV_GROUP_MIN_PAIRS": "1"}, lambda: prefix_case(45, 50, 300, 40, "K1s group kernel"))
if "cta" in which:  # K2: CTA per pair, TMA-staged tokens, inter-warp progress flags
    run({"B200LEV_BITVEC": "0", "B200LEV_CTA_KERNEL": "1"}, lambda: prefix_case(700, 650, 6, 30, "K2 CTA kernel"))
    run({"B200LEV_BITVEC": "0", "B200LEV_CTA_KERNEL": "1"},
        lambda: prefix_case(300, 280, 4, 30, "K2 CTA kernel, costs 3/3/4", ins_cost=3.0, del_cost=3.0, sub_cost=4.0))
if "fused" in which:  # fused bit-vector kernel (shared-memory CAS hash tables) + probe
    run({"B200LEV_BITVEC": "1", "B200LEV_BITVEC_MIN_PAIRS": "1"}, lambda: nbest_case("fused bit-vector kernel"))
    run({"B200LEV_BITVEC_MIN_PAIRS": "1", "B200LEV_GROUP_MIN_PAIRS": "1"},
        lambda: nbest_case("device-selected (probe + fork)"))
if "short" in which:  # short-reference bit-vector kernel: one and two words, prefix rows, bulk totals
    from b200lev import dist as D

    run({"B200LEV_BVSHORT_MIN_PAIRS": "1"}, lambda: prefix_case(30, 35, 70, 12, "short-reference kernel, one word"))
    run({"B200LEV_BVSHORT_MIN_PAIRS": "1"}, lambda: prefix_case(60, 50, 45, 300, "short-reference kernel, two words"))

    def bulk():
        r, h = toks(31, 1100, 500, eos=-1), toks(31, 1100, 500, eos=-1)
        er, acc = D.bulk_error_rate(torch.from_numpy(r).to(dev), torch.from_numpy(h).to(dev), eos=-1)
        exp = np.asarray(O.error_rate(r, h, eos=-1, include_eos=False, norm=False))
        same(er, exp, "bulk scoring: per-pair values")
        assert acc.tolist()[0] == float(exp.astype(np.float64).sum()) and acc.tolist()[2] == 1100.0
        print("ok bulk scoring: totals inside the short-reference kernel", flush=True)

    run({"B200LEV_BVS_CTAS": "2"}, bulk)
if "mask16" in which:  # packed two-pairs-per-warp mask kernel: ring of equality masks in shared memory
    def packed(R, H, N, V, what):
        r, h = toks(R, N, V), toks(H, N, V)
        same(F.optimal_completion(torch.from_numpy(r).to(dev), torch.from_numpy(h).to(dev), eos=0, warn=False),
             O.optimal_completion(r, h, eos=0), what)

    run({"B200LEV_MASK16_MIN_PAIRS": "1"}, lambda: packed(70, 150, 7, 9, "packed mask kernel, small alphabet (no table)"))
    run({"B200LEV_MASK16_MIN_PAIRS": "1"}, lambda: packed(200, 90, 5, 45, "packed mask kernel + warp kernel, rank table"))
if "completion" in which:
    r, h = toks(40, 6, 9), toks(45, 6, 9)
    same(F.optimal_completion(torch.from_numpy(r).to(dev), torch.from_numpy(h).to(dev), eos=0, warn=False),
         O.optimal_completion(r, h, eos=0), "optimal_completion (mask mode + uid + fill)")
if "loss" in which:
    r, h = toks(20, 5, 9), toks(22, 5, 9)
    lg = torch.randn(22, 5, 9, device=dev, requires_grad=True)
    loss = F.hard_optimal_completion_distillation_loss(lg, torch.from_numpy(r).to(dev), torch.from_numpy(h).to(dev),
                                                       eos=0, warn=False)
    loss.backward()
    exp, _ = O.hard_optimal_completion_distillation_loss(lg.detach().cpu().numpy(), r, h, eos=0)
    assert abs(loss.item() - float(exp)) < 1e-5
    h3 = toks(22, 20, 9).reshape(22, 5, 4)
    lp = torch.randn(5, 4, device=dev, requires_grad=True)
    F.minimum_error_rate_loss(lp, torch.from_numpy(r).to(dev), torch.from_numpy(h3).to(dev), eos=0,
                              warn=False).backward()
    print("ok losses", flush=True)
if "seqlp" in which:
    lg = torch.randn(12, 6, 40, device=dev, requires_grad=True)
    hy = torch.from_numpy(toks(12, 6, 40)).to(dev)
    F.sequence_log_probs(lg, hy, 0, eos=0).sum().backward()
    F.ctc_greedy_search(lg.detach(), None, 0)
    print("ok seqlp / ctc", flush=True)
if "ragged" in which:
    utts = [f"u{i}" for i in range(20)]
    rs = [rng.integers(0, 9, int(rng.integers(1, 12))) for _ in utts]
    hs = [rng.integers(0, 9, int(rng.integers(0, 12))) for _ in utts]
    S.score_corpora(S.TokenCorpus.from_sequences(utts, rs), S.TokenCorpus.from_sequences(utts, hs), quiet=True)
    print("ok bulk scoring (ragged kernel)", flush=True)
torch.cuda.synchronize()
print("driver done")
