"""Parity checks shared by the CPU (emulated kernels) and GPU (real kernels) suites.

Every check runs the PRODUCT host code (b200lev.functional / modules) and compares
with either the committed golden fixtures (reference outputs) or the CPU oracle on the
same seeded inputs.  Bars: bit-exact for integer/dyadic costs (distances, counts,
prefix tables, completion targets); rtol 1e-6 for non-dyadic costs, normalised rates,
losses and gradients (stated at each assert).
"""
import warnings

import numpy as np
import pytest
import torch

from oracle import oracle as O

FLOAT_COSTS = {(0.7, 1.1, 1.3), (0.3, 0.3, 0.3), (1.1, 0.9, 1.7)}
RTOL_FLOAT = 1e-6  # the north-star tolerance for non-integer costs / normalised values


def kw_of(p):
    return dict(eos=p["eos"], include_eos=p["include_eos"], batch_first=p["batch_first"],
                ins_cost=p["ins"], del_cost=p["del"], sub_cost=p["sub"])


def assert_same(act, exp, exact, what=""):
    act = act.detach().cpu().numpy() if hasattr(act, "detach") else np.asarray(act)
    assert act.shape == exp.shape, (what, act.shape, exp.shape)
    if exact:
        assert np.array_equal(act, exp), (what, np.abs(act.astype(np.float64) - exp).max())
    else:
        np.testing.assert_allclose(act, exp, rtol=RTOL_FLOAT, atol=0, err_msg=what)


def check_golden_string_matching(F, dev, golden, names=None):
    """error_rate / edit_distance / prefix_* / optimal_completion vs reference outputs."""
    n_checked = 0
    for case, p in golden.params.items():
        if names is not None and case not in names:
            continue
        exact = (p["ins"], p["del"], p["sub"]) not in FLOAT_COSTS
        ref = torch.from_numpy(golden.get(case, "ref")).to(dev)
        hyp = torch.from_numpy(golden.get(case, "hyp")).to(dev)
        kw = kw_of(p)
        for func in ("error_rate", "edit_distance"):
            if golden.has(case, func):
                act = getattr(F, func)(ref, hyp, norm=p["norm"], warn=False, **kw)
                assert_same(act, golden.get(case, func), exact, f"{case}.{func}")
                n_checked += 1
        for func in ("prefix_error_rates", "prefix_edit_distances"):
            if golden.has(case, func):
                act = getattr(F, func)(ref, hyp, norm=p["norm"], padding=p["padding"],
                                       exclude_last=p["exclude_last"], warn=False, **kw)
                assert_same(act, golden.get(case, func), exact, f"{case}.{func}")
                n_checked += 1
        if golden.has(case, "optimal_completion"):
            act = F.optimal_completion(ref, hyp, padding=p["padding"],
                                       exclude_last=p["exclude_last"], warn=False, **kw)
            assert act.dtype == torch.long
            assert_same(act, golden.get(case, "optimal_completion"), True, f"{case}.oc")
            n_checked += 1
    return n_checked


def check_golden_losses(F, dev, golden):
    n = 0
    for case, p in golden.params.items():
        g = golden
        ref = torch.from_numpy(g.get(case, "ref")).to(dev)
        hyp = torch.from_numpy(g.get(case, "hyp")).to(dev)
        go = torch.from_numpy(g.get(case, "grad_output")).to(dev) if g.has(case, "grad_output") else None
        if case.startswith("ocd"):
            x = torch.from_numpy(g.get(case, "logits")).to(dev).requires_grad_(True)
            w = torch.from_numpy(g.get(case, "weight")).to(dev) if p["weight"] else None
            loss = F.hard_optimal_completion_distillation_loss(
                x, ref, hyp, eos=p["eos"], include_eos=p["include_eos"],
                batch_first=p["batch_first"], weight=w, reduction=p["reduction"],
                ignore_index=p["ignore_index"], warn=False)
        else:
            x = torch.from_numpy(g.get(case, "log_probs")).to(dev).requires_grad_(True)
            loss = F.minimum_error_rate_loss(
                x, ref, hyp, eos=p["eos"], include_eos=p["include_eos"], sub_avg=p["sub_avg"],
                batch_first=p["batch_first"], norm=p["norm"], ins_cost=p["ins"],
                del_cost=p["del"], sub_cost=p["sub"], reduction=p["reduction"], warn=False)
        assert loss.dtype == x.dtype
        (grad,) = torch.autograd.grad([loss if go is None else (loss * go).sum()], [x])
        # fp32 losses/gradients: 1e-6 relative to the scale of the result (two fp32
        # implementations of a log-sum-exp differ by a few ulps of the largest term)
        exp_l, exp_g = g.get(case, "loss"), g.get(case, "grad")
        np.testing.assert_allclose(loss.detach().cpu().numpy(), exp_l, rtol=2e-6,
                                   atol=2e-6 * max(1.0, float(np.abs(exp_l).max())), err_msg=case)
        np.testing.assert_allclose(grad.cpu().numpy(), exp_g, rtol=2e-5,
                                   atol=1e-6 * max(1.0, float(np.abs(exp_g).max())), err_msg=case)
        n += 1
    return n


def random_tokens(rng, T, N, V, eos, pad, min_len=0, no_eos_frac=0.0):
    tok = rng.integers(1, max(V, 2), size=(T, N), dtype=np.int64)
    for n in range(N):
        if T == 0 or rng.random() < no_eos_frac:
            continue
        pos = int(rng.integers(min(min_len, T - 1), T))
        tok[pos, n] = eos
        tok[pos + 1:, n] = pad
    return tok


def check_vs_oracle(F, dev, seed, R, H, N, V, costs, eos=0, include_eos=True, norm=False,
                    batch_first=False, exclude_last=False, padding=-100, min_frac=0.3,
                    no_eos_frac=0.0, do_mask=True, dtype=torch.long, spread=1):
    """All DP-backed functionals on one random batch vs the oracle.  `spread` > 1 scales
    the token values so that their range exceeds 16 bits (32-bit compare paths)."""
    rng = np.random.default_rng(seed)
    ref = random_tokens(rng, R, N, V, eos if eos is not None else 0, -2, int(R * min_frac), no_eos_frac)
    hyp = random_tokens(rng, H, N, V, eos if eos is not None else 0, -3, int(H * min_frac), no_eos_frac)
    if spread != 1:
        ref = np.where(ref > 0, ref * spread, ref)
        hyp = np.where(hyp > 0, hyp * spread, hyp)
    if batch_first:
        ref, hyp = np.ascontiguousarray(ref.T), np.ascontiguousarray(hyp.T)
    exact = all(float(c) == round(float(c) * 8) / 8 for c in costs)  # dyadic => exact fp32 sums
    kw = dict(eos=eos, include_eos=include_eos, batch_first=batch_first, ins_cost=costs[0],
              del_cost=costs[1], sub_cost=costs[2])
    tr, th = torch.from_numpy(ref).to(dev).to(dtype), torch.from_numpy(hyp).to(dev).to(dtype)
    for func in ("error_rate", "edit_distance"):
        exp = getattr(O, func)(ref, hyp, norm=norm, **kw)
        act = getattr(F, func)(tr, th, norm=norm, warn=False, **kw)
        assert_same(act, exp, exact and not norm or exact, f"{func} seed={seed}")
    for func in ("prefix_error_rates", "prefix_edit_distances"):
        exp = getattr(O, func)(ref, hyp, norm=norm, padding=padding, exclude_last=exclude_last, **kw)
        act = getattr(F, func)(tr, th, norm=norm, padding=padding, exclude_last=exclude_last,
                               warn=False, **kw)
        assert_same(act, exp, exact, f"{func} seed={seed}")
    if do_mask and exact:
        exp = O.optimal_completion(ref, hyp, padding=padding, exclude_last=exclude_last, **kw)
        act = F.optimal_completion(tr, th, padding=padding, exclude_last=exclude_last, warn=False, **kw)
        assert_same(act, exp, True, f"optimal_completion seed={seed}")


def check_warnings(F, dev):
    """The three data-dependent warnings (SM:175-180, 202-217, 361-366/398-404)."""
    ref = torch.tensor([[1, 2], [2, 0], [3, 0]], device=dev)  # column 0 has no eos(0)
    hyp = torch.tensor([[1, 0], [0, 0]], device=dev)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        F.error_rate(ref, hyp, eos=0, include_eos=True, norm=False)
    assert any("transcription in ref did not" in str(x.message) for x in w)
    assert not any("transcription in hyp did not" in str(x.message) for x in w)
    ref = torch.tensor([[0, 1], [0, 0]], device=dev)  # column 0 is an empty ref
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        er = F.error_rate(ref, hyp, eos=0, norm=True)
        pe = F.prefix_error_rates(ref, hyp, eos=0, include_eos=False, norm=True)
    msgs = [str(x.message) for x in w]
    assert any("Error rates for entries will be 1 if any insertion" in m for m in msgs)
    assert any("0 for prefixes of length 0, 1 otherwise" in m for m in msgs)
    assert er.tolist()[0] == 1.0  # empty ref, non-empty hyp (SM:405)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        F.error_rate(ref, hyp, eos=0, norm=False, ins_cost=2.0)
    assert any("non-uniform error rates" in str(x.message) for x in w)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        F.error_rate(ref, hyp, eos=0, norm=True, ins_cost=2.0, warn=False)
        F.edit_distance(ref, hyp, eos=0, ins_cost=2.0)
    assert not w


def check_errors(F, dev):
    import pytest

    a = torch.zeros(3, 2, dtype=torch.long, device=dev)
    with pytest.raises(RuntimeError, match="must be 2 dimensional"):
        F.error_rate(a[0], a)
    with pytest.raises(RuntimeError, match="ref has batch size 2, but hyp has 3"):
        F.error_rate(a, torch.zeros(3, 3, dtype=torch.long, device=dev))
    with pytest.raises(RuntimeError, match="logits must be 3 dimensional"):
        F.hard_optimal_completion_distillation_loss(torch.zeros(3, 2, device=dev), a, a)
    with pytest.raises(RuntimeError, match="first two dims of logits"):
        F.hard_optimal_completion_distillation_loss(torch.zeros(4, 2, 5, device=dev), a, a)
    with pytest.raises(RuntimeError, match="must be a class idx"):
        F.hard_optimal_completion_distillation_loss(torch.zeros(3, 2, 5, device=dev), a, a, eos=7)
    with pytest.raises(RuntimeError, match="at least two samples"):
        F.minimum_error_rate_loss(torch.zeros(2, 1, device=dev), a,
                                  torch.zeros(3, 2, 1, dtype=torch.long, device=dev))
    with pytest.raises(RuntimeError, match="sample dimensions must match"):
        F.minimum_error_rate_loss(torch.zeros(2, 3, device=dev), a,
                                  torch.zeros(3, 2, 4, dtype=torch.long, device=dev))
    with pytest.raises(RuntimeError, match="not a valid value for reduction"):
        F.minimum_error_rate_loss(torch.zeros(2, 3, device=dev), a,
                                  torch.zeros(3, 2, 3, dtype=torch.long, device=dev),
                                  reduction="bad")


def check_wide_tokens(F, dev, R=70, H=40, N=9):
    """Tokens that differ only above bit 31 must not compare equal (64-bit path)."""
    rng = np.random.default_rng(11)
    ref = random_tokens(rng, R, N, 4, 0, -1, min_len=20)
    hyp = random_tokens(rng, H, N, 4, 0, -1, min_len=20)
    big = np.int64(1) << 32
    ref = np.where((ref > 0) & (rng.random(ref.shape) < 0.5), ref + big, ref)
    hyp = np.where((hyp > 0) & (rng.random(hyp.shape) < 0.5), hyp + 3 * big, hyp)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    for costs in ((1, 1, 1), (1, 2, 3)):
        kw = dict(eos=0, include_eos=True, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
        assert_same(F.edit_distance(tr, th, warn=False, **kw), O.edit_distance(ref, hyp, **kw), True, "wide ed")
        assert_same(F.prefix_error_rates(tr, th, warn=False, **kw), O.prefix_error_rates(ref, hyp, **kw),
                    True, "wide per")
        assert_same(F.optimal_completion(tr, th, warn=False, **kw), O.optimal_completion(ref, hyp, **kw),
                    True, "wide oc")
    # sanity: the narrowed tokens alone would have matched
    assert not np.array_equal(O.edit_distance(ref, hyp, eos=0),
                              O.edit_distance(ref.astype(np.int32), hyp.astype(np.int32), eos=0))


def check_nbest_batch(F, dev, seed, R, H, n_utts, nbest, V=30, shared=True, wide=False, **kw):
    """prefix_error_rates / error_rate on an n-best shaped batch: every reference repeated
    `nbest` times along the batch axis (`shared`), or a batch of unrelated references -- the two
    shapes between which the device-side path selection of lev_bitvec.cu decides."""
    rng = np.random.default_rng(seed)
    ref = random_tokens(rng, R, n_utts, V, 0, -2, 0, 0.1)
    hyp = random_tokens(rng, H, n_utts * nbest, V, 0, -3, 0, 0.1)
    if shared:
        ref = np.repeat(ref, nbest, axis=1)
    else:
        ref = random_tokens(rng, R, n_utts * nbest, V, 0, -2, 0, 0.1)
    if wide:  # tokens outside int32 whose low words collide with ordinary tokens
        ref[min(3, R - 1), :nbest] = (1 << 40) + 5
        hyp[min(2, H - 1), 1] = (1 << 40) + 5
        hyp[min(2, H - 1), 2] = 5
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    for func, okw in (("prefix_error_rates", dict(padding=-7)), ("error_rate", {}),
                      ("prefix_edit_distances", dict(padding=-7, exclude_last=True)),
                      ("edit_distance", {})):
        exp = getattr(O, func)(ref, hyp, eos=0, include_eos=True, **okw, **kw)
        act = getattr(F, func)(tr, th, eos=0, include_eos=True, warn=False, **okw, **kw)
        assert_same(act, exp, True, f"{func} nbest seed={seed} shared={shared}")


def check_grouped_references(F, dev, seed=0):
    """minimum_error_rate_loss on batches whose group size (samples per reference) is 8 or more:
    the call declares its references shared, so the fused bit-vector kernel takes it without a
    probe (lev_bitvec_route: grouped) -- group sizes that divide 32, that do not (a block of 32
    pairs then holds 5 references: two table passes), references of 65 .. 128 tokens (longer or
    shorter ones go elsewhere), sub_avg on and off, and the error rates themselves through the
    registered op."""
    from b200lev import _ops

    rng = np.random.default_rng(seed)
    for R, H, N, M in ((70, 60, 16, 8), (100, 101, 12, 12), (128, 90, 15, 9), (65, 70, 5, 32), (96, 40, 9, 16)):
        ref = random_tokens(rng, R, N, 40, 0, -1, 0, 0.1)
        hyp = random_tokens(rng, H, N * M, 40, 0, -1, 0, 0.1)
        exp_er = O.error_rate(np.repeat(ref, M, axis=1), hyp, eos=0, include_eos=True, norm=True)
        er, _ = _ops.string_matching_impl(torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev), 0, True,
                                          False, 1.0, 1.0, 1.0, True, False, False, 0, True, M)
        assert_same(er, exp_er, True, f"grouped error rates R={R} M={M}")
        lp = rng.standard_normal((N, M)).astype(np.float32)
        for sub_avg in (True, False):
            exp_loss, exp_grad = O.minimum_error_rate_loss(lp, ref, hyp.reshape(H, N, M), eos=0, sub_avg=sub_avg)
            x = torch.from_numpy(lp).to(dev).requires_grad_(True)
            loss = F.minimum_error_rate_loss(x, torch.from_numpy(ref).to(dev),
                                             torch.from_numpy(hyp.reshape(H, N, M)).to(dev), eos=0,
                                             sub_avg=sub_avg, warn=False)
            loss.backward()
            np.testing.assert_allclose(loss.item(), exp_loss, rtol=2e-6, atol=1e-7)
            np.testing.assert_allclose(x.grad.cpu().numpy(), exp_grad, rtol=2e-5, atol=1e-7)


# ---- sequence_log_probs ("next #1", _decoding.py:1516-1548) --------------------------------
# tolerances: fp64 1e-12; fp32 2e-6 relative (+2e-6 absolute: log_softmax of ~10-magnitude
# logits in fp32); bf16 / fp16 one unit in the last place of the result (each step is rounded
# to the dtype before the fp32 sum, as torch does, but torch's summation order differs).
SEQLP_TOL = {"float64": (1e-12, 1e-12), "float32": (2e-6, 2e-6), "bfloat16": (1.6e-2, 1e-2),
             "float16": (2e-3, 2e-3)}


def check_golden_seqlp(F, dev, golden, grads=True):
    n = 0
    for name, p in golden.params.items():
        dt = getattr(torch, p["dtype"])
        rtol, atol = SEQLP_TOL[p["dtype"]]
        logits = torch.from_numpy(golden.get(name, "logits")).to(dev).to(dt).requires_grad_(grads)
        hyp = torch.from_numpy(golden.get(name, "hyp").astype(np.int64)).to(dev)
        out = F.sequence_log_probs(logits, hyp, p["dim"], p["eos"])
        exp = golden.get(name, "out")
        assert out.dtype == dt and tuple(out.shape) == tuple(exp.shape), name
        np.testing.assert_allclose(out.detach().double().cpu().numpy(), exp, rtol=rtol, atol=atol,
                                   err_msg=f"{name} {p}")
        if grads:
            go = torch.from_numpy(golden.get(name, "grad_out")).to(dev).to(dt)
            (out * go).sum().backward()
            # gradients are |g| * softmax-sized: absolute tolerance scaled by |g|
            scale = float(np.abs(golden.get(name, "grad_out")).max()) if exp.size else 1.0
            np.testing.assert_allclose(logits.grad.double().cpu().numpy(), golden.get(name, "grad"),
                                       rtol=rtol, atol=atol * max(scale, 1.0), err_msg=f"grad {name} {p}")
        n += 1
    return n


def check_seqlp_vs_oracle(F, dev, seed, shape, dim, V, eos, dtype=torch.float32):
    rng = np.random.default_rng(seed)
    hyp = rng.integers(-1, V + 1, size=shape)
    lg = torch.tensor(rng.standard_normal(shape + (V,)) * 2.0).to(dtype)
    logits = lg.clone().to(dev).requires_grad_(True)
    out = F.sequence_log_probs(logits, torch.from_numpy(hyp).to(dev), dim, eos)
    g = rng.standard_normal(tuple(out.shape))
    (out * torch.tensor(g).to(dev).to(dtype)).sum().backward()
    exp, gexp = O.sequence_log_probs(lg.double().numpy(), hyp, dim, eos,
                                     grad_out=torch.tensor(g).to(dtype).double().numpy())
    rtol, atol = SEQLP_TOL[str(dtype).split(".")[-1]]
    np.testing.assert_allclose(out.detach().double().cpu().numpy(), exp, rtol=rtol, atol=atol * 4)
    np.testing.assert_allclose(logits.grad.double().cpu().numpy(), gexp, rtol=rtol,
                               atol=atol * max(1.0, float(np.abs(g).max()) if g.size else 1.0))


# ---- bulk-scoring front end (b200lev.scoring) against the reference command's own output ----
def _scoring_tensor(seq, kind):
    t = torch.tensor(seq, dtype=torch.long)
    if kind == "col1":
        return t.unsqueeze(-1)
    if kind == "timed":
        n = t.shape[0]
        start = torch.arange(n) * 3
        return torch.stack([t, start, start + 2], -1) if n else torch.zeros((0, 3), dtype=torch.long)
    return t


def build_scoring_dirs(golden, tmp):
    """Rebuild the token data directories make_golden_scoring.py ran the reference on."""
    import os

    def write(root, utts, prefix="", suffix=".pt", drop_ref=(), drop_hyp=()):
        for side, drop in (("ref", drop_ref), ("hyp", drop_hyp)):
            os.makedirs(os.path.join(root, side), exist_ok=True)
            for utt, d in utts.items():
                if utt not in drop:
                    torch.save(_scoring_tensor(d[side], d[side + "_kind"]),
                               os.path.join(root, side, prefix + utt + suffix))
            torch.save(torch.zeros(2, dtype=torch.long), os.path.join(root, side, "stray.bin"))

    A, B = golden["corpora"]["A"], golden["corpora"]["B"]
    for name, text in golden["files"].items():
        with open(os.path.join(tmp, name), "w") as f:
            f.write(text)
    write(os.path.join(tmp, "A"), A)
    write(os.path.join(tmp, "B"), B)
    write(os.path.join(tmp, "Apre"), A, prefix="tok_", suffix=".tok")
    write(os.path.join(tmp, "Amiss"), A, **golden["missing"])


def check_golden_scoring(scoring, golden, tmp):
    import os
    import warnings

    tmp = str(tmp)
    build_scoring_dirs(golden, tmp)
    n = 0
    for case in golden["cases"]:
        where, opts = case["where"], case["opts"]
        if "+" in where:
            dirs = [os.path.join(tmp, x) for x in where.split("+")]
        else:
            dirs = [os.path.join(tmp, where, "ref"), os.path.join(tmp, where, "hyp")]
        out = os.path.join(tmp, f"out{n}.txt")
        args = dirs + [out] + [os.path.join(tmp, o[1:]) if o.startswith("@") else o for o in opts]
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            if "raises" in case:
                exc = {"ValueError": ValueError, "ZeroDivisionError": ZeroDivisionError}[case["raises"]]
                with pytest.raises(exc) as info:
                    scoring.compute_torch_token_data_dir_error_rates(args)
                assert str(info.value) == case["message"].replace("{tmp}", tmp), (where, opts)
            else:
                assert scoring.compute_torch_token_data_dir_error_rates(args) == case["rc"], (where, opts)
                with open(out) as f:
                    got = f.read()
                assert got == case["out"], (where, opts, got[:200])
        missing = sorted(str(x.message) for x in w if "does not contain" in str(x.message))
        assert missing == [m.replace("{tmp}", tmp) for m in case["warned_missing"]], (where, opts)
        n += 1
    return n


def check_ragged_to_padded(dev, seed=0):
    """b200lev_ragged_to_padded against pad_sequence over (utterance + [eos]), the reference's
    own construction (command_line.py:1110-1121)."""
    from b200lev import _abi, _ops

    rng = np.random.default_rng(seed)
    n = 0
    for dtype in (torch.int16, torch.int32, torch.int64):
        for N, L in ((1, 0), (7, 5), (300, 40), (33, 1)):
            lens = rng.integers(0, L + 1, N)
            seqs = [torch.from_numpy(rng.integers(0, 1000, int(k))).to(dtype) for k in lens]
            off = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)).to(dev)
            flat = (torch.cat(seqs) if N else torch.zeros(0, dtype=dtype)).to(dev)
            T = int(lens.max()) + 1 + int(rng.integers(0, 3))
            eos = torch.tensor([-1], dtype=dtype)

            def expect(idx):
                rows = torch.nn.utils.rnn.pad_sequence([torch.cat([seqs[i], eos]) for i in idx],
                                                       padding_value=-2, batch_first=True)
                full = torch.full((len(idx), T), -2, dtype=dtype)
                full[:, :rows.shape[1]] = rows
                return full

            got = _ops.ragged_to_padded(flat, off, None, 0, N, T, -1, -2)
            assert got.dtype == dtype and torch.equal(got.cpu(), expect(range(N)))
            a, b = N // 3, N - N // 4
            got = _ops.ragged_to_padded(flat, off, None, a, b - a, T, -1, -2)
            assert torch.equal(got.cpu(), expect(range(a, b)))
            sel = rng.permutation(N)[: max(1, N // 2)]
            got = _ops.ragged_to_padded(flat, off, torch.from_numpy(sel).to(dev), 0, len(sel), T, -1, -2)
            assert torch.equal(got.cpu(), expect(sel.tolist()))
            n += 3
    flat = torch.zeros(4, dtype=torch.int32, device=dev)
    off = torch.tensor([0, 4], dtype=torch.int64, device=dev)
    with pytest.raises(_abi.B200LevError, match="int16/int32/int64"):
        _ops.ragged_to_padded(flat.to(torch.int8), off, None, 0, 1, 5, -1, -2)
    with pytest.raises(_abi.B200LevError, match="outside offsets"):
        _ops.ragged_to_padded(flat, off, None, 1, 1, 5, -1, -2)
    with pytest.raises(_abi.B200LevError, match="sel must hold"):
        _ops.ragged_to_padded(flat, off, torch.zeros(2, dtype=torch.int64, device=dev), 0, 1, 5, -1, -2)
    assert _ops.ragged_to_padded(flat, off, None, 0, 0, 3, -1, -2).shape == (0, 3)
    return n


# ---- ctc_greedy_search (_decoding.py:507-560) ------------------------------------------------
# relative, on a sum / product over T steps; a log-probability is max - logsumexp, so in logits
# mode each step also carries an absolute error of the order eps * |logsumexp| (1e-6 per step)
CTC_TOL = {"float32": 2e-6, "float64": 1e-12}


def _ctc_case(golden, name):
    p = golden.params[name]
    dt = getattr(torch, p["dtype"])
    logits = torch.from_numpy(golden.get(name, "logits")).to(dt)
    lens = torch.from_numpy(golden.get(name, "in_lens").astype(np.int64)) if p["lens"] else None
    return p, logits, lens


def check_golden_ctc(F, dev, golden):
    n = 0
    for name in golden.params:
        p, logits, lens = _ctc_case(golden, name)
        max_, paths, out_lens = F.ctc_greedy_search(logits.to(dev), None if lens is None else lens.to(dev),
                                                    p["blank_idx"], p["batch_first"], p["is_probs"])
        assert max_.dtype == logits.dtype and paths.dtype == torch.long and out_lens.dtype == torch.long
        np.testing.assert_array_equal(paths.cpu().numpy(), golden.get(name, "paths"), err_msg=f"{name} {p}")
        np.testing.assert_array_equal(out_lens.cpu().numpy(), golden.get(name, "out_lens"), err_msg=name)
        T = logits.shape[1 if p["batch_first"] else 0]
        tol = CTC_TOL[p["dtype"]]
        np.testing.assert_allclose(max_.double().cpu().numpy(), golden.get(name, "max").astype(np.float64),
                                   rtol=tol, atol=1e-30 if p["is_probs"] else tol * T, err_msg=f"{name} {p}")
        n += 1
    return n


def check_ctc_vs_oracle(F, dev, seed, T, N, V, batch_first, dtype=torch.float32, with_lens=True):
    """Forward and the gradient of max_ (logits mode) against the float64 oracle."""
    rng = np.random.default_rng(seed)
    shape = (N, T, V) if batch_first else (T, N, V)
    x = torch.tensor(rng.standard_normal(shape) * 2.0).to(dtype)
    lens = torch.from_numpy(rng.integers(0, T + 2, N)) if with_lens else None
    g = rng.standard_normal(N)
    logits = x.clone().to(dev).requires_grad_(True)
    max_, paths, out_lens = F.ctc_greedy_search(logits, None if lens is None else lens.to(dev), 1, batch_first)
    (max_ * torch.tensor(g).to(dev).to(dtype)).sum().backward()
    e_max, e_paths, e_lens, e_grad = O.ctc_greedy_search(x.double().numpy(), None if lens is None else lens.numpy(),
                                                         1, batch_first, False, grad_out=g)
    np.testing.assert_array_equal(paths.cpu().numpy(), e_paths)
    np.testing.assert_array_equal(out_lens.cpu().numpy(), e_lens)
    rtol, atol = SEQLP_TOL[str(dtype).replace("torch.", "")]
    np.testing.assert_allclose(max_.detach().double().cpu().numpy(), e_max, rtol=max(rtol, 2e-6), atol=max(atol, 2e-6 * T))
    np.testing.assert_allclose(logits.grad.double().cpu().numpy(), e_grad, rtol=rtol,
                               atol=atol * max(1.0, float(np.abs(g).max())))


def check_ctc_probs_gradient(F, dev, seed=0):
    """is_probs=True: the path probability is a product over the valid steps; its gradient equals
    torch's through the reference formula (_decoding.py:527-553), zeros among the chosen
    probabilities included, both layouts."""
    g = torch.Generator().manual_seed(seed)
    T, N, V = 9, 6, 7
    p = torch.rand(T, N, V, generator=g).softmax(2)
    p[2, 1, :] = 0.0
    p[2, 1, 3] = 1.0
    p[4, 2, :] = 0.0  # a step whose maximum is zero: the product is zero, its gradient is not
    lens = torch.tensor([9, 3, 7, 1, 6, 9])
    w = torch.rand(N, generator=g)
    for batch_first in (False, True):
        src = p.transpose(0, 1).contiguous() if batch_first else p
        x = src.clone().to(dev).requires_grad_(True)
        m, _, _ = F.ctc_greedy_search(x, lens.to(dev), batch_first=batch_first, is_probs=True)
        (ga,) = torch.autograd.grad(m, x, w.to(dev))
        y = src.clone().requires_grad_(True)
        yy = y if batch_first else y.transpose(0, 1)
        mx, _ = yy.max(2)
        mask = torch.arange(T).unsqueeze(0) < lens.unsqueeze(1)
        mref = mx.masked_fill(~mask, 1.0).prod(1)
        (gb,) = torch.autograd.grad(mref, y, w)
        assert torch.allclose(m.detach().cpu(), mref.detach(), rtol=1e-6, atol=1e-8)
        assert torch.allclose(ga.cpu(), gb, rtol=1e-5, atol=1e-8), (ga.cpu() - gb).abs().max()


def check_ctc_masked_classes(F, dev):
    """-inf logits (masked classes), including rows that START with -inf vectors and a class
    count that leaves a scalar tail: arg max, lengths and score against the oracle."""
    rng = np.random.default_rng(12)
    for V in (5, 37, 300, 1031):
        x = rng.standard_normal((11, 3, V)) * 2.0
        x[:, :, : V // 2] = -np.inf          # the first half of every row is masked
        x[rng.random((11, 3, V)) < 0.2] = -np.inf
        x[:, :, V - 1] = np.where(np.isinf(x).all(axis=2), 0.0, x[:, :, V - 1])  # no all-masked row
        t = torch.tensor(x, dtype=torch.float32)
        max_, paths, out_lens = F.ctc_greedy_search(t.to(dev), None, V - 1)
        e_max, e_paths, e_lens = O.ctc_greedy_search(t.double().numpy(), None, V - 1)
        np.testing.assert_array_equal(paths.cpu().numpy(), e_paths)
        np.testing.assert_array_equal(out_lens.cpu().numpy(), e_lens)
        np.testing.assert_allclose(max_.double().cpu().numpy(), e_max, rtol=2e-6, atol=2e-5)


# ---------------------------------------------------------------------------------------
# fill_after_eos and the nn.Module shells under nojit / trace / script
# ---------------------------------------------------------------------------------------
def check_completion_small_alphabets(F, dev, seed=0):
    """optimal_completion where the call's tokens span 31 / 32 / 33 / 40 values, around zero and
    far from it: up to 32 the bitmaps index tokens by their offset from the smallest one
    (lev_tokens_direct), above that by their rank in the sorted reference -- same outputs."""
    rng = np.random.default_rng(seed)
    for lo in (-17, 0, 5, 1 << 20, -(1 << 30)):
        for span in (2, 31, 32, 33, 40):
            R, H, N = 37, 33, 21
            ref = rng.integers(lo, lo + span, size=(R, N)).astype(np.int64)
            hyp = rng.integers(lo, lo + span, size=(H, N)).astype(np.int64)
            ref[0, 0], ref[1, 0] = lo, lo + span - 1  # the whole span is present
            eos = lo + 1
            for kw in (dict(eos=eos, include_eos=True), dict(eos=None), dict(eos=eos, include_eos=False, exclude_last=True)):
                exp = O.optimal_completion(ref, hyp, **kw)
                act = F.optimal_completion(torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev),
                                           warn=False, **kw)
                assert_same(act, exp, True, f"small alphabet lo={lo} span={span} {kw}")


def check_fill_after_eos(F, dev, seed=0):
    """SM:30-42 against the oracle: every axis, negative axes, integer and float fills, a
    broadcast ``value`` tensor, float "tokens" (the reference's trace placeholders), 1-D and
    0-sized inputs."""
    rng = np.random.default_rng(seed)
    tok = rng.integers(0, 5, (7, 6, 3))
    t = torch.from_numpy(tok).to(dev)
    for dim in (0, 1, 2, -1, -3):
        exp = O.fill_after_eos(tok, 2, dim=dim, fill=-9)
        assert np.array_equal(F.fill_after_eos(t, 2, dim=dim, fill=-9).cpu().numpy(), exp), dim
    assert np.array_equal(F.fill_after_eos(t, 3).cpu().numpy(), O.fill_after_eos(tok, 3))
    val = rng.standard_normal((7, 6, 4)).astype(np.float32)
    exp = O.fill_after_eos(tok[:, :, :1], 2, value=val)
    act = F.fill_after_eos(t[:, :, :1], 2, value=torch.from_numpy(val).to(dev))
    assert np.array_equal(act.cpu().numpy(), exp)
    flt = F.fill_after_eos(t.float(), 2, dim=1, fill=0.5)
    assert flt.dtype == torch.float32
    assert np.array_equal(flt.cpu().numpy(), O.fill_after_eos(tok.astype(np.float32), 2, dim=1, fill=0.5))
    one = torch.tensor([4, 1, 1, 3, 1], device=dev)
    assert F.fill_after_eos(one, 1, fill=7).tolist() == [4, 1, 7, 7, 7]
    assert F.fill_after_eos(torch.zeros((0, 3), dtype=torch.long, device=dev), 1).shape == (0, 3)
    big = rng.integers(0, 50, (300, 257))
    assert np.array_equal(F.fill_after_eos(torch.from_numpy(big).to(dev), 7, dim=0).cpu().numpy(),
                          O.fill_after_eos(big, 7, dim=0))
    assert np.array_equal(F.fill_after_eos(torch.from_numpy(big).to(dev), 7, dim=1).cpu().numpy(),
                          O.fill_after_eos(big, 7, dim=1))


def _jit(module, jit_type, example):
    if jit_type == "script":
        return torch.jit.script(module)
    if jit_type == "trace":
        return torch.jit.trace(module, example)
    return module


def check_modules(F, M, dev, jit_type):
    """Every module of the family (modules.py:115-124 of the reference), plain, traced with the
    tiny placeholder inputs the reference's tests use (TS:43, 86, 150, 219, 249-255) and
    scripted: same numbers as the functional on inputs of OTHER shapes than the example's,
    which is what catches shape logic baked into a graph."""
    rng = np.random.default_rng(17)
    eos = 0
    ref_np, hyp_np = random_tokens(rng, 9, 6, 5, eos, -1), random_tokens(rng, 11, 6, 5, eos, -1)
    ref, hyp = torch.from_numpy(ref_np).to(dev), torch.from_numpy(hyp_np).to(dev)
    tok11 = (torch.full((1, 1), eos, dtype=torch.long, device=dev),) * 2
    flt11 = (torch.zeros(1, 1, device=dev),) * 2  # the reference traces with float tokens too
    cases = [
        (M.ErrorRate(eos=eos, warn=False), flt11, F.error_rate, dict(eos=eos, warn=False)),
        (M.ErrorRate(eos=eos, include_eos=True, norm=False, ins_cost=2.0, warn=False), tok11,
         F.error_rate, dict(eos=eos, include_eos=True, norm=False, ins_cost=2.0, warn=False)),
        (M.EditDistance(eos=eos, ins_cost=3.0, del_cost=3.0, sub_cost=4.0), tok11, F.edit_distance,
         dict(eos=eos, ins_cost=3.0, del_cost=3.0, sub_cost=4.0)),
        (M.PrefixErrorRates(eos=eos, padding=-3, warn=False), tok11, F.prefix_error_rates,
         dict(eos=eos, padding=-3, warn=False)),
        (M.PrefixEditDistances(eos=eos, exclude_last=True, norm=True, warn=False), tok11,
         F.prefix_edit_distances, dict(eos=eos, exclude_last=True, norm=True, warn=False)),
        (M.OptimalCompletion(eos=eos, padding=-7), tok11, F.optimal_completion,
         dict(eos=eos, padding=-7)),
        (M.OptimalCompletion(eos=None, exclude_last=True, include_eos=False), tok11,
         F.optimal_completion, dict(eos=None, exclude_last=True, include_eos=False)),
    ]
    for mod, example, fn, kw in cases:
        jm = _jit(mod, jit_type, example)
        for r, h in ((ref, hyp), (ref[:, :3], hyp[:5, :3])):
            want = fn(r, h, **kw)
            got = jm(r, h)
            assert got.shape == want.shape and torch.equal(got, want), (type(mod).__name__, jit_type)
            assert np.array_equal(got.cpu().numpy(), getattr(O, fn.__name__)(
                r.cpu().numpy(), h.cpu().numpy(), **{k: v for k, v in kw.items() if k != "warn"}))
    # batch_first modules
    mod = M.PrefixErrorRates(eos=eos, batch_first=True, warn=False)
    jm = _jit(mod, jit_type, tok11)
    assert torch.equal(jm(ref.t(), hyp.t()), F.prefix_error_rates(ref, hyp, eos=eos, warn=False).t())
    # FillAfterEndOfSequence (TS:31-52: traced on 1-element float placeholders, run on 3-D)
    fa = M.FillAfterEndOfSequence(4)
    jf = _jit(fa, jit_type, (torch.empty(1, device=dev), torch.empty(1, device=dev)))
    tok = torch.from_numpy(rng.integers(0, 5, (8, 6))).to(dev)
    logits = torch.randn(8, 6, 5, device=dev)
    if jit_type != "trace":  # a module traced with (tokens, value) takes exactly those two
        assert np.array_equal(jf(tok).cpu().numpy(), O.fill_after_eos(tok.cpu().numpy(), 4))
    assert np.array_equal(jf(tok.unsqueeze(2), logits).cpu().numpy(),
                          O.fill_after_eos(tok.unsqueeze(2).cpu().numpy(), 4, value=logits.cpu().numpy()))
    # HardOptimalCompletionDistillationLoss: forward + gradient, sizes other than the example's
    V = 5
    for reduction in ("mean", "sum", "none"):
        ocd = M.HardOptimalCompletionDistillationLoss(eos=eos, reduction=reduction)
        jo = _jit(ocd, jit_type, (torch.empty(1, 1, V, device=dev),) + tok11)
        lg = torch.randn(11, 6, V, device=dev, requires_grad=True)
        loss = jo(lg, ref, hyp)
        exp_loss, exp_grad = O.hard_optimal_completion_distillation_loss(
            lg.detach().cpu().numpy(), ref_np, hyp_np, eos=eos, reduction=reduction,
            ignore_index=-100, grad_output=None)
        assert np.allclose(loss.detach().cpu().numpy(), exp_loss, rtol=2e-6, atol=2e-6), reduction
        (loss if reduction != "none" else loss.sum()).backward()
        assert np.allclose(lg.grad.cpu().numpy(), exp_grad, rtol=2e-5, atol=1e-6), reduction
    # MinimumErrorRateLoss: traced on (2, 2) / (2, 2, 2) placeholders, run on 6 x 4 samples,
    # 2-D and 3-D references (TS:224-270)
    nb, ns = 6, 4
    hyp3_np = random_tokens(rng, 7, nb * ns, 5, eos, -1).reshape(7, nb, ns)
    hyp3 = torch.from_numpy(hyp3_np).to(dev)
    ex = (torch.empty(2, 2, device=dev), torch.zeros(2, 2, dtype=torch.long, device=dev),
          torch.zeros(2, 2, 2, dtype=torch.long, device=dev))
    for reduction, sub_avg in (("mean", True), ("sum", False), ("none", True)):
        mw = M.MinimumErrorRateLoss(eos=eos, sub_avg=sub_avg, reduction=reduction)
        jw = _jit(mw, jit_type, ex)
        lp = torch.randn(nb, ns, device=dev, requires_grad=True)
        for r3 in (ref, ref.unsqueeze(-1).repeat(1, 1, ns)):
            lp.grad = None
            loss = jw(lp, r3, hyp3)
            exp_loss, exp_grad = O.minimum_error_rate_loss(
                lp.detach().cpu().numpy(), ref_np, hyp3_np, eos=eos, sub_avg=sub_avg,
                reduction=reduction,
                grad_output=None)
            assert np.allclose(loss.detach().cpu().numpy(), exp_loss, rtol=2e-6, atol=2e-6)
            (loss if reduction != "none" else loss.sum()).backward()
            assert np.allclose(lp.grad.cpu().numpy(), exp_grad, rtol=2e-5, atol=1e-6)
    mb = M.MinimumErrorRateLoss(eos=eos, batch_first=True)
    jb = _jit(mb, jit_type, ex)
    lp = torch.randn(nb, ns, device=dev)
    assert torch.allclose(jb(lp, ref.t(), hyp3.permute(1, 2, 0)),
                          F.minimum_error_rate_loss(lp, ref, hyp3, eos=eos))
    if jit_type != "nojit":  # the checks stay dynamic in a graph (SM:1417-1450)
        with pytest.raises(Exception, match="sample dimensions must match"):
            jw(torch.randn(nb, ns + 1, device=dev), ref, hyp3)


# ---------------------------------------------------------------------------------------
# N-best producers' step functions (SURVEY 8f #3)
# ---------------------------------------------------------------------------------------
def _decode_case(golden, name):
    p = golden.params[name]
    get = lambda f: golden.get(name, f) if golden.has(name, f) else None  # noqa: E731
    return p, get


def check_golden_decode(F, dev, golden):
    """tests/golden/decode.npz (outputs of the unmodified reference): beam_search_advance bit
    for bit -- paths, lengths, sources, scores (the padding columns' tokens are uninitialised in
    the reference and skipped); random_walk_advance replayed on the reference's random stream
    where the device allows it (CPU tensors here are computed on the GPU, whose stream differs),
    and checked against the oracle with the tokens torch drew."""
    n = 0
    for name in golden.names("beam"):
        p, get = _decode_case(golden, name)
        t = lambda a: None if a is None else torch.from_numpy(a).to(dev)  # noqa: E731
        y_next, y_lens, lp, src = F.beam_search_advance(t(get("log_probs_t")), p["width"], t(get("log_probs_prev")),
                                                        t(get("y_prev")), t(get("y_prev_lens")))
        K = p["K"]
        assert np.array_equal(y_next.cpu().numpy()[:, :, :K], get("y_next")[:, :, :K]), name
        assert y_next.shape == get("y_next").shape, name
        assert np.array_equal(y_lens.cpu().numpy(), get("y_next_lens")), name
        assert np.array_equal(lp.cpu().numpy(), get("log_probs_next")), name
        assert np.array_equal(src.cpu().numpy(), get("next_src")), name
        assert lp.dtype == t(get("log_probs_t")).dtype
        n += 1
    for name in golden.names("walk"):
        p, get = _decode_case(golden, name)
        t = lambda a: None if a is None else torch.from_numpy(a).to(dev)  # noqa: E731
        torch.manual_seed(p["seed"])
        y_next, lp = F.random_walk_advance(t(get("log_probs_t")), t(get("log_probs_prev")), t(get("y_prev")),
                                           t(get("y_prev_lens")))
        assert y_next.shape == get("y_next").shape, name
        N = y_next.shape[1]
        lens = get("y_prev_lens")
        pos = lens if lens is not None else np.full(N, get("y_prev").shape[0])
        drawn = y_next.cpu().numpy()[pos, np.arange(N)]
        ey, elp = O.random_walk_advance(get("log_probs_t"), get("log_probs_prev"), get("y_prev"), drawn, lens)
        assert np.array_equal(y_next.cpu().numpy(), ey), name
        assert np.allclose(lp.cpu().numpy(), elp, rtol=1e-6, atol=1e-6), name
        if dev.type == "cpu" and y_next.device.type == "cpu" and not torch.cuda.is_available():
            # same device, same stream as the reference's run: the draw itself reproduces
            assert np.array_equal(y_next.numpy(), get("y_next")), name
        n += 1
    return n


def check_decode_vs_oracle(F, dev, seed=0):
    """Random shapes incl. ties (coarse dtypes), too-narrow candidate sets, strided inputs, a
    vocabulary-sized step, and the error messages (_decoding.py:95-116, 1249-1265)."""
    g = torch.Generator().manual_seed(seed)
    for dtype in (torch.float32, torch.float64, torch.bfloat16, torch.float16):
        for (N, Kp, V, W, S) in ((3, 4, 50, 6, 5), (2, 2, 3, 9, 2), (4, 8, 2000, 8, 10), (1, 1, 1, 1, 0)):
            lpt = torch.randn(N, Kp, V, generator=g).to(dtype)
            lpp = torch.randn(N, Kp, generator=g).to(dtype)
            yp = torch.randint(0, V, (S, N, Kp), generator=g)
            lens = torch.randint(0, S + 1, (N, Kp), generator=g)
            for ln in (None, lens):
                got = F.beam_search_advance(lpt.to(dev), W, lpp.to(dev), yp.to(dev), None if ln is None else ln.to(dev))
                f64 = dtype == torch.float64
                npd = lambda a: a.double().numpy() if f64 else a.float().numpy()  # noqa: E731
                if dtype in (torch.bfloat16, torch.float16):
                    # the oracle sums in fp32 and rounds like torch: emulate the rounding
                    cand = (lpp.float().unsqueeze(2) + lpt.float()).to(dtype).float().numpy()
                    exp = O.beam_search_advance(cand, W, np.zeros((N, Kp), np.float32), yp.numpy(),
                                                None if ln is None else ln.numpy())
                else:
                    exp = O.beam_search_advance(npd(lpt), W, npd(lpp), yp.numpy(), None if ln is None else ln.numpy())
                assert np.array_equal(got[0].cpu().numpy(), exp[0]), (dtype, N, Kp, V, W, S)
                assert np.array_equal(got[1].cpu().numpy(), exp[1])
                assert np.array_equal(got[2].float().cpu().numpy() if not f64 else got[2].cpu().numpy(),
                                      exp[2].astype(np.float64 if f64 else np.float32))
                assert np.array_equal(got[3].cpu().numpy(), exp[3])
    # strided log-probabilities (a transposed view)
    lpt = torch.randn(7, 3, 4, generator=g).permute(1, 2, 0)
    got = F.beam_search_advance(lpt.to(dev), 5, torch.zeros(3, 4).to(dev), torch.zeros((0, 3, 4), dtype=torch.long).to(dev))
    exp = O.beam_search_advance(lpt.numpy(), 5, np.zeros((3, 4), np.float32), np.zeros((0, 3, 4), np.int64))
    assert np.array_equal(got[3].cpu().numpy(), exp[3]) and np.array_equal(got[0].cpu().numpy(), exp[0])
    z = torch.zeros
    with pytest.raises(RuntimeError, match="log_probs_t must be 3 dimensional"):
        F.beam_search_advance(z(2, 3).to(dev), 1, z(2, 3).to(dev), z(0, 2, 3, dtype=torch.long).to(dev))
    with pytest.raises(RuntimeError, match="Expected width to be >= 1"):
        F.beam_search_advance(z(2, 3, 4).to(dev), 0, z(2, 3).to(dev), z(0, 2, 3, dtype=torch.long).to(dev))
    with pytest.raises(RuntimeError, match="Expected log_probs_prev to be of shape"):
        F.beam_search_advance(z(2, 3, 4).to(dev), 1, z(2, 4).to(dev), z(0, 2, 3, dtype=torch.long).to(dev))
    with pytest.raises(RuntimeError, match="Invalid lengths for t=0"):
        F.beam_search_advance(z(2, 3, 4).to(dev), 1, z(2, 3).to(dev), z(0, 2, 3, dtype=torch.long).to(dev),
                              torch.ones(2, 3, dtype=torch.long).to(dev))
    with pytest.raises(RuntimeError, match="log_probs_t must be 2-dimensional"):
        F.random_walk_advance(z(2, 3, 4).to(dev), z(2).to(dev), z(0, 2, dtype=torch.long).to(dev))
    with pytest.raises(RuntimeError, match="Expected dim 1 of y_prev"):
        F.random_walk_advance(z(2, 3).to(dev), z(2).to(dev), z(0, 3, dtype=torch.long).to(dev))
    # greedy decoding through the step function (tests/test_decoding.py:283-294 of the reference)
    T, N, C = 9, 4, 20
    logits = torch.randn(T, N, C, generator=g).to(dev)
    y = torch.empty((0, N, 1), dtype=torch.long, device=dev)
    lp = torch.zeros((N, 1), device=dev)
    for lt in logits:
        y, _, lp, _ = F.beam_search_advance(lt.unsqueeze(1), 1, lp, y)
    mx, am = logits.max(2)
    assert torch.equal(y.squeeze(2), am) and torch.allclose(lp.squeeze(1), mx.sum(0))


def check_golden_seqlp_packed(F, dev, golden):
    """sequence_log_probs with PackedSequence logits (_decoding.py:1551-1586) against the
    reference's outputs and gradients (fp32: 2e-6 relative + 2e-6 absolute)."""
    n = 0
    for name in golden.names("ps"):
        p = golden.params[name]
        data = torch.from_numpy(golden.get(name, "data")).to(dev).requires_grad_(True)
        parts = list(data.split(p["lens"]))
        packed = torch.nn.utils.rnn.pack_sequence(parts, enforce_sorted=p["enforce_sorted"])
        hyp = torch.from_numpy(golden.get(name, "hyp")).to(dev)
        out = F.sequence_log_probs(packed, hyp, p["dim"])
        assert np.allclose(out.detach().cpu().numpy(), golden.get(name, "out"), rtol=2e-6, atol=2e-6), name
        (grad,) = torch.autograd.grad(out, data, torch.from_numpy(golden.get(name, "grad_out")).to(dev))
        assert np.allclose(grad.cpu().numpy(), golden.get(name, "grad"), rtol=2e-6, atol=2e-6), name
        n += 1
    with pytest.raises(RuntimeError, match="either a Tensor or PackedSequence"):
        F.sequence_log_probs([1, 2], torch.zeros(2, 2, dtype=torch.long))
    return n
