"""pairwise_error_rates / pairwise_edit_distances (every reference of a group against every
hypothesis of it) and minimum_bayes_risk.

The definition is the materialised cross product: out[g, a, b] is error_rate (edit_distance) of
reference (g, a) against hypothesis (g, b).  The expected values come from the oracle on those
materialised pairs and are compared bit for bit, on the SIMT emulator (tests/emu) and on the
device.  minimum_bayes_risk is compared with a float64 numpy restatement of its formula.
"""
import ctypes
import warnings

import numpy as np
import pytest
import torch

import parity_cases as PC
from oracle import oracle as O

COSTS = [(1, 1, 1), (3, 3, 4), (1, 2, 3), (0.5, 1.0, 0.25), (0.7, 1.1, 1.3)]
SHAPES = [(1, 1), (3, 5), (8, 8), (5, 13)]  # (A, B); 5 x 13 = 65 pairs: groups straddle warps
# (norm, eos, include_eos), rotated over the cases
VARIANTS = [(True, 0, False), (False, 0, True), (True, None, False), (False, 0, False)]


def _materialise(ref, hyp):
    """(R, G, A) and (H, G, B) -> the (R, G*A*B) and (H, G*A*B) pairs, pair (g*A + a)*B + b."""
    R, G, A = ref.shape
    H, _, B = hyp.shape
    refx = np.repeat(ref.reshape(R, G * A), B, axis=1)
    hypx = np.ascontiguousarray(np.broadcast_to(hyp[:, :, None, :], (H, G, A, B)).reshape(H, G * A * B))
    return refx, hypx


def _expected(ref, hyp, costs=(1, 1, 1), eos=None, include_eos=False, norm=True, mistakes=True, flags=False):
    refx, hypx = _materialise(ref, hyp)
    out, fl, _, _ = O.string_matching(refx, hypx, eos, include_eos, False, *costs, norm=norm,
                                      return_mistakes=mistakes)
    out = out.reshape(ref.shape[1], ref.shape[2], hyp.shape[2])
    return (out, fl) if flags else out


def _groups(seed, R, H, G, A, B, V=7, eos=0, no_eos_frac=0.0, min_frac=0.3):
    rng = np.random.default_rng(seed)
    ref = PC.random_tokens(rng, R, G * A, V, eos, -2, int(R * min_frac), no_eos_frac).reshape(R, G, A)
    hyp = PC.random_tokens(rng, H, G * B, V, eos, -3, int(H * min_frac), no_eos_frac).reshape(H, G, B)
    return ref, hyp


def _route(capfd):
    err = capfd.readouterr().err
    if "short cross form" in err:
        return "short"
    assert "gather + final" in err, err
    return "gather"


def _same_as_materialised(F, act, exp, ref, hyp, costs, mistakes, dev=torch.device("cpu"), **kw):
    """Bit for bit with the oracle; for non-dyadic costs, where the library's error_rate itself
    agrees with the oracle to rtol 1e-6 only (parity_cases.FLOAT_COSTS), bit for bit with the
    library's error_rate / edit_distance on the materialised pairs."""
    if costs not in PC.FLOAT_COSTS:
        assert np.array_equal(act, exp), (mistakes, np.abs(act - exp).max())
        return
    np.testing.assert_allclose(act, exp, rtol=PC.RTOL_FLOAT, atol=0)
    refx, hypx = _materialise(ref, hyp)
    f = F.error_rate if mistakes else F.edit_distance
    lib = f(torch.from_numpy(refx).to(dev), torch.from_numpy(hypx).to(dev), ins_cost=costs[0], del_cost=costs[1],
            sub_cost=costs[2], warn=False, **kw)
    assert np.array_equal(act.reshape(-1), lib.cpu().numpy())


def _call(F, ref, hyp, costs, mistakes=True, dev=torch.device("cpu"), dtype=torch.long, **kw):
    f = F.pairwise_error_rates if mistakes else F.pairwise_edit_distances
    tr = torch.from_numpy(ref).to(dev).to(dtype)
    th = torch.from_numpy(hyp).to(dev).to(dtype)
    out = f(tr, th, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2], warn=False, **kw)
    assert out.dtype == torch.float32 and out.device == tr.device
    return out.cpu().numpy()


# ---- the library on the SIMT emulator ---------------------------------------------------------
@pytest.fixture(scope="module")
def F():
    from emu_backend import emulated_kernels

    with emulated_kernels():
        import b200lev.functional as F_

        yield F_


@pytest.fixture
def traced(monkeypatch):
    """Small batches take the short cross form too (the suite pins its threshold at 64 pairs), and
    the library says which form served the call."""
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    monkeypatch.setenv("B200LEV_TRACE", "1")


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("costs", COSTS)
@pytest.mark.parametrize("R", [1, 31, 32, 33, 63, 64, 65, 130])
def test_definition_vs_oracle(F, traced, capfd, R, costs, shape):
    """Bit for bit against the oracle on the materialised pairs, both functionals; unit costs with
    R <= 64 take the short cross form, everything else the gather path."""
    A, B = shape
    G = max(1, 40 // (A * B)) if R <= 64 else 2
    k = (R + len(str(costs)) + A) % len(VARIANTS)
    norm, eos, include_eos = VARIANTS[k]
    ref, hyp = _groups(R * 7 + A * B + len(str(costs)), R, R + 3, G, A, B, no_eos_frac=0.2)
    kw = dict(eos=eos, include_eos=include_eos, norm=norm)
    for mistakes in (True, False):
        exp = _expected(ref, hyp, costs, mistakes=mistakes, **kw)
        act = _call(F, ref, hyp, costs, mistakes, **kw)
        assert act.shape == (G, A, B)
        route = _route(capfd)
        _same_as_materialised(F, act, exp, ref, hyp, costs, mistakes, **kw)
        assert route == ("short" if costs == (1, 1, 1) and R <= 64 else "gather")


@pytest.mark.parametrize("norm", [True, False])
@pytest.mark.parametrize("eos", [None, 0])
@pytest.mark.parametrize("include_eos", [True, False])
@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4)])
def test_options(F, traced, capfd, norm, eos, include_eos, costs):
    ref, hyp = _groups(11, 20, 24, 3, 4, 6, no_eos_frac=0.3)
    for mistakes in (True, False):
        exp = _expected(ref, hyp, costs, eos=eos, include_eos=include_eos, norm=norm, mistakes=mistakes)
        act = _call(F, ref, hyp, costs, mistakes, eos=eos, include_eos=include_eos, norm=norm)
        assert np.array_equal(act, exp)
    assert _route(capfd) == ("short" if costs == (1, 1, 1) else "gather")


@pytest.mark.parametrize("dtype", [torch.int8, torch.int16, torch.int32, torch.long])
@pytest.mark.parametrize("R", [20, 50, 90])
def test_token_widths(F, traced, capfd, dtype, R):
    ref, hyp = _groups(R + 11, R, R - 5, 3, 4, 5, V=9)
    for costs in ((1, 1, 1), (3, 3, 4)):
        exp = _expected(ref, hyp, costs, eos=0)
        assert np.array_equal(_call(F, ref, hyp, costs, dtype=dtype, eos=0), exp)
        assert _route(capfd) == ("short" if costs == (1, 1, 1) and R <= 64 else "gather")


@pytest.mark.parametrize("R", [20, 40, 80])
@pytest.mark.parametrize("side", ["ref", "hyp", "both"])
def test_tokens_outside_int32(F, traced, capfd, R, side):
    """Tokens whose low 32 bits collide with other tokens are compared exactly on both forms (the
    gather keeps the 8-byte tokens)."""
    ref, hyp = _groups(R + len(side), R, R + 2, 2, 5, 4, V=5)
    big = np.int64(1) << 32
    if side in ("ref", "both"):
        ref = np.where(ref % 2 == 1, ref + big, ref)
    if side in ("hyp", "both"):
        hyp = np.where(hyp % 3 == 1, hyp + big * 3, hyp)
    for costs in ((1, 1, 1), (1, 2, 3)):
        assert np.array_equal(_call(F, ref, hyp, costs, eos=0), _expected(ref, hyp, costs, eos=0))
        assert _route(capfd) == ("short" if costs == (1, 1, 1) and R <= 64 else "gather")


@pytest.mark.parametrize("R", [24, 70])
def test_batch_first_and_strided(F, traced, capfd, R):
    ref, hyp = _groups(R, R, R + 4, 3, 3, 7)
    for costs in ((1, 1, 1), (1, 2, 3)):
        exp = _expected(ref, hyp, costs, eos=0)
        # batch_first: (G, A, R) and (G, B, H), contiguous -- the gather path
        rb = torch.from_numpy(np.ascontiguousarray(ref.transpose(1, 2, 0)))
        hb = torch.from_numpy(np.ascontiguousarray(hyp.transpose(1, 2, 0)))
        act = F.pairwise_error_rates(rb, hb, eos=0, batch_first=True, ins_cost=costs[0], del_cost=costs[1],
                                     sub_cost=costs[2], warn=False)
        assert np.array_equal(act.numpy(), exp)
        assert _route(capfd) == "gather"
        # views of the sequence-first tensors: every other hypothesis of a wider group, every
        # other position
        th = torch.from_numpy(np.repeat(hyp, 2, axis=2))[:, :, ::2]
        act = F.pairwise_error_rates(torch.from_numpy(ref), th, eos=0, ins_cost=costs[0], del_cost=costs[1],
                                     sub_cost=costs[2], warn=False)
        assert np.array_equal(act.numpy(), exp)
        capfd.readouterr()
        tr2 = torch.from_numpy(np.repeat(ref, 2, axis=0))[::2]
        th2 = torch.from_numpy(np.repeat(hyp, 2, axis=0))[::2]
        act = F.pairwise_error_rates(tr2, th2, eos=0, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2],
                                     warn=False)
        assert np.array_equal(act.numpy(), exp)
        assert _route(capfd) == ("short" if costs == (1, 1, 1) and R <= 64 else "gather")


def _sliced(a, k, batch_first):
    """A view of `a` (T, G, K) whose member axis is cut from a wider tensor: its group and member
    axes do not merge, so flattening it copies.  (G, K, T) with batch_first."""
    T, G, K = a.shape
    wide = np.concatenate([a, a[:, :, :k] + 1], 2)
    if batch_first:
        return torch.from_numpy(np.ascontiguousarray(wide.transpose(1, 2, 0)))[:, :K, :]
    return torch.from_numpy(wide)[:, :, :K]


@pytest.mark.parametrize("batch_first", [False, True])
@pytest.mark.parametrize("R", [20, 70])
def test_views_that_do_not_merge(F, R, batch_first):
    """Member axes sliced from wider tensors (the flattened tokens are copies): the same values as
    the contiguous call, both functionals and minimum_bayes_risk; ref and hyp of one shape, so that
    a freed copy would be reused at once."""
    ref, hyp = _groups(R + 5, R, R, 4, 6, 6)
    tr, th = _sliced(ref, 3, batch_first), _sliced(hyp, 2, batch_first)
    for costs in ((1, 1, 1), (1, 2, 3)):
        for mistakes in (True, False):
            f = F.pairwise_error_rates if mistakes else F.pairwise_edit_distances
            kw = dict(eos=0, batch_first=batch_first, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2],
                      warn=False)
            act = f(tr, th, **kw)
            assert torch.equal(act, f(tr.contiguous(), th.contiguous(), **kw))
            assert np.array_equal(act.numpy(), _expected(ref, hyp, costs, eos=0, norm=mistakes, mistakes=mistakes))
    lp = torch.from_numpy(np.random.default_rng(R).normal(size=(4, 6)))
    best, risk = F.minimum_bayes_risk(lp, th, eos=0, batch_first=batch_first, warn=False)
    cbest, crisk = F.minimum_bayes_risk(lp, th.contiguous(), eos=0, batch_first=batch_first, warn=False)
    assert torch.equal(best, cbest) and torch.equal(risk, crisk)
    _check_mbr(best, risk, _mbr_expected(lp.numpy(), hyp, eos=0), torch.float64)


@pytest.mark.parametrize("R", [30, 66])
def test_warnings(F, R):
    """The three warnings fire exactly where error_rate on the materialised pairs fires them."""
    ref, hyp = _groups(R + 1, R, R, 3, 3, 4, no_eos_frac=0.5)
    ref[0, 1, :2] = 0  # empty references
    refx, hypx = _materialise(ref, hyp)

    def msgs(f, *args, **kw):
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            out = f(*args, **kw)
        return out, sorted(str(x.message) for x in w)

    for include_eos in (True, False):
        for norm in (True, False):
            for costs in ((1, 1, 1), (1, 2, 3)):
                kw = dict(eos=0, include_eos=include_eos, norm=norm, ins_cost=costs[0], del_cost=costs[1],
                          sub_cost=costs[2])
                exp, exp_w = msgs(F.error_rate, torch.from_numpy(refx), torch.from_numpy(hypx), **kw)
                act, act_w = msgs(F.pairwise_error_rates, torch.from_numpy(ref), torch.from_numpy(hyp), **kw)
                assert np.array_equal(act.numpy().reshape(-1), exp.numpy()) and act_w == exp_w
                exp, exp_w = msgs(F.edit_distance, torch.from_numpy(refx), torch.from_numpy(hypx), **kw)
                act, act_w = msgs(F.pairwise_edit_distances, torch.from_numpy(ref), torch.from_numpy(hyp), **kw)
                assert np.array_equal(act.numpy().reshape(-1), exp.numpy()) and act_w == exp_w
                _, w = msgs(F.pairwise_error_rates, torch.from_numpy(ref), torch.from_numpy(hyp), warn=False, **kw)
                assert not w


@pytest.mark.parametrize("R", [10, 80])
def test_empty_sequences_and_sizes(F, R):
    ref, hyp = _groups(R + 3, R, R, 4, 3, 5)
    ref[0, :, 0] = 0  # empty references
    hyp[0, :, 1] = 0  # empty hypotheses
    ref[0, 1, :] = hyp[0, 1, :] = 0  # both, a whole group
    for costs in ((1, 1, 1), (1, 2, 3)):
        for norm in (True, False):
            exp = _expected(ref, hyp, costs, eos=0, norm=norm)
            assert np.array_equal(_call(F, ref, hyp, costs, eos=0, norm=norm), exp)
    # zero-length sequences
    for Rz, Hz in ((0, 5), (5, 0), (0, 0)):
        r0, h0 = np.zeros((Rz, 2, 3), np.int64) + 2, np.zeros((Hz, 2, 4), np.int64) + 3
        got = F.pairwise_edit_distances(torch.from_numpy(r0), torch.from_numpy(h0))
        assert got.shape == (2, 3, 4) and (got == max(Rz, Hz)).all()
    # empty G, A or B: an empty output
    for G, A, B in ((0, 3, 4), (2, 0, 4), (2, 3, 0)):
        got = F.pairwise_error_rates(torch.ones(6, G, A, dtype=torch.long), torch.ones(7, G, B, dtype=torch.long))
        assert got.shape == (G, A, B) and got.dtype == torch.float32
        got = F.pairwise_error_rates(torch.ones(G, A, 6, dtype=torch.long), torch.ones(G, B, 7, dtype=torch.long),
                                     batch_first=True)
        assert got.shape == (G, A, B)


def test_shape_errors(F):
    z = torch.zeros
    with pytest.raises(RuntimeError, match="ref and hyp must be 3 dimensional"):
        F.pairwise_error_rates(z(3, 2, dtype=torch.long), z(3, 2, 2, dtype=torch.long))
    with pytest.raises(RuntimeError, match="ref and hyp must be 3 dimensional"):
        F.pairwise_edit_distances(z(3, 2, 2, dtype=torch.long), z(3, 2, 2, 1, dtype=torch.long))
    with pytest.raises(RuntimeError, match="ref and hyp group dimensions must match"):
        F.pairwise_error_rates(z(3, 2, 2, dtype=torch.long), z(3, 3, 2, dtype=torch.long))
    with pytest.raises(RuntimeError, match="ref and hyp group dimensions must match"):
        F.pairwise_error_rates(z(2, 2, 3, dtype=torch.long), z(3, 2, 3, dtype=torch.long), batch_first=True)
    with pytest.raises(RuntimeError, match="log_probs must be 2 dimensional"):
        F.minimum_bayes_risk(z(3), z(4, 3, 2, dtype=torch.long))
    with pytest.raises(RuntimeError, match="hyp must be 3 dimensional"):
        F.minimum_bayes_risk(z(3, 2), z(4, 6, dtype=torch.long))
    with pytest.raises(RuntimeError, match="ref and hyp batch_size and sample dimensions must match"):
        F.minimum_bayes_risk(z(3, 2), z(4, 3, 3, dtype=torch.long))
    with pytest.raises(RuntimeError, match="ref and hyp batch_size and sample dimensions must match"):
        F.minimum_bayes_risk(z(3, 2), z(3, 2, 4, dtype=torch.long))  # batch_first=False: (H, N, M)


# ---- minimum_bayes_risk -----------------------------------------------------------------------
TOL = {torch.float32: 1e-5, torch.float64: 1e-12, torch.float16: 2e-3, torch.bfloat16: 1.6e-2}


def _mbr_expected(lp, hyp, eos=None, include_eos=True, norm=True, costs=(1, 1, 1)):
    """float64 restatement: softmax of each row, risk = p @ er (er[n, a, i]: hypothesis i scored
    against hypothesis a as the reference)."""
    er = _expected(hyp, hyp, costs, eos=eos, include_eos=include_eos, norm=norm, mistakes=norm).astype(np.float64)
    lp = lp.astype(np.float64)
    with np.errstate(invalid="ignore"):
        p = np.exp(lp - lp.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    return np.einsum("na,nai->ni", p, er)


def _check_mbr(best, risk, exp, dtype):
    tol = TOL[dtype]
    assert best.dtype == torch.long and risk.dtype == dtype
    r = risk.double().cpu().numpy()
    np.testing.assert_allclose(r, exp, rtol=tol, atol=tol)
    b = best.cpu().numpy()
    # best is the arg min of the returned risk, lowest index on ties
    assert np.array_equal(b, r.argmin(1))
    # and the float64 arg min wherever the runner-up is further away than the tolerance
    srt = np.sort(exp, 1)
    clear = (srt[:, 1] - srt[:, 0] > 4 * tol * np.maximum(1.0, np.abs(srt[:, 0]))) if exp.shape[1] > 1 else \
        np.ones(len(exp), bool)
    assert np.array_equal(b[clear], exp.argmin(1)[clear])
    return clear


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16, torch.float64])
@pytest.mark.parametrize("M", [1, 3, 16, 40])
def test_mbr_vs_float64(F, dtype, M):
    rng = np.random.default_rng(M)
    N = 12
    hyp = PC.random_tokens(rng, 18, N * M, 6, 0, -2, 3).reshape(18, N, M)
    lp = torch.from_numpy(rng.normal(size=(N, M)) * 2).to(dtype)
    best, risk = F.minimum_bayes_risk(lp, torch.from_numpy(hyp), eos=0, warn=False)
    exp = _mbr_expected(lp.double().numpy(), hyp, eos=0)
    clear = _check_mbr(best, risk, exp, dtype)
    assert clear.mean() > (0.5 if dtype in (torch.float32, torch.float64) else 0.2)
    if M == 1:
        assert (risk == 0).all() and (best == 0).all()


@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4)])
@pytest.mark.parametrize("norm", [True, False])
def test_mbr_options_and_batch_first(F, costs, norm):
    rng = np.random.default_rng(3)
    N, M, H = 9, 6, 25
    hyp = PC.random_tokens(rng, H, N * M, 5, 0, -2, 3).reshape(H, N, M)
    lp = torch.from_numpy(rng.normal(size=(N, M)))
    kw = dict(eos=0, include_eos=False, norm=norm, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
    exp = _mbr_expected(lp.numpy(), hyp, eos=0, include_eos=False, norm=norm, costs=costs)
    best, risk = F.minimum_bayes_risk(lp, torch.from_numpy(hyp), warn=False, **kw)
    _check_mbr(best, risk, exp, torch.float64)
    hb = torch.from_numpy(np.ascontiguousarray(hyp.transpose(1, 2, 0)))
    best2, risk2 = F.minimum_bayes_risk(lp, hb, batch_first=True, warn=False, **kw)
    assert torch.equal(best2, best) and torch.equal(risk2, risk)
    # a strided log_probs view
    wide = torch.zeros(N, 2 * M, dtype=lp.dtype)
    wide[:, ::2] = lp
    best3, risk3 = F.minimum_bayes_risk(wide[:, ::2], torch.from_numpy(hyp), warn=False, **kw)
    assert torch.equal(best3, best) and torch.equal(risk3, risk)


def test_mbr_ties_and_zero_weights(F):
    rng = np.random.default_rng(5)
    N, M, H = 10, 7, 15
    hyp = PC.random_tokens(rng, H, N * M, 6, 0, -2, 3).reshape(H, N, M)
    hyp[:, :, 4] = hyp[:, :, 1]  # duplicates: bitwise identical risks
    hyp[:, :, 6] = hyp[:, :, 1]
    lp = rng.normal(size=(N, M))
    lp[:, 2] = -np.inf  # zero weight
    lp[0, :] = 0.0  # uniform weights
    hyp[:, 0, :] = hyp[:, 0, :1]  # every hypothesis of group 0 the same: all risks 0, best 0
    for dtype in (torch.float32, torch.float16, torch.float64):
        best, risk = F.minimum_bayes_risk(torch.from_numpy(lp).to(dtype), torch.from_numpy(hyp), eos=0, warn=False)
        r = risk.double().numpy()
        assert np.array_equal(r[:, 4], r[:, 1]) and np.array_equal(r[:, 6], r[:, 1])
        assert best[0] == 0 and (risk[0] == 0).all()
        b = best.numpy()
        assert not np.isin(b, [4, 6]).any()  # a tie goes to the lowest index
        exp = _mbr_expected(lp, hyp, eos=0)
        _check_mbr(best, risk, exp, dtype)
        # the -inf hypothesis carries no weight: dropping it changes nothing
        keep = [0, 1, 3, 4, 5, 6]
        er = _expected(hyp, hyp, eos=0, include_eos=True).astype(np.float64)
        p = np.exp(lp[:, keep] - lp[:, keep].max(1, keepdims=True))
        p /= p.sum(1, keepdims=True)
        np.testing.assert_allclose(r, np.einsum("na,nai->ni", p, er[:, keep, :]), rtol=TOL[dtype], atol=TOL[dtype])


def test_mbr_empty(F):
    best, risk = F.minimum_bayes_risk(torch.zeros(0, 4), torch.zeros(5, 0, 4, dtype=torch.long))
    assert best.shape == (0,) and risk.shape == (0, 4)


def test_modules_script_and_trace(F):
    import b200lev.modules as M

    ref, hyp = _groups(3, 20, 22, 3, 2, 4)
    mod = M.PairwiseErrorRates(eos=0, ins_cost=1.0, del_cost=2.0, sub_cost=3.0, warn=False)
    exp = _expected(ref, hyp, (1, 2, 3), eos=0)
    tr, th = torch.from_numpy(ref), torch.from_numpy(hyp)
    assert np.array_equal(mod(tr, th).numpy(), exp)
    assert np.array_equal(torch.jit.script(mod)(tr, th).numpy(), exp)
    traced = torch.jit.trace(mod, (tr, th))
    ref2, hyp2 = _groups(4, 70, 40, 2, 5, 3)  # other shapes than the example
    exp2 = _expected(ref2, hyp2, (1, 2, 3), eos=0)
    assert np.array_equal(traced(torch.from_numpy(ref2), torch.from_numpy(hyp2)).numpy(), exp2)
    assert "eos=0" in repr(mod)

    mod = M.PairwiseEditDistances(eos=0)
    exp = _expected(ref, hyp, eos=0, norm=False, mistakes=False)
    assert np.array_equal(torch.jit.script(mod)(tr, th).numpy(), exp)
    traced = torch.jit.trace(mod, (tr, th))
    assert np.array_equal(traced(torch.from_numpy(ref2), torch.from_numpy(hyp2)).numpy(),
                          _expected(ref2, hyp2, eos=0, norm=False, mistakes=False))

    mod = M.MinimumBayesRisk(eos=0, warn=False)
    rng = np.random.default_rng(0)
    lp = torch.from_numpy(rng.normal(size=(3, 4))).float()
    h = torch.from_numpy(PC.random_tokens(rng, 12, 12, 5, 0, -2, 2).reshape(12, 3, 4))
    best, risk = mod(lp, h)
    sbest, srisk = torch.jit.script(mod)(lp, h)
    assert torch.equal(best, sbest) and torch.equal(risk, srisk)
    traced = torch.jit.trace(mod, (lp, h))
    lp2 = torch.from_numpy(rng.normal(size=(5, 6))).float()
    h2 = torch.from_numpy(PC.random_tokens(rng, 20, 30, 5, 0, -2, 2).reshape(20, 5, 6))
    tb, tr_ = traced(lp2, h2)
    _check_mbr(tb, tr_, _mbr_expected(lp2.double().numpy(), h2.numpy(), eos=0), torch.float32)
    assert tb.shape == (5,)
    with pytest.raises(ValueError):
        M.MinimumBayesRisk(norm="yes")


def test_registered_ops_have_fakes(F):
    """One registered op per functional, with a fake: the shapes depend on the input shapes only."""
    from torch._subclasses.fake_tensor import FakeTensorMode

    with FakeTensorMode():
        out, flags = torch.ops.b200lev.pairwise(torch.empty(9, 4, 3, dtype=torch.long),
                                                torch.empty(7, 4, 5, dtype=torch.long), 0, False, False,
                                                1.0, 1.0, 1.0, True, True)
        assert out.shape == (4, 3, 5) and out.dtype == torch.float32 and flags.shape == (1,)
        best, risk, flags = torch.ops.b200lev.minimum_bayes_risk(
            torch.empty(4, 6, dtype=torch.float16), torch.empty(4, 6, 11, dtype=torch.long), 0, True, True,
            True, 1.0, 1.0, 1.0)
        assert best.shape == (4,) and best.dtype == torch.long
        assert risk.shape == (4, 6) and risk.dtype == torch.float16


# ---- C entry point statuses -------------------------------------------------------------------
@pytest.fixture(scope="module")
def abi():
    from emu_backend import emulated_kernels

    with emulated_kernels():
        from b200lev import _abi

        yield _abi


def _tokens(abi, T, N, seed):
    a = np.random.default_rng(seed).integers(1, 5, (T, N)).astype(np.int64)
    t = abi.Tokens(a.ctypes.data if a.size else None, 8, T, N, N, 1)
    t.keep = a
    return t


def _cross(abi, ref, hyp, A, B, costs=(1.0, 1.0, 1.0), ref_group=1, out="buf", ws="buf", ws_short=0):
    L = abi.lib()
    o = abi.Opts(1, 0, 0, *costs, 0, 0, -1, 1, ref_group)
    nbytes = L.b200lev_final_cross_workspace_bytes(ctypes.byref(ref), ctypes.byref(hyp), A, B, ctypes.byref(o))
    P = max(int(ref.N) * max(B, 0), 1)
    ws = np.zeros(max(nbytes, 1), np.uint8) if ws == "buf" else ws
    out = np.full(P, -7, np.float32) if out == "buf" else out
    flags = np.zeros(1, np.int32)
    rc = L.b200lev_final_cross(ctypes.byref(ref), ctypes.byref(hyp), A, B, ctypes.byref(o),
                               None if out is None else out.ctypes.data, None if ws is None else ws.ctypes.data,
                               nbytes - ws_short, flags.ctypes.data, 0)
    return rc, out, nbytes


def test_abi_statuses(abi, monkeypatch):
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    OK, ERR_ARG, ERR_WORKSPACE = 0, -1, -3
    ref, hyp = _tokens(abi, 6, 6, 0), _tokens(abi, 5, 8, 1)  # G = 2, A = 3, B = 4
    for costs in ((1.0, 1.0, 1.0), (1.0, 2.0, 3.0)):
        rc, out, nbytes = _cross(abi, ref, hyp, 3, 4, costs)
        assert rc == OK and (out >= 0).all()
        assert _cross(abi, ref, hyp, 3, 4, costs, ws_short=1)[0] == ERR_WORKSPACE
        assert _cross(abi, ref, hyp, 3, 4, costs, out=None)[0] == ERR_ARG
        assert _cross(abi, ref, hyp, 3, 4, costs, ws=None)[0] == ERR_ARG
    # the short cross form needs no gather buffer: the workspace is what b200lev_final needs for the
    # expanded pairs (ref_group = B); the gather path adds the gathered hypotheses
    L = abi.lib()
    hypx = _tokens(abi, 5, 24, 1)
    final_bytes = L.b200lev_workspace_bytes(ctypes.byref(ref), ctypes.byref(hypx), 0, 0)
    assert _cross(abi, ref, hyp, 3, 4)[2] == final_bytes
    gathered = -(-5 * 24 * 8 // 128) * 128
    assert _cross(abi, ref, hyp, 3, 4, (1.0, 2.0, 3.0))[2] == final_bytes + gathered + 128
    assert _cross(abi, ref, hyp, -1, 4)[0] == ERR_ARG
    assert _cross(abi, ref, hyp, 3, -4)[0] == ERR_ARG
    assert _cross(abi, ref, hyp, 4, 4)[0] == ERR_ARG  # ref->N != G*A
    assert _cross(abi, ref, hyp, 3, 3)[0] == ERR_ARG  # hyp->N != G*B
    assert _cross(abi, ref, _tokens(abi, 5, 9, 1), 3, 4)[0] == ERR_ARG
    big = _tokens(abi, 1, 1 << 16, 2)  # G = 1, A = B = 65 536: 2^32 pairs
    assert _cross(abi, big, big, 1 << 16, 1 << 16, out=None, ws=None)[0] == ERR_ARG
    assert b"2^31" in abi.lib().b200lev_last_error()
    assert _cross(abi, ref, hyp, 3, 4, ref_group=2)[0] == ERR_ARG
    assert b"ref_group" in abi.lib().b200lev_last_error()
    # no pairs: nothing to write, NULL buffers are fine
    assert _cross(abi, _tokens(abi, 6, 0, 0), _tokens(abi, 5, 0, 1), 3, 4, out=None, ws=None)[0] == OK
    assert _cross(abi, ref, _tokens(abi, 5, 0, 1), 3, 0, out=None, ws=None)[0] == OK
    # the MBR epilogue
    er = np.zeros(2 * 3 * 3, np.float32)
    lp = np.zeros((2, 3), np.float32)
    risk = np.zeros((2, 3), np.float32)
    best = np.zeros(2, np.int64)
    mbr = L.b200lev_mbr
    assert mbr(er.ctypes.data, lp.ctypes.data, 0, 2, 3, 3, 1, risk.ctypes.data, best.ctypes.data, 0) == OK
    assert mbr(er.ctypes.data, lp.ctypes.data, 0, 2, 0, 3, 1, risk.ctypes.data, best.ctypes.data, 0) == ERR_ARG
    assert mbr(er.ctypes.data, lp.ctypes.data, 0, -1, 3, 3, 1, risk.ctypes.data, best.ctypes.data, 0) == ERR_ARG
    assert mbr(er.ctypes.data, lp.ctypes.data, 7, 2, 3, 3, 1, risk.ctypes.data, best.ctypes.data, 0) == ERR_ARG
    assert mbr(None, lp.ctypes.data, 0, 2, 3, 3, 1, risk.ctypes.data, best.ctypes.data, 0) == ERR_ARG
    assert mbr(None, None, 0, 0, 3, 3, 1, None, None, 0) == OK


# ---- the device ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def FG():
    import b200lev.functional as F_

    return F_


def _nbest_words(G, M, T, V=10_000, seed=0):
    """N-best lists of word sequences: G groups of M hypotheses of up to T - 1 words, eos -1;
    the hypotheses of a group are edits of one another."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, V, (T, G, 1))
    hyp = np.where(rng.random((T, G, M)) < 0.15, rng.integers(0, V, (T, G, M)), base)
    lens = rng.integers(T // 3, T, (G, M))
    pos = np.arange(T)[:, None, None]
    hyp = np.where(pos < lens, hyp, -1)
    return hyp


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["a", "b", "c"])
def test_gpu_full_size_vs_materialised(FG, shape, monkeypatch, capfd):
    """The shapes of scripts/bench_pairwise.py at full size, bit for bit against error_rate on the
    materialised pairs (the route as the trace says)."""
    dev = torch.device("cuda")
    G, M, T, costs = {"a": (4096, 16, 31, (1, 1, 1)), "b": (16384, 8, 100, (1, 1, 1)),
                      "c": (4096, 16, 31, (3, 3, 4))}[shape]
    h = torch.from_numpy(_nbest_words(G, M, T)).to(dev)
    kw = dict(eos=-1, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2], warn=False)
    monkeypatch.setenv("B200LEV_TRACE", "1")
    act = FG.pairwise_error_rates(h, h, **kw)
    torch.cuda.synchronize()
    assert _route(capfd) == ("short" if shape == "a" else "gather")
    monkeypatch.delenv("B200LEV_TRACE")
    idx = torch.arange(G * M * M, device=dev)
    g, a, b = idx // (M * M), idx // M % M, idx % M
    flat = h.reshape(T, G * M)
    exp = FG.error_rate(flat.index_select(1, g * M + a), flat.index_select(1, g * M + b), **kw)
    assert torch.equal(act.reshape(-1), exp)
    ed = FG.pairwise_edit_distances(h, h, **kw)
    assert torch.equal(ed.reshape(-1), FG.edit_distance(flat.index_select(1, g * M + a),
                                                        flat.index_select(1, g * M + b), **kw))


@pytest.mark.gpu
def test_gpu_mbr_vs_torch_composition(FG):
    dev = torch.device("cuda")
    G, M, T = 4096, 16, 31
    h = torch.from_numpy(_nbest_words(G, M, T, seed=1)).to(dev)
    lp = torch.randn(G, M, device=dev, dtype=torch.float64).log_softmax(1)
    for dtype in (torch.float32, torch.float64):
        best, risk = FG.minimum_bayes_risk(lp.to(dtype), h, eos=-1, warn=False)
        er = FG.pairwise_error_rates(h, h, eos=-1, include_eos=True, warn=False)
        exp = torch.einsum("na,nai->ni", lp.softmax(1), er.double())
        tol = TOL[dtype]
        torch.testing.assert_close(risk.double(), exp, rtol=tol, atol=tol)
        assert torch.equal(best, risk.argmin(1))
        srt = exp.sort(1).values
        clear = srt[:, 1] - srt[:, 0] > 4 * tol
        assert clear.float().mean() > 0.5
        assert torch.equal(best[clear], exp.argmin(1)[clear])


@pytest.mark.gpu
@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4)])
def test_gpu_cuda_graph_replay(FG, costs):
    dev = torch.device("cuda")
    h = torch.from_numpy(_nbest_words(512, 8, 31, seed=2)).to(dev)
    lp = torch.randn(512, 8, device=dev)
    kw = dict(eos=-1, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2], warn=False)
    eager = FG.pairwise_error_rates(h, h, **kw)
    eb, er = FG.minimum_bayes_risk(lp, h, **kw)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        FG.pairwise_error_rates(h, h, **kw)
        FG.minimum_bayes_risk(lp, h, **kw)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = FG.pairwise_error_rates(h, h, **kw)
        best, risk = FG.minimum_bayes_risk(lp, h, **kw)
    out.fill_(-1)
    best.fill_(-1)
    risk.fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager) and torch.equal(best, eb) and torch.equal(risk, er)


@pytest.mark.gpu
@pytest.mark.parametrize("batch_first", [False, True])
def test_gpu_views_that_do_not_merge(FG, batch_first):
    """As test_views_that_do_not_merge, on the device (the caching allocator hands a freed block out
    again at once)."""
    dev = torch.device("cuda")
    ref, hyp = _groups(7, 30, 30, 64, 8, 8)
    tr, th = _sliced(ref, 3, batch_first).to(dev), _sliced(hyp, 2, batch_first).to(dev)
    for costs in ((1, 1, 1), (1, 2, 3)):
        kw = dict(eos=0, batch_first=batch_first, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2],
                  warn=False)
        act = FG.pairwise_error_rates(tr, th, **kw)
        assert torch.equal(act, FG.pairwise_error_rates(tr.contiguous(), th.contiguous(), **kw))
        assert np.array_equal(act.cpu().numpy(), _expected(ref, hyp, costs, eos=0))
    lp = torch.randn(64, 8, device=dev)
    best, risk = FG.minimum_bayes_risk(lp, th, eos=0, batch_first=batch_first, warn=False)
    cbest, crisk = FG.minimum_bayes_risk(lp, th.contiguous(), eos=0, batch_first=batch_first, warn=False)
    assert torch.equal(best, cbest) and torch.equal(risk, crisk)


@pytest.mark.gpu
def test_gpu_host_tensors_in_and_out(FG):
    ref, hyp = _groups(12, 40, 45, 50, 3, 4)
    for costs in ((1, 1, 1), (3, 3, 4)):
        exp = _expected(ref, hyp, costs, eos=0)
        act = FG.pairwise_error_rates(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, ins_cost=costs[0],
                                      del_cost=costs[1], sub_cost=costs[2], warn=False)
        assert act.device.type == "cpu" and np.array_equal(act.numpy(), exp)
    rng = np.random.default_rng(0)
    lp = torch.from_numpy(rng.normal(size=(50, 4)))
    best, risk = FG.minimum_bayes_risk(lp, torch.from_numpy(hyp), eos=0, warn=False)
    assert best.device.type == "cpu" and risk.device.type == "cpu"
    _check_mbr(best, risk, _mbr_expected(lp.numpy(), hyp, eos=0), torch.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("costs", COSTS)
@pytest.mark.parametrize("R", [31, 64, 100])
def test_gpu_definition_vs_oracle(FG, R, costs, monkeypatch):
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    ref, hyp = _groups(R + len(str(costs)), R, R + 3, 97, 5, 13, no_eos_frac=0.2)
    for mistakes in (True, False):
        exp = _expected(ref, hyp, costs, eos=0, norm=mistakes, mistakes=mistakes)
        act = _call(FG, ref, hyp, costs, mistakes, dev=torch.device("cuda"), eos=0, norm=mistakes)
        _same_as_materialised(FG, act, exp, ref, hyp, costs, mistakes, dev=torch.device("cuda"), eos=0,
                              norm=mistakes)
