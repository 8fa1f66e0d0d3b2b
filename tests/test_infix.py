"""infix_edit_distance / infix_matches: the cheapest match of each reference anywhere inside its
hypothesis, and where it lies.

The CPU restatement (tests/infix_oracle.py) is pinned to the reference's edit_distance (the C oracle)
through identities that define the feature independently of the kernels: the distance is the
minimum of edit_distance(ref, hyp[s:e]) over every stretch, bit for bit; the match it reports
rescores to that distance; and for integer and dyadic costs the end is the first position reaching
it and the start the last one for that end.  The library is then compared with the restatement bit
for bit, on the SIMT emulator (tests/emu) and on the device.
"""
import ctypes
import os
import sys
import warnings

import numpy as np
import pytest
import torch

import counts_oracle as CO
import infix_oracle as IO
import parity_cases as PC
from oracle import oracle as O
from test_error_counts import COSTS

ALL_COSTS = COSTS + [(0.3, 0.3, 0.3)]


def _dyadic(costs):
    return all(float(c) * 8 == round(float(c) * 8) for c in costs)


def _stretches(ref, hyp, r, h, costs):
    """edit_distance of every reference against every stretch hyp[s:e] of its hypothesis, one C
    oracle call: a list per pair of ((s, e), value)."""
    N = ref.shape[1]
    pad = min(ref.min(initial=0), hyp.min(initial=0)) - 1  # an eos no token equals
    owner, se = [], []
    for n in range(N):
        for s in range(h[n] + 1):
            for e in range(s, h[n] + 1):
                owner.append(n)
                se.append((s, e))
    M = len(owner)
    refs = np.full((int(r.max(initial=0)) + 1, M), pad, np.int64)
    hyps = np.full((int(h.max(initial=0)) + 1, M), pad, np.int64)
    for k, (n, (s, e)) in enumerate(zip(owner, se)):
        refs[:r[n], k] = ref[:r[n], n]
        hyps[:e - s, k] = hyp[s:e, n]
    ed = O.edit_distance(refs, hyps, eos=int(pad), include_eos=False, norm=False, ins_cost=costs[0],
                         del_cost=costs[1], sub_cost=costs[2])
    out = [[] for _ in range(N)]
    for k, n in enumerate(owner):
        out[n].append((se[k], np.float32(ed[k])))
    return out


def _check_identities(ref, hyp, costs, eos=None, include_eos=False):
    """The oracle against the reference's edit_distance on every stretch."""
    dist, start, end = IO.infix(ref, hyp, eos=eos, include_eos=include_eos, ins_cost=costs[0],
                                del_cost=costs[1], sub_cost=costs[2])
    r, _ = CO._lengths(ref, eos, include_eos)
    h, _ = CO._lengths(hyp, eos, include_eos)
    for n, cand in enumerate(_stretches(ref, hyp, r, h, costs)):
        vals = {k: v for k, v in cand}
        m = min(v for _, v in cand)
        assert 0 <= start[n] <= end[n] <= h[n]
        if not _dyadic(costs):
            # The reference takes the fp32 deletion term as min_k v[k] + (fl(j*d) - fl(k*d)), the
            # library (and this restatement) by run origin; for costs such as (0.7, 1.1, 1.3) the
            # two can differ in the last bit (DESIGN 9i), so only closeness is asserted here
            assert np.isclose(dist[n], m, rtol=1e-6, atol=0), (n, dist[n], m)
            assert np.isclose(vals[(start[n], end[n])], dist[n], rtol=1e-6, atol=0), n
            continue
        assert dist[n].tobytes() == m.tobytes(), (n, dist[n], m)
        assert vals[(start[n], end[n])].tobytes() == dist[n].tobytes(), n
        e_min = min(e for (s, e), v in cand if v == m)
        s_max = max(s for (s, e), v in cand if v == m and e == e_min)
        assert (start[n], end[n]) == (s_max, e_min), n


# ---- the CPU restatement against the reference -------------------------------------------
@pytest.mark.parametrize("costs", ALL_COSTS)
def test_oracle_every_stretch(costs):
    rng = np.random.default_rng(len(str(costs)))
    for R, H in ((1, 12), (3, 9), (6, 12), (12, 4), (5, 0)):
        ref = PC.random_tokens(rng, R, 24, 4, 0, -2, 0, 0.1)
        hyp = PC.random_tokens(rng, H, 24, 4, 0, -3, 0, 0.1) if H else np.zeros((0, 24), np.int64)
        _check_identities(ref, hyp, costs, eos=0)
        _check_identities(ref, hyp, costs, eos=0, include_eos=True)


@pytest.mark.parametrize("costs", ALL_COSTS)
def test_oracle_golden_pairs(golden_sm, costs):
    n = 0
    for case, p in golden_sm.params.items():
        ref, hyp = golden_sm.get(case, "ref"), golden_sm.get(case, "hyp")
        if p["batch_first"]:
            ref, hyp = ref.T, hyp.T
        if ref.shape[1] != hyp.shape[1]:
            continue
        _check_identities(ref, hyp, costs, eos=p["eos"], include_eos=p["include_eos"])
        n += 1
    assert n >= 60


def test_oracle_planted_twice():
    rng = np.random.default_rng(0)
    for costs in ALL_COSTS:
        ref = rng.integers(10, 20, (9, 5))
        hyp = rng.integers(1, 8, (60, 5))
        hyp[7:16] = ref
        hyp[40:49] = ref
        dist, start, end = IO.infix(ref, hyp, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
        assert (dist == 0).all() and (start == 7).all() and (end == 16).all()


# ---- the library on the SIMT emulator ---------------------------------------------------------
@pytest.fixture(scope="module")
def F():
    from emu_backend import emulated_kernels

    with emulated_kernels():
        import b200lev.functional as F_

        yield F_


def _batch(seed, R, H, N, V=6, eos=0, no_eos_frac=0.0, min_frac=0.3):
    rng = np.random.default_rng(seed)
    ref = PC.random_tokens(rng, R, N, V, eos, -2, int(R * min_frac), no_eos_frac)
    hyp = PC.random_tokens(rng, H, N, V, eos, -3, int(H * min_frac), no_eos_frac)
    return ref, hyp


def _route(F, capfd, fn):
    """Runs fn with B200LEV_TRACE set; returns (result, the infix trace line)."""
    os.environ["B200LEV_TRACE"] = "1"
    try:
        capfd.readouterr()
        out = fn()
    finally:
        del os.environ["B200LEV_TRACE"]
    lines = [ln for ln in capfd.readouterr().err.splitlines() if "b200lev: infix" in ln]
    return out, lines


def _vs_oracle(F, dev, ref, hyp, costs=(1, 1, 1), dtype=torch.long, hdtype=None, norm=False, **kw):
    """Both functionals against the oracle, bit for bit."""
    c = dict(ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
    exp = IO.infix(ref, hyp, **c, **kw)
    tr = torch.from_numpy(ref).to(dev).to(dtype)
    th = torch.from_numpy(hyp).to(dev).to(hdtype or dtype)
    d, s, e = F.infix_matches(tr, th, warn=False, **c, **kw)
    assert d.dtype == torch.float32 and s.dtype == torch.long and e.dtype == torch.long
    assert d.device == tr.device
    assert np.array_equal(d.cpu().numpy().view(np.int32), exp[0].view(np.int32))
    assert np.array_equal(s.cpu().numpy(), exp[1]) and np.array_equal(e.cpu().numpy(), exp[2])
    dn = F.infix_edit_distance(tr, th, warn=False, norm=norm, **c, **kw)
    expn = IO.infix(ref, hyp, norm=norm, **c, **kw)[0]
    assert np.array_equal(dn.cpu().numpy().view(np.int32), expn.view(np.int32))
    return exp


def _short_expected(R, costs, same_width=True):
    uniform = costs[0] == costs[1] == costs[2] and costs[0] > 0
    return R <= 64 and R >= 1 and uniform and same_width


@pytest.mark.parametrize("costs", ALL_COSTS)
@pytest.mark.parametrize("R", [1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257])
def test_random_vs_oracle(F, capfd, monkeypatch, R, costs):
    """Ks's infix kind (distance only, unit costs, R <= 64) and K1 with and without the start
    channel, across its strip widths (32 * C columns for C = 1, 2, 4, 8; several strips past 256)."""
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    N = 34 if R <= 65 else 3
    ref, hyp = _batch(R * 7 + len(str(costs)), R, R + 5, N, no_eos_frac=0.2)
    # some hypotheses hold their reference inside noise
    for n in range(0, N, 3):
        hyp[3:3 + R // 2, n] = np.where(ref[:R // 2, n] == 0, 1, ref[:R // 2, n])
    _, lines = _route(F, capfd, lambda: _vs_oracle(F, torch.device("cpu"), ref, hyp, costs, eos=0))
    assert len(lines) == 2
    assert "spans" in lines[0] and "lev_warp_kernel" in lines[0]
    assert ("lev_bv_short_kernel (infix kind)" in lines[1]) == _short_expected(R, costs), lines[1]


@pytest.mark.parametrize("dtype", [torch.int8, torch.int16, torch.int32, torch.long])
@pytest.mark.parametrize("R", [20, 50, 90])
def test_token_widths(F, capfd, monkeypatch, dtype, R):
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    ref, hyp = _batch(R + 11, R, R + 9, 33, V=9)
    for costs in ((1, 1, 1), (3, 3, 4)):
        _, lines = _route(F, capfd, lambda: _vs_oracle(F, torch.device("cpu"), ref, hyp, costs, dtype=dtype, eos=0))
        assert ("infix kind" in lines[1]) == _short_expected(R, costs)


@pytest.mark.parametrize("R", [20, 40, 80])
@pytest.mark.parametrize("side", ["ref", "hyp", "both"])
def test_tokens_outside_int32(F, R, side):
    """Tokens whose low 32 bits collide with other tokens: exact compares on every form."""
    ref, hyp = _batch(R + len(side), R, R + 6, 35, V=5)
    big = np.int64(1) << 32
    if side in ("ref", "both"):
        ref = np.where(ref % 2 == 1, ref + big, ref)
    if side in ("hyp", "both"):
        hyp = np.where(hyp % 3 == 1, hyp + big * 3, hyp)
    for costs in ((1, 1, 1), (1, 2, 3), (0.7, 1.1, 1.3)):
        _vs_oracle(F, torch.device("cpu"), ref, hyp, costs, eos=0)


def test_mixed_token_widths(F, capfd, monkeypatch):
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    ref, hyp = _batch(5, 30, 36, 33)
    _, lines = _route(F, capfd, lambda: _vs_oracle(F, torch.device("cpu"), ref, hyp, dtype=torch.int32,
                                                   hdtype=torch.long, eos=0))
    assert "infix kind" not in lines[1]  # Ks reads one token width


@pytest.mark.parametrize("R", [24, 70])
def test_batch_first_strided_and_eos_none(F, monkeypatch, R):
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    cpu = torch.device("cpu")
    ref, hyp = _batch(R, R, R + 8, 34)
    exp = IO.infix(ref, hyp, eos=0, ins_cost=1, del_cost=2, sub_cost=3)
    rb, hb = np.ascontiguousarray(ref.T), np.ascontiguousarray(hyp.T)
    got = _vs_oracle(F, cpu, rb, hb, (1, 2, 3), eos=0, batch_first=True)
    assert all(np.array_equal(a, b) for a, b in zip(got, exp))
    # strided views: every other pair of a wider batch, every other row
    big_r, big_h = np.repeat(ref, 2, axis=1), np.repeat(hyp, 2, axis=1)
    for costs in ((1, 2, 3), (1, 1, 1)):
        e = IO.infix(ref, hyp, eos=0, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
        for tr, th in ((torch.from_numpy(big_r)[:, ::2], torch.from_numpy(big_h)[:, ::2]),
                       (torch.from_numpy(np.repeat(ref, 2, axis=0))[::2],
                        torch.from_numpy(np.repeat(hyp, 2, axis=0))[::2])):
            d, s, en = F.infix_matches(tr, th, eos=0, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2],
                                       warn=False)
            assert np.array_equal(d.numpy(), e[0]) and np.array_equal(s.numpy(), e[1])
            assert np.array_equal(en.numpy(), e[2])
            d = F.infix_edit_distance(tr, th, eos=0, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2],
                                      warn=False)
            assert np.array_equal(d.numpy(), e[0])
    # no eos: the full padded lengths
    _vs_oracle(F, cpu, ref, hyp, (3, 3, 4))
    _vs_oracle(F, cpu, ref, hyp, (1, 1, 1))


@pytest.mark.parametrize("R", [30, 66])
def test_missing_eos_warnings(F, monkeypatch, R):
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    ref, hyp = _batch(R + 1, R, R + 4, 32, no_eos_frac=0.5)
    for include_eos in (True, False):
        exp = IO.infix(ref, hyp, eos=0, include_eos=include_eos, return_flags=True)
        fl = exp[3]
        for fn in (F.infix_matches, F.infix_edit_distance):
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                act = fn(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, include_eos=include_eos)
            msgs = [str(x.message) for x in w]
            d = act[0] if isinstance(act, tuple) else act
            assert np.array_equal(d.numpy(), exp[0])
            assert any("in ref did not" in m for m in msgs) == bool(include_eos and fl & 1)
            assert any("in hyp did not" in m for m in msgs) == bool(include_eos and fl & 2)
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                fn(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, include_eos=include_eos, warn=False)
            assert not w
        assert include_eos == bool(fl & 3)


@pytest.mark.parametrize("R", [10, 80])
@pytest.mark.parametrize("costs", [(1, 1, 1), (2, 2, 2), (1, 2, 3), (0.7, 1.1, 1.3)])
def test_norm_and_empty_sequences(F, monkeypatch, R, costs):
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    ref, hyp = _batch(R + 3, R, R + 2, 33)
    ref[0, ::3] = 0  # empty references
    hyp[0, 1::3] = 0  # empty hypotheses
    ref[0, 2::5] = hyp[0, 2::5] = 0  # both
    exp = _vs_oracle(F, torch.device("cpu"), ref, hyp, costs, eos=0, norm=True)
    assert (exp[0][::3] == 0).all() and (exp[1][::3] == 0).all() and (exp[2][::3] == 0).all()
    assert (exp[1][1::3] == 0).all() and (exp[2][1::3] == 0).all()
    r, _ = CO._lengths(ref, 0, False)
    e0 = np.float32(costs[1]) * r[1::3].astype(np.float32)
    if costs[0] == costs[1] == costs[2]:
        e0 = r[1::3].astype(np.float32) * np.float32(costs[0])
    assert np.array_equal(exp[0][1::3], e0)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        d = F.infix_edit_distance(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, norm=True,
                                  ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
    assert any("ref contains empty transcripts" in str(x.message) for x in w)
    assert (d.numpy()[::3] == 0).all()
    # zero-length tensors
    for Rz, Hz in ((0, 5), (5, 0), (0, 0)):
        r0, h0 = np.zeros((Rz, 4), np.int64) + 2, np.zeros((Hz, 4), np.int64) + 3
        d, s, e = F.infix_matches(torch.from_numpy(r0), torch.from_numpy(h0), ins_cost=costs[0],
                                  del_cost=costs[1], sub_cost=costs[2])
        exp0 = IO.infix(r0, h0, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
        assert np.array_equal(d.numpy(), exp0[0]) and s.tolist() == [0] * 4 and e.tolist() == [0] * 4
    for fn in (F.infix_matches, F.infix_edit_distance):
        out = fn(torch.zeros(5, 0, dtype=torch.long), torch.zeros(6, 0, dtype=torch.long))
        for t in (out if isinstance(out, tuple) else (out,)):
            assert t.shape == (0,)


def test_planted_twice(F, monkeypatch):
    """A reference planted verbatim twice in noise: distance 0 at the earlier occurrence."""
    monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    rng = np.random.default_rng(3)
    for R in (9, 40, 100):
        ref = rng.integers(10, 20, (R, 6))
        hyp = rng.integers(1, 8, (3 * R + 20, 6))
        hyp[7:7 + R] = ref
        hyp[2 * R + 10:3 * R + 10] = ref
        for costs in ((1, 1, 1), (3, 3, 4), (0.7, 1.1, 1.3)):
            c = dict(ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
            d, s, e = F.infix_matches(torch.from_numpy(ref), torch.from_numpy(hyp), **c)
            assert (d == 0).all() and (s == 7).all() and (e == 7 + R).all()
            assert (F.infix_edit_distance(torch.from_numpy(ref), torch.from_numpy(hyp), **c) == 0).all()


def test_shape_errors(F):
    for fn in (F.infix_matches, F.infix_edit_distance):
        with pytest.raises(RuntimeError, match="2 dimensional"):
            fn(torch.zeros(3, dtype=torch.long), torch.zeros(3, 2, dtype=torch.long))
        with pytest.raises(RuntimeError, match="ref has batch size 2, but hyp has 3"):
            fn(torch.zeros(3, 2, dtype=torch.long), torch.zeros(3, 3, dtype=torch.long))


def test_modules_script_and_trace(F):
    import b200lev.modules as M

    ref, hyp = _batch(3, 20, 26, 8)
    c = dict(ins_cost=1.0, del_cost=2.0, sub_cost=3.0)
    tr, th = torch.from_numpy(ref), torch.from_numpy(hyp)
    ref2, hyp2 = _batch(4, 70, 40, 5)  # other shapes than the example
    tr2, th2 = torch.from_numpy(ref2), torch.from_numpy(hyp2)
    exp = IO.infix(ref, hyp, eos=0, **c)
    exp2 = IO.infix(ref2, hyp2, eos=0, **c)
    mod = M.InfixMatches(eos=0, **c)
    for m in (mod, torch.jit.script(mod)):
        got = m(tr, th)
        assert all(np.array_equal(a.numpy(), b) for a, b in zip(got, exp))
    traced = torch.jit.trace(mod, (tr, th))
    assert all(np.array_equal(a.numpy(), b) for a, b in zip(traced(tr2, th2), exp2))
    assert "eos=0" in repr(mod)
    modd = M.InfixEditDistance(eos=0, norm=True, **c)
    expn = IO.infix(ref, hyp, eos=0, norm=True, **c)[0]
    expn2 = IO.infix(ref2, hyp2, eos=0, norm=True, **c)[0]
    for m in (modd, torch.jit.script(modd)):
        assert np.array_equal(m(tr, th).numpy(), expn)
    assert np.array_equal(torch.jit.trace(modd, (tr, th))(tr2, th2).numpy(), expn2)
    assert "norm=True" in repr(modd)


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


def _call(abi, ref, hyp, ref_group=1, norm=0, dist="buf", start="buf", end="buf", ws="buf", ws_short=0):
    L = abi.lib()
    o = abi.Opts(0, 0, 0, 1.0, 2.0, 3.0, norm, 0, -1, 0, ref_group)
    nbytes = L.b200lev_workspace_bytes(ctypes.byref(ref), ctypes.byref(hyp), 0, 0)
    ws = np.zeros(nbytes, np.uint8) if ws == "buf" else ws
    n = max(int(hyp.N), 1)
    dist = np.full(n, 7, np.float32) if dist == "buf" else dist
    start = np.full(n, 7, np.int64) if start == "buf" else start
    end = np.full(n, 7, np.int64) if end == "buf" else end
    flags = np.zeros(1, np.int32)
    ptr = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    rc = L.b200lev_infix(ctypes.byref(ref), ctypes.byref(hyp), ctypes.byref(o), ptr(dist), ptr(start),
                         ptr(end), ptr(ws), nbytes - ws_short, flags.ctypes.data, 0)
    return rc, dist, start, end


def test_abi_statuses(abi):
    OK, ERR_ARG, ERR_WORKSPACE = 0, -1, -3
    ref, hyp = _tokens(abi, 6, 3, 0), _tokens(abi, 9, 3, 1)
    rc, d, s, e = _call(abi, ref, hyp)
    exp = IO.infix(ref.keep, hyp.keep, ins_cost=1, del_cost=2, sub_cost=3)
    assert rc == OK and np.array_equal(d, exp[0]) and np.array_equal(s, exp[1]) and np.array_equal(e, exp[2])
    rc, d, s, e = _call(abi, ref, hyp, start=None, end=None, norm=1)  # distances only: norm applies
    assert rc == OK and np.array_equal(d, IO.infix(ref.keep, hyp.keep, norm=True, ins_cost=1, del_cost=2,
                                                   sub_cost=3)[0])
    assert _call(abi, ref, hyp, start=None)[0] == ERR_ARG  # one span pointer NULL
    assert _call(abi, ref, hyp, end=None)[0] == ERR_ARG
    assert _call(abi, ref, hyp, norm=1)[0] == ERR_ARG  # norm with spans
    assert b"norm" in abi.lib().b200lev_last_error()
    assert _call(abi, _tokens(abi, 6, 1, 0), hyp, ref_group=3)[0] == ERR_ARG
    assert _call(abi, ref, hyp, ref_group=2)[0] == ERR_ARG
    assert b"ref_group" in abi.lib().b200lev_last_error()
    assert _call(abi, ref, _tokens(abi, 5, 2, 1))[0] == ERR_ARG  # batch mismatch
    assert _call(abi, ref, hyp, ws_short=1)[0] == ERR_WORKSPACE
    assert _call(abi, ref, hyp, dist=None)[0] == ERR_ARG
    assert _call(abi, ref, hyp, ws=None)[0] == ERR_ARG
    # no pairs: nothing to write, NULL buffers are fine
    assert _call(abi, _tokens(abi, 6, 0, 0), _tokens(abi, 5, 0, 1), dist=None, start=None, end=None,
                 ws=None)[0] == OK


# ---- the device ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def FG():
    import b200lev.functional as F_

    return F_


@pytest.mark.gpu
@pytest.mark.parametrize("costs", ALL_COSTS)
@pytest.mark.parametrize("R", [1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257])
def test_gpu_random_vs_oracle(FG, capfd, R, costs):
    N = 700 if R <= 65 else 90
    ref, hyp = _batch(R * 7 + len(str(costs)), R, R + 5, N, no_eos_frac=0.2)
    for n in range(0, N, 3):
        hyp[3:3 + R // 2, n] = np.where(ref[:R // 2, n] == 0, 1, ref[:R // 2, n])
    _, lines = _route(FG, capfd, lambda: _vs_oracle(FG, torch.device("cuda"), ref, hyp, costs, eos=0))
    assert ("infix kind" in lines[1]) == _short_expected(R, costs)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.int8, torch.int16, torch.int32, torch.long])
@pytest.mark.parametrize("R", [20, 50, 90])
def test_gpu_token_widths_and_wide_tokens(FG, dtype, R):
    dev = torch.device("cuda")
    ref, hyp = _batch(R + 11, R, R + 9, 1000, V=9)
    for costs in ((1, 1, 1), (3, 3, 4), (0.7, 1.1, 1.3)):
        _vs_oracle(FG, dev, ref, hyp, costs, dtype=dtype, eos=0)
    if dtype == torch.long:
        big = np.int64(1) << 32
        for costs in ((1, 1, 1), (1, 2, 3)):
            _vs_oracle(FG, dev, np.where(ref % 2 == 1, ref + big, ref), hyp, costs, eos=0)
            _vs_oracle(FG, dev, ref, np.where(hyp % 3 == 1, hyp + 3 * big, hyp), costs, eos=0)
    _vs_oracle(FG, dev, ref, hyp, dtype=torch.int32, hdtype=dtype, eos=0)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [30, 100])
def test_gpu_layouts_flags_and_norm(FG, R):
    dev = torch.device("cuda")
    ref, hyp = _batch(R, R, R + 4, 999, no_eos_frac=0.3)
    ref[0, ::7] = 0
    hyp[0, 3::7] = 0
    for costs in ((1, 1, 1), (1, 2, 3)):
        exp = IO.infix(ref, hyp, eos=0, include_eos=True, ins_cost=costs[0], del_cost=costs[1],
                       sub_cost=costs[2], return_flags=True)
        rb, hb = torch.from_numpy(ref.T.copy()).to(dev), torch.from_numpy(hyp.T.copy()).to(dev)
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            d, s, e = FG.infix_matches(rb, hb, eos=0, include_eos=True, batch_first=True, ins_cost=costs[0],
                                       del_cost=costs[1], sub_cost=costs[2])
        assert np.array_equal(d.cpu().numpy(), exp[0]) and np.array_equal(s.cpu().numpy(), exp[1])
        assert np.array_equal(e.cpu().numpy(), exp[2])
        assert exp[3] == 3 and len(w) == 2
        _vs_oracle(FG, dev, ref, hyp, costs, eos=0, norm=True)
    _vs_oracle(FG, dev, ref, hyp, (0.7, 1.1, 1.3))  # eos=None


@pytest.mark.gpu
def test_gpu_host_tensors_in_and_out(FG):
    ref, hyp = _batch(12, 40, 120, 500)
    for costs in ((1, 1, 1), (3, 3, 4)):
        c = dict(ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
        exp = IO.infix(ref, hyp, eos=0, **c)
        d, s, e = FG.infix_matches(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, **c)
        assert d.device.type == "cpu" and s.device.type == "cpu" and e.device.type == "cpu"
        assert np.array_equal(d.numpy(), exp[0]) and np.array_equal(s.numpy(), exp[1])
        assert np.array_equal(e.numpy(), exp[2])
        dd = FG.infix_edit_distance(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, **c)
        assert dd.device.type == "cpu" and np.array_equal(dd.numpy(), exp[0])


@pytest.mark.gpu
@pytest.mark.parametrize("R", [31, 100])
def test_gpu_cuda_graph_replay(FG, R):
    dev = torch.device("cuda")
    ref, hyp = _batch(R, R, 3 * R, 2048)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    for costs in ((1, 1, 1), (1, 2, 3)):
        c = dict(eos=0, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2], warn=False)
        eager = FG.infix_matches(tr, th, **c) + (FG.infix_edit_distance(tr, th, **c),)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            FG.infix_matches(tr, th, **c)
            FG.infix_edit_distance(tr, th, **c)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = FG.infix_matches(tr, th, **c) + (FG.infix_edit_distance(tr, th, **c),)
        for t in out:
            t.fill_(-1)
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(out, eager))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["a", "c", "d"])
def test_gpu_benchmark_shapes_vs_shifted_prefix(FG, shape):
    """The benchmark shapes at full size: dist equals the shifted-prefix composition, and each match
    rescored with edit_distance gives dist back."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import bench_infix as BI

    dev = torch.device("cuda")
    ref, hyp, costs, eos = BI.make(shape, dev)
    c = dict(ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
    d = FG.infix_edit_distance(ref, hyp, eos=eos, warn=False, **c)
    dm, s, e = FG.infix_matches(ref, hyp, eos=eos, warn=False, **c)
    assert torch.equal(d, dm)
    if shape != "d":
        assert torch.equal(d, BI.shifted_prefix(ref, hyp, costs, eos))
    # rescore hyp[start:end] (the rest set to eos)
    pos = torch.arange(hyp.shape[0], device=dev)[:, None]
    keep = (pos >= s[None]) & (pos < e[None])
    idx = (pos + s[None]).clamp(max=hyp.shape[0] - 1)
    sub = torch.where(pos < (e - s)[None], torch.gather(hyp, 0, idx), torch.full_like(hyp, eos))
    assert int(keep.sum()) == int((e - s).sum())
    ed = FG.edit_distance(ref, torch.cat([sub, torch.full_like(hyp[:1], eos)]), eos=eos, warn=False, **c)
    assert torch.equal(ed, d)
