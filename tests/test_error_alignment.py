"""error_alignment: per pair the edit operations along the path error_counts counts.

The CPU restatement (tests/alignment_oracle.py) is pinned to the counts restatement, and through
it to the reference: its op histogram equals counts_oracle.error_counts on every stored golden
case, on the sclite fixture and on random pairs.  The library is then compared with the
restatement bit for bit, on the SIMT emulator (tests/emu) and on the device.
"""
import ctypes
import warnings

import numpy as np
import pytest
import torch

import alignment_oracle as AO
import counts_oracle as CO
import parity_cases as PC

KNOWN = [  # ref, hyp, (ins, del, sub), ops
    ("kitten", "sitting", (1, 1, 1), "SCCCSCI"),
    ("sitting", "kitten", (1, 1, 1), "SCCCSCD"),
    ("foot", "bot", (1, 1, 1), "DSCC"),
    ("ab", "ba", (1, 1, 1), "SS"),
    ("ab", "ba", (1, 1, 2), "DCI"),
    ("abcd", "acbd", (1, 1, 1), "CSSC"),
    ("abc", "xaby", (3, 3, 4), "ICCS"),
    ("abcd", "xbcdy", (3, 3, 4), "SCCCI"),
    ("abc", "", (1, 1, 1), "DDD"),
    ("", "abc", (1, 1, 1), "III"),
]
COSTS = [(1, 1, 1), (3, 3, 4), (1, 2, 3), (0.5, 1.0, 0.25), (0.7, 1.1, 1.3)]


def _col(s):
    return np.array([ord(c) for c in s], np.int64).reshape(len(s), 1)


def _letters(ops):
    return "".join(AO.OPS[o] for o in ops if o >= 0)


def _kw(costs):
    return dict(ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])


# ---- the CPU restatement against the counts restatement ----------------------------------
@pytest.mark.parametrize("k", range(len(KNOWN)))
def test_oracle_known_answers(k):
    r, h, c, exp = KNOWN[k]
    ops = AO.error_alignment(_col(r), _col(h), **_kw(c))
    assert ops.shape == (len(r) + len(h), 1) and ops.dtype == np.int8
    assert _letters(ops[:, 0]) == exp
    assert (ops[len(exp):] == -1).all()


def test_oracle_histogram_vs_golden(golden_sm):
    n = 0
    for case, p in golden_sm.params.items():
        if not golden_sm.has(case, "error_rate"):
            continue
        ref, hyp = golden_sm.get(case, "ref"), golden_sm.get(case, "hyp")
        kw = dict(eos=p["eos"], include_eos=p["include_eos"], batch_first=p["batch_first"],
                  ins_cost=p["ins"], del_cost=p["del"], sub_cost=p["sub"])
        ops = AO.error_alignment(ref, hyp, **kw)
        assert np.array_equal(AO.histogram(ops, p["batch_first"]), CO.error_counts(ref, hyp, **kw)), case
        n += 1
    assert n >= 80


def test_oracle_histogram_sclite(golden_sclite):
    z = golden_sclite
    kw = dict(eos=-1, include_eos=False, ins_cost=3.0, del_cost=3.0, sub_cost=4.0)
    ops = AO.error_alignment(z["ref"], z["hyp"], **kw)
    assert np.array_equal(AO.histogram(ops), CO.error_counts(z["ref"], z["hyp"], **kw))


@pytest.mark.parametrize("costs", COSTS)
def test_oracle_histogram_random(costs):
    rng = np.random.default_rng(len(str(costs)))
    for R, H in ((0, 4), (5, 0), (7, 9), (12, 3), (3, 12)):
        ref, hyp = rng.integers(0, 4, (R, 80)), rng.integers(0, 4, (H, 80))
        ops = AO.error_alignment(ref, hyp, eos=0, **_kw(costs))
        assert np.array_equal(AO.histogram(ops), CO.error_counts(ref, hyp, eos=0, **_kw(costs)))


# ---- the library on the SIMT emulator ---------------------------------------------------------
@pytest.fixture(scope="module")
def F():
    from emu_backend import emulated_kernels

    with emulated_kernels():
        import b200lev.functional as F_

        yield F_


def _batch(seed, R, H, N, V=7, eos=0, no_eos_frac=0.0, min_frac=0.3):
    rng = np.random.default_rng(seed)
    ref = PC.random_tokens(rng, R, N, V, eos, -2, int(R * min_frac), no_eos_frac)
    hyp = PC.random_tokens(rng, H, N, V, eos, -3, int(H * min_frac), no_eos_frac)
    return ref, hyp


def _vs_oracle(F, dev, ref, hyp, costs=(1, 1, 1), dtype=torch.long, **kw):
    exp = AO.error_alignment(ref, hyp, **_kw(costs), **kw)
    tr, th = torch.from_numpy(ref).to(dev).to(dtype), torch.from_numpy(hyp).to(dev).to(dtype)
    act = F.error_alignment(tr, th, warn=False, **_kw(costs), **kw)
    assert act.dtype == torch.int8 and act.device == tr.device
    assert np.array_equal(act.cpu().numpy(), exp)
    return exp


def test_known_answers(F):
    for r, h, c, exp in KNOWN:
        got = F.error_alignment(torch.from_numpy(_col(r)), torch.from_numpy(_col(h)), **_kw(c))
        assert _letters(got[:, 0].tolist()) == exp


@pytest.mark.parametrize("costs", COSTS)
@pytest.mark.parametrize("R", [1, 31, 32, 33, 63, 64, 65, 130, 300])
def test_random_vs_oracle(F, R, costs):
    """Short form (R <= 64: 32 and 64 columns), long form with one strip (R <= 127 / 255) and with
    several (R = 300 with fp32 cells: three strips of 128 columns; int32: two of 256)."""
    N = 40 if R <= 64 else (12 if R < 300 else 4)
    ref, hyp = _batch(R * 7 + len(str(costs)), R, R + 3, N, no_eos_frac=0.2)
    exp = _vs_oracle(F, torch.device("cpu"), ref, hyp, costs, eos=0)
    assert np.array_equal(AO.histogram(exp), CO.error_counts(ref, hyp, eos=0, **_kw(costs)))


@pytest.mark.parametrize("dtype", [torch.int8, torch.int16, torch.int32, torch.long])
@pytest.mark.parametrize("R", [20, 50, 90])
def test_token_widths(F, dtype, R):
    ref, hyp = _batch(R + 11, R, R - 5, 37, V=9)
    _vs_oracle(F, torch.device("cpu"), ref, hyp, (3, 3, 4), dtype=dtype, eos=0)
    _vs_oracle(F, torch.device("cpu"), ref, hyp, (1, 1, 1), dtype=dtype, eos=0)


@pytest.mark.parametrize("R", [20, 40, 80])
@pytest.mark.parametrize("side", ["ref", "hyp", "both"])
def test_tokens_outside_int32(F, R, side):
    ref, hyp = _batch(R + len(side), R, R + 2, 35, V=5)
    big = np.int64(1) << 32
    if side in ("ref", "both"):
        ref = np.where(ref % 2 == 1, ref + big, ref)
    if side in ("hyp", "both"):
        hyp = np.where(hyp % 3 == 1, hyp + big * 3, hyp)
    for costs in ((1, 1, 1), (1, 2, 3)):
        _vs_oracle(F, torch.device("cpu"), ref, hyp, costs, eos=0)


def test_mixed_token_widths(F):
    ref, hyp = _batch(5, 30, 30, 33)
    exp = AO.error_alignment(ref, hyp, eos=0)
    act = F.error_alignment(torch.from_numpy(ref).int(), torch.from_numpy(hyp), eos=0)
    assert np.array_equal(act.numpy(), exp)


@pytest.mark.parametrize("R", [24, 70])
def test_batch_first_strided_and_eos_none(F, R):
    cpu = torch.device("cpu")
    ref, hyp = _batch(R, R, R + 4, 34)
    rb, hb = np.ascontiguousarray(ref.T), np.ascontiguousarray(hyp.T)
    exp = _vs_oracle(F, cpu, rb, hb, (1, 2, 3), eos=0, batch_first=True)
    assert exp.shape == (34, 2 * R + 4)
    assert np.array_equal(exp.T, AO.error_alignment(ref, hyp, eos=0, ins_cost=1, del_cost=2, sub_cost=3))
    seq = exp.T
    big_r, big_h = np.repeat(ref, 2, axis=1), np.repeat(hyp, 2, axis=1)
    act = F.error_alignment(torch.from_numpy(big_r)[:, ::2], torch.from_numpy(big_h)[:, ::2], eos=0,
                            ins_cost=1, del_cost=2, sub_cost=3)
    assert np.array_equal(act.numpy(), seq)
    tr2, th2 = torch.from_numpy(np.repeat(ref, 2, axis=0))[::2], torch.from_numpy(np.repeat(hyp, 2, axis=0))[::2]
    act = F.error_alignment(tr2, th2, eos=0, ins_cost=1, del_cost=2, sub_cost=3)
    assert np.array_equal(act.numpy(), seq)
    # no eos: every path runs through the full padded lengths
    exp = _vs_oracle(F, cpu, ref, hyp, (3, 3, 4))
    ref_pos, hyp_pos = AO.histogram(exp)[:, :3].sum(1), AO.histogram(exp)[:, [0, 1, 3]].sum(1)
    assert (ref_pos == R).all() and (hyp_pos == R + 4).all()


@pytest.mark.parametrize("R", [30, 66])
def test_missing_eos_warnings(F, R):
    ref, hyp = _batch(R + 1, R, R, 32, no_eos_frac=0.5)
    for include_eos in (True, False):
        exp, fl = AO.error_alignment(ref, hyp, eos=0, include_eos=include_eos, return_flags=True)
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            act = F.error_alignment(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, include_eos=include_eos)
        msgs = [str(x.message) for x in w]
        assert np.array_equal(act.numpy(), exp)
        assert any("in ref did not" in m for m in msgs) == bool(include_eos and fl & 1)
        assert any("in hyp did not" in m for m in msgs) == bool(include_eos and fl & 2)
        assert include_eos == bool(fl & 3)
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            F.error_alignment(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, include_eos=include_eos,
                              warn=False)
        assert not w


@pytest.mark.parametrize("R", [10, 80])
def test_empty_references_and_hypotheses(F, R):
    ref, hyp = _batch(R + 3, R, R, 33)
    ref[0, ::3] = 0  # empty references
    hyp[0, 1::3] = 0  # empty hypotheses
    ref[0, 2::5] = hyp[0, 2::5] = 0  # both
    exp = _vs_oracle(F, torch.device("cpu"), ref, hyp, (1, 2, 3), eos=0)
    assert ((exp[:, ::3] == 3) | (exp[:, ::3] == -1)).all()
    assert ((exp[:, 1::3] == 2) | (exp[:, 1::3] == -1)).all()
    assert (exp[:, 2::5] == -1).all()
    for Rz, Hz in ((0, 5), (5, 0), (0, 0)):
        r0, h0 = np.zeros((Rz, 4), np.int64) + 2, np.zeros((Hz, 4), np.int64) + 3
        got = F.error_alignment(torch.from_numpy(r0), torch.from_numpy(h0))
        assert got.shape == (Rz + Hz, 4) and got.dtype == torch.int8
        assert got.tolist() == [[2] * 4] * Rz + [[3] * 4] * Hz
    got = F.error_alignment(torch.zeros(5, 0, dtype=torch.long), torch.zeros(6, 0, dtype=torch.long))
    assert got.shape == (11, 0)
    got = F.error_alignment(torch.zeros(0, 5, dtype=torch.long), torch.zeros(0, 6, dtype=torch.long),
                            batch_first=True)
    assert got.shape == (0, 11)


def test_shape_errors(F):
    with pytest.raises(RuntimeError, match="2 dimensional"):
        F.error_alignment(torch.zeros(3, dtype=torch.long), torch.zeros(3, 2, dtype=torch.long))
    with pytest.raises(RuntimeError, match="ref has batch size 2, but hyp has 3"):
        F.error_alignment(torch.zeros(3, 2, dtype=torch.long), torch.zeros(3, 3, dtype=torch.long))


@pytest.mark.parametrize("batch_first", [False, True])
def test_alignment_positions(F, batch_first):
    """C joins equal tokens and S different ones; ref_pos runs 0 .. r-1 and hyp_pos 0 .. h-1 in
    order, -1 on the steps that do not consume that side and on padding."""
    ref, hyp = _batch(9, 40, 45, 30, V=4)
    r, h = CO._lengths(ref, 0, False)[0], CO._lengths(hyp, 0, False)[0]
    tr, th = torch.from_numpy(ref), torch.from_numpy(hyp)
    if batch_first:
        tr, th = tr.t().contiguous(), th.t().contiguous()
    ops = F.error_alignment(tr, th, eos=0, batch_first=batch_first, ins_cost=3, del_cost=3, sub_cost=4)
    ref_pos, hyp_pos = F.alignment_positions(ops, batch_first)
    assert ref_pos.dtype == hyp_pos.dtype == torch.long and ref_pos.shape == ops.shape
    if batch_first:
        ops, ref_pos, hyp_pos = ops.t(), ref_pos.t(), hyp_pos.t()
    ops, ref_pos, hyp_pos = ops.numpy(), ref_pos.numpy(), hyp_pos.numpy()
    for n in range(ref.shape[1]):
        o, rp, hp = ops[:, n], ref_pos[:, n], hyp_pos[:, n]
        assert rp[rp >= 0].tolist() == list(range(r[n]))
        assert hp[hp >= 0].tolist() == list(range(h[n]))
        assert ((rp >= 0) == ((o >= 0) & (o != 3))).all() and ((hp >= 0) == ((o >= 0) & (o != 2))).all()
        both = (o == 0) | (o == 1)
        eq = ref[rp[both], n] == hyp[hp[both], n]
        assert (eq == (o[both] == 0)).all()
    scripted = torch.jit.script(F.alignment_positions)
    again = scripted(torch.from_numpy(ops), False)
    assert np.array_equal(again[0].numpy(), ref_pos) and np.array_equal(again[1].numpy(), hyp_pos)


def test_module_script_and_trace(F):
    import b200lev.modules as M

    ref, hyp = _batch(3, 20, 22, 8)
    mod = M.ErrorAlignment(eos=0, ins_cost=1.0, del_cost=2.0, sub_cost=3.0)
    exp = AO.error_alignment(ref, hyp, eos=0, ins_cost=1, del_cost=2, sub_cost=3)
    tr, th = torch.from_numpy(ref), torch.from_numpy(hyp)
    assert np.array_equal(mod(tr, th).numpy(), exp)
    assert np.array_equal(torch.jit.script(mod)(tr, th).numpy(), exp)
    traced = torch.jit.trace(mod, (tr, th))
    ref2, hyp2 = _batch(4, 70, 40, 5)  # other shapes than the example: the long form
    exp2 = AO.error_alignment(ref2, hyp2, eos=0, ins_cost=1, del_cost=2, sub_cost=3)
    assert np.array_equal(traced(torch.from_numpy(ref2), torch.from_numpy(hyp2)).numpy(), exp2)
    assert "eos=0" in repr(mod)


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


def _call(abi, ref, hyp, ref_group=1, out="buf", ws="buf", ws_short=0):
    L = abi.lib()
    o = abi.Opts(1, 0, 0, 1.0, 1.0, 1.0, 0, 0, -1, 1, ref_group)
    nbytes = L.b200lev_workspace_bytes(ctypes.byref(ref), ctypes.byref(hyp), 3, 0)
    ws = np.zeros(nbytes, np.uint8) if ws == "buf" else ws
    T = int(ref.T + hyp.T)
    out = np.full((max(T, 1), max(int(hyp.N), 1)), 7, np.int8) if out == "buf" else out
    flags = np.zeros(1, np.int32)
    rc = L.b200lev_error_alignment(ctypes.byref(ref), ctypes.byref(hyp), ctypes.byref(o),
                                   None if out is None else out.ctypes.data, int(hyp.N), 1,
                                   None if ws is None else ws.ctypes.data, nbytes - ws_short,
                                   flags.ctypes.data, 0)
    return rc, out


@pytest.mark.parametrize("R", [6, 70])
def test_abi_statuses(abi, R):
    OK, ERR_ARG, ERR_WORKSPACE = 0, -1, -3
    ref, hyp = _tokens(abi, R, 3, 0), _tokens(abi, 5, 3, 1)
    rc, out = _call(abi, ref, hyp)
    assert rc == OK
    assert AO.histogram(out).tolist() == CO.error_counts(ref.keep, hyp.keep).tolist()
    assert _call(abi, ref, _tokens(abi, 5, 2, 1))[0] == ERR_ARG  # batch mismatch
    assert _call(abi, ref, hyp, ws_short=1)[0] == ERR_WORKSPACE
    assert _call(abi, ref, hyp, out=None)[0] == ERR_ARG
    assert _call(abi, ref, hyp, ws=None)[0] == ERR_ARG
    assert _call(abi, _tokens(abi, R, 1, 0), hyp, ref_group=3)[0] == ERR_ARG
    assert b"ref_group" in abi.lib().b200lev_last_error()
    # nothing to write: no pairs, or no steps (R + H = 0); NULL buffers are fine
    assert _call(abi, _tokens(abi, R, 0, 0), _tokens(abi, 5, 0, 1), out=None, ws=None)[0] == OK
    assert _call(abi, _tokens(abi, 0, 3, 0), _tokens(abi, 0, 3, 1), out=None, ws=None)[0] == OK


def test_workspace_kinds_keep_their_sizes(abi):
    """Kinds 0-2 report the sizes they reported before kind 3 existed (pinned); kind 3 is the final
    layout plus the trace region (and, long form, one int32 per pair), each rounded to 128 bytes."""
    L = abi.lib()
    before = {  # (R, H, N): sizes of kinds 0, 1, 2 without the alignment kind
        (31, 31, 1000): (357632, 873600, 485632),
        (64, 70, 33): (31488, 75776, 41088),
        (65, 40, 12): (12416, 28288, 14592),
        (300, 310, 5): (34432, 114816, 40704),
    }

    def up(n):
        return -(-n // 128) * 128

    for (R, H, N), exp in before.items():
        ref, hyp = _tokens(abi, R, N, 0), _tokens(abi, H, N, 1)
        size = [L.b200lev_workspace_bytes(ctypes.byref(ref), ctypes.byref(hyp), k, 0) for k in range(4)]
        assert tuple(size[:3]) == exp
        if R <= 64:
            extra = up(4 * (2 if R <= 32 else 4) * H * N)
        else:
            per_pair = max((R + 32 * C) // (32 * C) * (H + 31) * 32 * (C // 4) for C in (8, 4))
            extra = up(per_pair * N) + up(4 * N)
        assert size[3] == size[0] + extra


# ---- the device ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def FG():
    import b200lev.functional as F_

    return F_


@pytest.mark.gpu
@pytest.mark.parametrize("costs", COSTS)
@pytest.mark.parametrize("R", [1, 31, 32, 33, 63, 64, 65, 130, 300])
def test_gpu_random_vs_oracle(FG, R, costs):
    N = 777 if R <= 130 else 100
    ref, hyp = _batch(R * 7 + len(str(costs)), R, R + 3, N, no_eos_frac=0.2)
    _vs_oracle(FG, torch.device("cuda"), ref, hyp, costs, eos=0)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.int8, torch.int16, torch.int32, torch.long])
@pytest.mark.parametrize("R", [20, 50, 90])
def test_gpu_token_widths_and_wide_tokens(FG, dtype, R):
    dev = torch.device("cuda")
    ref, hyp = _batch(R + 11, R, R - 5, 1000, V=9)
    _vs_oracle(FG, dev, ref, hyp, (3, 3, 4), dtype=dtype, eos=0)
    _vs_oracle(FG, dev, ref, hyp, (1, 1, 1), dtype=dtype, eos=0)
    if dtype == torch.long:
        big = np.int64(1) << 32
        _vs_oracle(FG, dev, np.where(ref % 2 == 1, ref + big, ref), hyp, (1, 2, 3), eos=0)
        _vs_oracle(FG, dev, ref, np.where(hyp % 3 == 1, hyp + 3 * big, hyp), (1, 1, 1), eos=0)
    else:
        exp = AO.error_alignment(ref, hyp, eos=0)
        act = FG.error_alignment(torch.from_numpy(ref).to(dev).to(dtype), torch.from_numpy(hyp).to(dev), eos=0)
        assert np.array_equal(act.cpu().numpy(), exp)  # mixed widths: the long form


@pytest.mark.gpu
@pytest.mark.parametrize("R", [30, 100])
def test_gpu_layouts_and_flags(FG, R):
    dev = torch.device("cuda")
    ref, hyp = _batch(R, R, R + 4, 999, no_eos_frac=0.3)
    ref[0, ::7] = 0
    hyp[0, 3::7] = 0
    exp, fl = AO.error_alignment(ref, hyp, eos=0, include_eos=True, ins_cost=1, del_cost=2, sub_cost=3,
                                 return_flags=True)
    rb, hb = torch.from_numpy(ref.T.copy()).to(dev), torch.from_numpy(hyp.T.copy()).to(dev)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        act = FG.error_alignment(rb, hb, eos=0, include_eos=True, batch_first=True, ins_cost=1, del_cost=2,
                                 sub_cost=3)
    assert np.array_equal(act.cpu().numpy(), exp.T)
    assert fl == 3 and len(w) == 2
    _vs_oracle(FG, dev, ref, hyp, (0.7, 1.1, 1.3))  # eos=None
    # strided views of both sides
    tr = torch.from_numpy(np.repeat(ref, 2, axis=1)).to(dev)[:, ::2]
    th = torch.from_numpy(np.repeat(hyp, 2, axis=0)).to(dev)[::2]
    act = FG.error_alignment(tr, th, eos=0, ins_cost=3, del_cost=3, sub_cost=4, warn=False)
    assert np.array_equal(act.cpu().numpy(), AO.error_alignment(ref, hyp, eos=0, ins_cost=3, del_cost=3,
                                                                  sub_cost=4))


@pytest.mark.gpu
@pytest.mark.parametrize("R", [40, 90])
def test_gpu_host_tensors_in_and_out(FG, R):
    ref, hyp = _batch(12, R, R + 5, 500)
    exp = AO.error_alignment(ref, hyp, eos=0, ins_cost=3, del_cost=3, sub_cost=4)
    act = FG.error_alignment(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, ins_cost=3, del_cost=3,
                             sub_cost=4)
    assert act.device.type == "cpu" and np.array_equal(act.numpy(), exp)


def _histogram(ops):
    return torch.stack([(ops == k).sum(0) for k in range(4)], 1)


@pytest.mark.gpu
def test_gpu_cfg4_full_size(FG):
    """The bulk-scoring shape (1 M pairs, T = 31): the op histogram equals error_counts on every
    pair on the device, and a slice matches the oracle."""
    import bench

    dev = torch.device("cuda")
    ref, hyp, _ = bench.Workload(4).make(1_000_000, 0)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    kw = dict(eos=-1, include_eos=False, ins_cost=3.0, del_cost=3.0, sub_cost=4.0)
    ops = FG.error_alignment(tr, th, warn=False, **kw)
    assert ops.shape == (ref.shape[0] + hyp.shape[0], ref.shape[1])
    cnt = FG.error_counts(tr, th, warn=False, **kw)
    assert torch.equal(_histogram(ops), cnt)
    sl = slice(123_456, 123_456 + 4096)
    exp = AO.error_alignment(ref[:, sl], hyp[:, sl], **kw)
    assert np.array_equal(ops[:, sl].cpu().numpy(), exp)


@pytest.mark.gpu
def test_gpu_long_pairs_cfg5_shape(FG):
    """R = H = 2000 (cfg5 shape, few pairs): the multi-strip long form, histogram = error_counts."""
    dev = torch.device("cuda")
    rng = np.random.default_rng(5)
    ref = torch.from_numpy(rng.integers(1, 30, (2000, 6))).to(dev)
    hyp = ref.clone()
    hyp[rng.integers(0, 2000, 300)] = torch.from_numpy(rng.integers(1, 30, (300, 6))).to(dev)
    hyp = torch.roll(hyp, 7, 0)
    for costs in ((1, 1, 1), (3, 3, 4), (0.7, 1.1, 1.3)):
        ops = FG.error_alignment(ref, hyp, warn=False, **_kw(costs))
        cnt = FG.error_counts(ref, hyp, warn=False, **_kw(costs))
        assert torch.equal(_histogram(ops), cnt)
        assert ((ops >= 0).sum(0) == cnt[:, [0, 1, 2]].sum(1) + cnt[:, 3]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("R", [31, 100])
def test_gpu_cuda_graph_replay(FG, R):
    dev = torch.device("cuda")
    ref, hyp = _batch(R, R, R, 2048)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    eager = FG.error_alignment(tr, th, eos=0, ins_cost=1, del_cost=2, sub_cost=3, warn=False)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        FG.error_alignment(tr, th, eos=0, ins_cost=1, del_cost=2, sub_cost=3, warn=False)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = FG.error_alignment(tr, th, eos=0, ins_cost=1, del_cost=2, sub_cost=3, warn=False)
    out.fill_(-7)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
