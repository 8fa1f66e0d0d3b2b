"""error_counts: per pair (correct, substitutions, deletions, insertions) along the path the count
mode of error_rate takes (_string.py:292-314).

The CPU restatement (tests/counts_oracle.py) is pinned to the reference through exact
identities on its stored outputs: S + D + I is error_rate(norm=False), ins*I + del*D + sub*S is
edit_distance for integer and dyadic costs, C + S + D is the reference length.  The library is
then compared with the restatement bit for bit, on the SIMT emulator (tests/emu) and on the device.
"""
import ctypes
import os
import socket
import warnings

import numpy as np
import pytest
import torch

import counts_oracle as CO
import parity_cases as PC
from oracle import oracle as O

KNOWN = [  # ref, hyp, (ins, del, sub), (C, S, D, I)
    ("kitten", "sitting", (1, 1, 1), (4, 2, 0, 1)),
    ("sitting", "kitten", (1, 1, 1), (4, 2, 1, 0)),
    ("foot", "bot", (1, 1, 1), (2, 1, 1, 0)),
    ("ab", "ba", (1, 1, 1), (0, 2, 0, 0)),
    ("ab", "ba", (1, 1, 2), (1, 0, 1, 1)),
    ("ab", "ba", (3, 3, 4), (1, 0, 1, 1)),
    ("abcd", "acbd", (1, 1, 1), (2, 2, 0, 0)),
    ("abc", "", (1, 1, 1), (0, 0, 3, 0)),
    ("", "abc", (1, 1, 1), (0, 0, 0, 3)),
    ("abcd", "xbcdy", (3, 3, 4), (3, 1, 0, 1)),
]
COSTS = [(1, 1, 1), (3, 3, 4), (1, 2, 3), (0.5, 1.0, 0.25), (0.7, 1.1, 1.3)]
FLOAT_COSTS = {(0.7, 1.1, 1.3), (0.3, 0.3, 0.3), (1.1, 0.9, 1.7)}


def _col(s):
    return np.array([ord(c) for c in s], np.int64).reshape(len(s), 1)


def _known_batch():
    """The known-answer pairs as (T, N) columns padded with eos = 0."""
    R = max(len(r) for r, _, _, _ in KNOWN)
    H = max(len(h) for _, h, _, _ in KNOWN)
    ref = np.zeros((R + 1, len(KNOWN)), np.int64)
    hyp = np.zeros((H + 1, len(KNOWN)), np.int64)
    for n, (r, h, _, _) in enumerate(KNOWN):
        ref[:len(r), n] = _col(r)[:, 0]
        hyp[:len(h), n] = _col(h)[:, 0]
    return ref, hyp


def _check_identities(cnt, ref_len=None, hyp_len=None):
    assert (cnt >= 0).all()
    if ref_len is not None:
        assert np.array_equal(cnt[:, 0] + cnt[:, 1] + cnt[:, 2], ref_len)
    if hyp_len is not None:
        assert np.array_equal(cnt[:, 0] + cnt[:, 1] + cnt[:, 3], hyp_len)


# ---- the CPU restatement against the reference -------------------------------------------
@pytest.mark.parametrize("k", range(len(KNOWN)))
def test_oracle_known_answers(k):
    r, h, c, exp = KNOWN[k]
    got = CO.error_counts(_col(r), _col(h), ins_cost=c[0], del_cost=c[1], sub_cost=c[2])
    assert tuple(got[0].tolist()) == exp


def test_oracle_identities_vs_golden(golden_sm):
    """On every stored case: the counts reproduce the reference's error_rate bit for bit (norm:
    fp32(S + D + I) / fp32(r), 1 / 0 for an empty reference) and, for integer / dyadic costs, its
    edit_distance as ins*I + del*D + sub*S."""
    n = nd = 0
    for case, p in golden_sm.params.items():
        if not golden_sm.has(case, "error_rate"):
            continue
        ref, hyp = golden_sm.get(case, "ref"), golden_sm.get(case, "hyp")
        costs = (p["ins"], p["del"], p["sub"])
        cnt = CO.error_counts(ref, hyp, eos=p["eos"], include_eos=p["include_eos"],
                             batch_first=p["batch_first"], ins_cost=costs[0], del_cost=costs[1],
                             sub_cost=costs[2])
        C, S, D, I = cnt.T
        r, h = C + S + D, C + S + I
        _, _, ref_lens, hyp_lens = O.string_matching(ref, hyp, p["eos"], p["include_eos"], p["batch_first"],
                                                     *costs)
        assert np.array_equal(r, ref_lens) and np.array_equal(h, hyp_lens), case
        errs = (S + D + I).astype(np.float32)
        rr = r.astype(np.float32)
        if p["norm"]:
            exp = np.where(r > 0, errs / np.where(r > 0, rr, np.float32(1)), (h > 0).astype(np.float32))
        else:
            exp = errs
        assert np.array_equal(golden_sm.get(case, "error_rate"), exp.astype(np.float32)), case
        if all(float(c) * 8 == round(float(c) * 8) for c in costs):
            dist = (np.float32(costs[0]) * I + np.float32(costs[1]) * D + np.float32(costs[2]) * S).astype(np.float32)
            if p["norm"]:
                dist = np.where(r > 0, dist / np.where(r > 0, rr, np.float32(1)),
                                (h > 0).astype(np.float32))
            assert np.array_equal(golden_sm.get(case, "edit_distance"), dist.astype(np.float32)), case
            nd += 1
        n += 1
    assert n >= 80 and nd >= 50


def test_oracle_sclite(golden_sclite):
    """NIST sclite fixture, costs 3 / 3 / 4 as the bulk-scoring command uses them."""
    z = golden_sclite
    cnt = CO.error_counts(z["ref"], z["hyp"], eos=-1, include_eos=False, ins_cost=3.0, del_cost=3.0,
                         sub_cost=4.0)
    C, S, D, I = cnt.T
    assert len(C) == 50
    assert np.array_equal(S + D + I, z["errs"])
    assert np.array_equal(C + S + D, z["ref_lens"])


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
    exp = CO.error_counts(ref, hyp, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2], **kw)
    tr, th = torch.from_numpy(ref).to(dev).to(dtype), torch.from_numpy(hyp).to(dev).to(dtype)
    act = F.error_counts(tr, th, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2], warn=False, **kw)
    assert act.dtype == torch.long and act.device == tr.device
    assert np.array_equal(act.cpu().numpy(), exp)
    return exp


def test_known_answers(F):
    ref, hyp = _known_batch()
    for n, (_, _, c, exp) in enumerate(KNOWN):
        got = F.error_counts(torch.from_numpy(ref[:, n:n + 1]), torch.from_numpy(hyp[:, n:n + 1]), eos=0,
                             ins_cost=c[0], del_cost=c[1], sub_cost=c[2])
        assert tuple(got[0].tolist()) == exp


@pytest.mark.parametrize("costs", COSTS)
@pytest.mark.parametrize("R", [1, 31, 32, 33, 63, 64, 65, 130])
def test_random_vs_oracle(F, R, costs):
    """Both forms (short: R <= 64, 32 and 64 columns; long: K0 + K1 across its strip widths)."""
    N = 40 if R <= 64 else 12
    ref, hyp = _batch(R * 7 + len(str(costs)), R, R + 3, N, no_eos_frac=0.2)
    _vs_oracle(F, torch.device("cpu"), ref, hyp, costs, eos=0)


@pytest.mark.parametrize("dtype", [torch.int8, torch.int16, torch.int32])
@pytest.mark.parametrize("R", [20, 50, 90])
def test_token_widths(F, dtype, R):
    ref, hyp = _batch(R + 11, R, R - 5, 37, V=9)
    _vs_oracle(F, torch.device("cpu"), ref, hyp, (3, 3, 4), dtype=dtype, eos=0)
    _vs_oracle(F, torch.device("cpu"), ref, hyp, (1, 1, 1), dtype=dtype, eos=0)


@pytest.mark.parametrize("R", [20, 40, 80])
@pytest.mark.parametrize("side", ["ref", "hyp", "both"])
def test_tokens_outside_int32(F, R, side):
    """Tokens whose low 32 bits collide with other tokens: exact compares on both forms, with wide
    tokens in the references (exact warp path) or only in the hypotheses."""
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
    exp = CO.error_counts(ref, hyp, eos=0)
    act = F.error_counts(torch.from_numpy(ref).int(), torch.from_numpy(hyp), eos=0)
    assert np.array_equal(act.numpy(), exp)


@pytest.mark.parametrize("R", [24, 70])
def test_batch_first_strided_and_eos_none(F, R):
    cpu = torch.device("cpu")
    ref, hyp = _batch(R, R, R + 4, 34)
    # batch_first, contiguous
    rb, hb = np.ascontiguousarray(ref.T), np.ascontiguousarray(hyp.T)
    exp = _vs_oracle(F, cpu, rb, hb, (1, 2, 3), eos=0, batch_first=True)
    assert np.array_equal(exp, CO.error_counts(ref, hyp, eos=0, ins_cost=1, del_cost=2, sub_cost=3))
    # strided views: every other pair of a wider batch, every other row
    big_r, big_h = np.repeat(ref, 2, axis=1), np.repeat(hyp, 2, axis=1)
    tr, th = torch.from_numpy(big_r)[:, ::2], torch.from_numpy(big_h)[:, ::2]
    act = F.error_counts(tr, th, eos=0, ins_cost=1, del_cost=2, sub_cost=3, warn=False)
    assert np.array_equal(act.numpy(), exp)
    tr2, th2 = torch.from_numpy(np.repeat(ref, 2, axis=0))[::2], torch.from_numpy(np.repeat(hyp, 2, axis=0))[::2]
    act = F.error_counts(tr2, th2, eos=0, ins_cost=1, del_cost=2, sub_cost=3, warn=False)
    assert np.array_equal(act.numpy(), exp)
    # no eos: the full padded lengths
    exp = _vs_oracle(F, cpu, ref, hyp, (3, 3, 4))
    _check_identities(exp, np.full(ref.shape[1], R), np.full(hyp.shape[1], R + 4))


@pytest.mark.parametrize("R", [30, 66])
def test_missing_eos_warnings(F, R):
    ref, hyp = _batch(R + 1, R, R, 32, no_eos_frac=0.5)
    for include_eos in (True, False):
        exp, fl = CO.error_counts(ref, hyp, eos=0, include_eos=include_eos, return_flags=True)
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            act = F.error_counts(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, include_eos=include_eos)
        msgs = [str(x.message) for x in w]
        assert np.array_equal(act.numpy(), exp)
        assert any("in ref did not" in m for m in msgs) == bool(include_eos and fl & 1)
        assert any("in hyp did not" in m for m in msgs) == bool(include_eos and fl & 2)
        assert include_eos == bool(fl & 3)
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            F.error_counts(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, include_eos=include_eos,
                           warn=False)
        assert not w


@pytest.mark.parametrize("R", [10, 80])
def test_empty_references_and_hypotheses(F, R):
    ref, hyp = _batch(R + 3, R, R, 33)
    ref[0, ::3] = 0  # empty references
    hyp[0, 1::3] = 0  # empty hypotheses
    ref[0, 2::5] = hyp[0, 2::5] = 0  # both
    exp = _vs_oracle(F, torch.device("cpu"), ref, hyp, (1, 2, 3), eos=0)
    assert (exp[::3, [0, 1, 2]] == 0).all()
    assert (exp[1::3, [0, 1, 3]] == 0).all()
    # zero-length tensors
    for Rz, Hz in ((0, 5), (5, 0), (0, 0)):
        r0, h0 = np.zeros((Rz, 4), np.int64) + 2, np.zeros((Hz, 4), np.int64) + 3
        got = F.error_counts(torch.from_numpy(r0), torch.from_numpy(h0))
        assert got.tolist() == [[0, 0, Rz, Hz]] * 4
    assert F.error_counts(torch.zeros(5, 0, dtype=torch.long), torch.zeros(6, 0, dtype=torch.long)).shape == (0, 4)


def test_shape_errors(F):
    with pytest.raises(RuntimeError, match="2 dimensional"):
        F.error_counts(torch.zeros(3, dtype=torch.long), torch.zeros(3, 2, dtype=torch.long))
    with pytest.raises(RuntimeError, match="ref has batch size 2, but hyp has 3"):
        F.error_counts(torch.zeros(3, 2, dtype=torch.long), torch.zeros(3, 3, dtype=torch.long))


def test_module_script_and_trace(F):
    import b200lev.modules as M

    ref, hyp = _batch(3, 20, 22, 8)
    mod = M.ErrorCounts(eos=0, ins_cost=1.0, del_cost=2.0, sub_cost=3.0)
    exp = CO.error_counts(ref, hyp, eos=0, ins_cost=1, del_cost=2, sub_cost=3)
    tr, th = torch.from_numpy(ref), torch.from_numpy(hyp)
    assert np.array_equal(mod(tr, th).numpy(), exp)
    assert np.array_equal(torch.jit.script(mod)(tr, th).numpy(), exp)
    traced = torch.jit.trace(mod, (tr, th))
    ref2, hyp2 = _batch(4, 70, 40, 5)  # other shapes than the example: the long form
    exp2 = CO.error_counts(ref2, hyp2, eos=0, ins_cost=1, del_cost=2, sub_cost=3)
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
    nbytes = L.b200lev_workspace_bytes(ctypes.byref(ref), ctypes.byref(hyp), 0, 0)
    ws = np.zeros(nbytes, np.uint8) if ws == "buf" else ws
    out = np.full((max(int(hyp.N), 1), 4), 7, np.int64) if out == "buf" else out
    flags = np.zeros(1, np.int32)
    rc = L.b200lev_error_counts(ctypes.byref(ref), ctypes.byref(hyp), ctypes.byref(o),
                                None if out is None else out.ctypes.data,
                                None if ws is None else ws.ctypes.data, nbytes - ws_short,
                                flags.ctypes.data, 0)
    return rc, out


def test_abi_statuses(abi):
    OK, ERR_ARG, ERR_WORKSPACE = 0, -1, -3
    ref, hyp = _tokens(abi, 6, 3, 0), _tokens(abi, 5, 3, 1)
    rc, out = _call(abi, ref, hyp)
    assert rc == OK and (out.sum(1) >= 5).all()
    assert _call(abi, ref, _tokens(abi, 5, 2, 1))[0] == ERR_ARG  # batch mismatch
    assert _call(abi, ref, hyp, ws_short=1)[0] == ERR_WORKSPACE
    assert _call(abi, ref, hyp, out=None)[0] == ERR_ARG
    assert _call(abi, ref, hyp, ws=None)[0] == ERR_ARG
    # an n-best layout is not served: ref_group must be 1
    assert _call(abi, _tokens(abi, 6, 1, 0), hyp, ref_group=3)[0] == ERR_ARG
    assert b"ref_group" in abi.lib().b200lev_last_error()
    # no pairs: nothing to write, NULL buffers are fine
    assert _call(abi, _tokens(abi, 6, 0, 0), _tokens(abi, 5, 0, 1), out=None, ws=None)[0] == OK


# ---- two ranks, gloo --------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, ref, hyp, q):
    import sys

    import torch.distributed as dist

    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from emu_backend import emulated_kernels

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        with emulated_kernels():
            from b200lev import dist as D

            lo, hi = D.shard_bounds(hyp.shape[1], rank, world)
            per, totals = D.bulk_error_counts(torch.from_numpy(ref[:, lo:hi]), torch.from_numpy(hyp[:, lo:hi]),
                                              eos=-1, ins_cost=3.0, del_cost=3.0, sub_cost=4.0)
            q.put((rank, lo, hi, per.numpy(), totals.numpy()))
    finally:
        dist.destroy_process_group()


def test_two_rank_bulk_error_counts():
    import torch.multiprocessing as mp

    rng = np.random.default_rng(1)
    P = 42
    ref = PC.random_tokens(rng, 12, P, 9, -1, -2, min_len=3)
    hyp = PC.random_tokens(rng, 13, P, 9, -1, -2, min_len=3)
    exp = CO.error_counts(ref, hyp, eos=-1, ins_cost=3.0, del_cost=3.0, sub_cost=4.0)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ref, hyp, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, lo, hi, per, totals in got:
        assert np.array_equal(per, exp[lo:hi])
        assert totals.dtype == np.int64 and totals.tolist() == exp.sum(0).tolist()


# ---- the device ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def FG():
    import b200lev.functional as F_

    return F_


@pytest.mark.gpu
@pytest.mark.parametrize("costs", COSTS)
@pytest.mark.parametrize("R", [1, 31, 32, 33, 63, 64, 65, 130])
def test_gpu_random_vs_oracle(FG, R, costs):
    ref, hyp = _batch(R * 7 + len(str(costs)), R, R + 3, 777, no_eos_frac=0.2)
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


@pytest.mark.gpu
@pytest.mark.parametrize("R", [30, 100])
def test_gpu_layouts_and_flags(FG, R):
    dev = torch.device("cuda")
    ref, hyp = _batch(R, R, R + 4, 999, no_eos_frac=0.3)
    ref[0, ::7] = 0
    hyp[0, 3::7] = 0
    exp, fl = CO.error_counts(ref, hyp, eos=0, include_eos=True, ins_cost=1, del_cost=2, sub_cost=3,
                             return_flags=True)
    rb, hb = torch.from_numpy(ref.T.copy()).to(dev), torch.from_numpy(hyp.T.copy()).to(dev)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        act = FG.error_counts(rb, hb, eos=0, include_eos=True, batch_first=True, ins_cost=1, del_cost=2,
                              sub_cost=3)
    assert np.array_equal(act.cpu().numpy(), exp)
    assert fl == 3 and len(w) == 2
    _vs_oracle(FG, dev, ref, hyp, (0.7, 1.1, 1.3))  # eos=None


@pytest.mark.gpu
def test_gpu_host_tensors_in_and_out(FG):
    ref, hyp = _batch(12, 40, 45, 500)
    exp = CO.error_counts(ref, hyp, eos=0, ins_cost=3, del_cost=3, sub_cost=4)
    act = FG.error_counts(torch.from_numpy(ref), torch.from_numpy(hyp), eos=0, ins_cost=3, del_cost=3,
                          sub_cost=4)
    assert act.device.type == "cpu" and np.array_equal(act.numpy(), exp)


@pytest.mark.gpu
@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4)])
def test_gpu_cfg4_identities(FG, costs):
    """The bulk-scoring shape (1 M pairs, T = 31): every identity against the library's own
    error_rate and edit_distance on the device, and a slice against the oracle."""
    import bench

    dev = torch.device("cuda")
    ref, hyp, _ = bench.Workload(4).make(1_000_000, 0)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    kw = dict(eos=-1, include_eos=False, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
    cnt = FG.error_counts(tr, th, warn=False, **kw)
    C, S, D, I = cnt.unbind(1)
    er = FG.error_rate(tr, th, norm=False, warn=False, **kw)
    ed = FG.edit_distance(tr, th, norm=False, warn=False, **kw)
    rl = (tr == -1).int().argmax(0)
    hl = (th == -1).int().argmax(0)
    assert torch.equal(C + S + D, rl.long()) and torch.equal(C + S + I, hl.long())
    assert torch.equal((S + D + I).float(), er)
    assert torch.equal((costs[0] * I + costs[1] * D + costs[2] * S).float(), ed)
    sl = slice(123_456, 123_456 + 4096)
    exp = CO.error_counts(ref[:, sl], hyp[:, sl], **kw)
    assert np.array_equal(cnt[sl].cpu().numpy(), exp)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [31, 100])
def test_gpu_cuda_graph_replay(FG, R):
    dev = torch.device("cuda")
    ref, hyp = _batch(R, R, R, 2048)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    eager = FG.error_counts(tr, th, eos=0, ins_cost=1, del_cost=2, sub_cost=3, warn=False)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        FG.error_counts(tr, th, eos=0, ins_cost=1, del_cost=2, sub_cost=3, warn=False)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = FG.error_counts(tr, th, eos=0, ins_cost=1, del_cost=2, sub_cost=3, warn=False)
    out.fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
