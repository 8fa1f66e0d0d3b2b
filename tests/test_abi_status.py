"""Status codes of the C entry points for string matching, called directly through the ctypes
binding with hand-built token views (the Python layer rejects most of these arguments before
they reach the library).  Runs on the SIMT emulator (tests/emu)."""
import ctypes

import numpy as np
import pytest

from emu_backend import emulated_kernels

OK, ERR_ARG, ERR_WORKSPACE = 0, -1, -3  # include/b200lev.h
WS_FINAL, WS_COMPLETION, WS_PREFIX = 0, 1, 2
ENTRIES = ["final", "final_sums", "prefix", "completion_count", "completion_fill"]
KIND = {"final": WS_FINAL, "final_sums": WS_FINAL, "prefix": WS_PREFIX,
        "completion_count": WS_COMPLETION, "completion_fill": WS_COMPLETION}


@pytest.fixture(scope="module")
def abi():
    with emulated_kernels():
        from b200lev import _abi

        yield _abi


def _tokens(abi, T, N, seed):
    """An int64 (T, N) sequence-first view; the array is kept alive on the returned struct."""
    a = np.random.default_rng(seed).integers(1, 5, (T, N)).astype(np.int64)
    a[T - 1:, :] = 0
    t = abi.Tokens(a.ctypes.data if a.size else None, 8, T, N, N, 1)
    t.keep = a
    return t


def _opts(abi, exclude_last=0):
    return abi.Opts(1, 0, 0, 1.0, 1.0, 1.0, 0, exclude_last, -1, 1, 1)


def _ptr(a):
    return None if a is None else a.ctypes.data


def _call(abi, name, ref, hyp, o, out="buf", ws="buf", ws_short=0, acc="buf", U=3):
    """Calls b200lev_<name> with buffers big enough for the shapes unless told otherwise:
    "buf" = a right-sized buffer, None = a NULL pointer.  Returns (status, out buffer)."""
    L = abi.lib()
    nbytes = L.b200lev_workspace_bytes(ctypes.byref(ref), ctypes.byref(hyp), KIND[name],
                                       o.exclude_last)
    ws = np.zeros(nbytes, np.uint8) if ws == "buf" else ws
    n = max(int(hyp.N), 1)
    rows = max(int(hyp.T) + 1, 1)
    if out == "buf":
        dtype = np.int64 if name == "completion_fill" else (np.int32 if name == "completion_count"
                                                             else np.float32)
        out = np.full(rows * n * U, 7, dtype)
    acc = np.zeros(3, np.float64) if acc == "buf" else acc
    flags = np.zeros(1, np.int32)
    r, h, po = ctypes.byref(ref), ctypes.byref(hyp), ctypes.byref(o)
    size = nbytes - ws_short
    if name == "final":
        rc = L.b200lev_final(r, h, po, _ptr(out), _ptr(ws), size, _ptr(flags), 0)
    elif name == "final_sums":
        rc = L.b200lev_final_sums(r, h, po, _ptr(out), _ptr(ws), size, _ptr(flags), _ptr(acc), 0)
    elif name == "prefix":
        rc = L.b200lev_prefix(r, h, po, _ptr(out), n, 1, _ptr(ws), size, _ptr(flags), 0)
    elif name == "completion_count":
        rc = L.b200lev_completion_count(r, h, po, _ptr(ws), size, _ptr(out), _ptr(flags), 0)
    else:
        rc = L.b200lev_completion_fill(r, h, po, _ptr(ws), size, U, _ptr(out), n * U, U, 0)
    return rc, out


@pytest.mark.parametrize("name", ENTRIES)
def test_batch_mismatch(abi, name):
    ref, hyp = _tokens(abi, 6, 2, 0), _tokens(abi, 5, 3, 1)
    assert _call(abi, name, ref, hyp, _opts(abi))[0] == ERR_ARG


@pytest.mark.parametrize("name", ENTRIES)
def test_short_workspace(abi, name):
    ref, hyp = _tokens(abi, 6, 3, 0), _tokens(abi, 5, 3, 1)
    assert _call(abi, name, ref, hyp, _opts(abi), ws_short=1)[0] == ERR_WORKSPACE


@pytest.mark.parametrize("name", ENTRIES)
@pytest.mark.parametrize("missing", ["out", "ws"])
def test_null_buffer(abi, name, missing):
    """A NULL output or workspace with pairs to compute.  (completion_fill reports both as a bad
    workspace.)"""
    ref, hyp = _tokens(abi, 6, 3, 0), _tokens(abi, 5, 3, 1)
    rc = _call(abi, name, ref, hyp, _opts(abi), **{missing: None})[0]
    assert rc == (ERR_WORKSPACE if name == "completion_fill" else ERR_ARG)


@pytest.mark.parametrize("name", ENTRIES)
def test_empty_batch(abi, name):
    """No pairs: nothing to compute, so NULL buffers are fine.  completion_count still writes
    U = 0."""
    ref, hyp = _tokens(abi, 6, 0, 0), _tokens(abi, 5, 0, 1)
    if name == "completion_count":
        rc, umax = _call(abi, name, ref, hyp, _opts(abi), ws=None)
        assert rc == OK and umax[0] == 0
    else:
        assert _call(abi, name, ref, hyp, _opts(abi), out=None, ws=None)[0] == OK


def test_prefix_without_rows(abi):
    """exclude_last with H == 0 leaves no prefix rows: OK, and nothing is written."""
    ref, hyp = _tokens(abi, 6, 3, 0), _tokens(abi, 0, 3, 1)
    rc, out = _call(abi, "prefix", ref, hyp, _opts(abi, exclude_last=1))
    assert rc == OK and (out == 7).all()


@pytest.mark.parametrize("n", [3, 0])
def test_final_sums_needs_acc(abi, n):
    ref, hyp = _tokens(abi, 6, n, 0), _tokens(abi, 5, n, 1)
    assert _call(abi, "final_sums", ref, hyp, _opts(abi), acc=None)[0] == ERR_ARG


@pytest.mark.parametrize("name", ENTRIES)
def test_well_formed_call(abi, name):
    """The same buffers with nothing wrong: OK (so the statuses above come from the one fault)."""
    ref, hyp = _tokens(abi, 6, 3, 0), _tokens(abi, 5, 3, 1)
    assert _call(abi, name, ref, hyp, _opts(abi))[0] == OK
