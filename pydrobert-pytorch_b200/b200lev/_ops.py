"""Host side of the custom-op layer: tensor plumbing around the C ABI.

Each public call of the reference's string-matching family maps to registered torch ops
(``torch.ops.b200lev.*``) whose bodies allocate the outputs/workspace with torch, hand
raw device pointers, strides and the current CUDA stream to ``libb200lev.so`` and return.
PyTorch is used for device memory, streams and autograd wiring only; every number is
produced by the hand-written kernels.

The ops are what ``torch.jit.script`` / ``torch.jit.trace`` / ``torch.compile`` see: one
opaque node per call, shapes and checks inside, so nothing data- or shape-dependent is
baked into a graph.  Each op is a plain Python function (``*_impl``) registered with
``torch.library.custom_op``; plain eager code may call the ``*_impl`` function directly
and skip the dispatcher round trip.

There is no CPU fallback: the computation always runs on a CUDA device.  Tensors that live
on the host are copied to the current CUDA device and the results back (``_host.Placement``).
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import _abi, _host

_INT_DTYPES = _host._INT_DTYPES
_FLOAT_CODES = {torch.float32: _abi.F32, torch.float16: _abi.F16, torch.bfloat16: _abi.BF16,
                torch.float64: _abi.F64}


def _as_tokens(t: Tensor) -> Tensor:
    """Token tensors are "long tensors" in the reference (_string.py:588-596) but its
    tests also trace with float placeholders; normalise without copying when the dtype
    is already a signed integer type the kernels read directly."""
    t = t.detach()  # _string.py:186-187
    if t.dtype in _INT_DTYPES:
        return t
    if t.dtype == torch.uint8:
        return t.to(torch.int16)
    return t.to(torch.long)


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream(dev: torch.device) -> int:
    """The caller's current stream on `dev` as a raw handle (a small call is host-bound: the
    Stream object torch.cuda.current_stream builds costs 6 us of a 40 us call)."""
    if _raw_stream is not None:
        return _raw_stream(dev.index if dev.index is not None else torch.cuda.current_device())
    return torch.cuda.current_stream(dev).cuda_stream


class _DeviceGuard:
    """`with torch.cuda.device(dev)` that does nothing when `dev` is current already."""
    __slots__ = ("idx", "prev")

    def __init__(self, dev: torch.device):
        self.idx = -1 if dev.index is None else dev.index
        self.prev = -1

    def __enter__(self):
        if self.idx >= 0:
            prev = torch.cuda.current_device()
            if prev != self.idx:
                torch.cuda.set_device(self.idx)
                self.prev = prev
        return self

    def __exit__(self, *exc):
        if self.prev >= 0:
            torch.cuda.set_device(self.prev)
        return False


def _tok_struct(t: Tensor, batch_first: bool) -> _abi.Tokens:
    if batch_first:  # the transpose of _string.py:181-183, as a stride swap
        n, T = t.shape
        sn, st = t.stride()
    else:
        T, n = t.shape
        st, sn = t.stride()
    return _abi.Tokens(t.data_ptr(), t.element_size(), T, n, st, sn)


def _opts(eos: Optional[int], include_eos: bool, ins: float, del_: float, sub: float, norm: bool,
          exclude_last: bool, padding: int, return_mistakes: bool, ref_group: int) -> _abi.Opts:
    return _abi.Opts(int(eos is not None), 0 if eos is None else int(eos), int(include_eos),
                     float(ins), float(del_), float(sub), int(norm), int(exclude_last),
                     int(padding), int(return_mistakes), int(ref_group))


def _shapes(ref: Tensor, hyp: Tensor, batch_first: bool, ref_group: int) -> Tuple[int, int, int]:
    if ref.dim() != 2 or hyp.dim() != 2:
        raise RuntimeError("ref and hyp must be 2 dimensional")  # _string.py:166-167
    if batch_first:
        (nr, R), (n, H) = ref.shape, hyp.shape
    else:
        (R, nr), (H, n) = ref.shape, hyp.shape
    if nr * ref_group != n:  # _string.py:191-194
        raise RuntimeError(f"ref has batch size {nr * ref_group}, but hyp has {n}")
    return R, H, n


# ---------------------------------------------------------------------------------------
# string matching: final / prefix
# ---------------------------------------------------------------------------------------
def _string_matching_device(ref: Tensor, hyp: Tensor, dev: torch.device, eos: Optional[int],
                            include_eos: bool, batch_first: bool, ins_cost: float, del_cost: float,
                            sub_cost: float, norm: bool, prefix: bool, exclude_last: bool,
                            padding: int, return_mistakes: bool, ref_group: int
                            ) -> Tuple[Tensor, Tensor]:
    """Device tensors in, device tensors out (the body shared by the ops below)."""
    H = hyp.shape[1] if batch_first else hyp.shape[0]
    n = hyp.shape[0] if batch_first else hyp.shape[1]
    L = _abi.lib()
    with _DeviceGuard(dev):
        rt, ht = _tok_struct(ref, batch_first), _tok_struct(hyp, batch_first)
        o = _opts(eos, include_eos, ins_cost, del_cost, sub_cost, norm, exclude_last, padding,
                  return_mistakes, ref_group)
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        nbytes = L.b200lev_workspace_bytes(ctypes.byref(rt), ctypes.byref(ht), 2 if prefix else 0,
                                           int(exclude_last))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        st = _stream(dev)
        if not prefix:
            out = torch.empty(n, dtype=torch.float32, device=dev)
            _abi.check(L.b200lev_final(ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o),
                                       out.data_ptr(), ws.data_ptr(), nbytes, flags.data_ptr(), st))
        else:
            hout = H + (0 if exclude_last else 1)
            if batch_first:  # _string.py:387-388
                out = torch.empty((n, hout), dtype=torch.float32, device=dev)
                si, sn = 1, hout
            else:
                out = torch.empty((hout, n), dtype=torch.float32, device=dev)
                si, sn = n, 1
            _abi.check(L.b200lev_prefix(ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o),
                                        out.data_ptr(), si, sn, ws.data_ptr(), nbytes,
                                        flags.data_ptr(), st))
    return out, flags


def string_matching_impl(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool,
                         batch_first: bool, ins_cost: float, del_cost: float, sub_cost: float,
                         norm: bool, prefix: bool, exclude_last: bool, padding: int,
                         return_mistakes: bool, ref_group: int) -> Tuple[Tensor, Tensor]:
    """``_string_matching`` (_string.py:146-406) minus the mask mode.

    Returns ``(out, flags)``: fp32 ``(N,)`` or ``(H', N)`` / ``(N, H')`` and the int32[1]
    warning flags (``_abi.FLAG_*``), both on the device of ``ref``.  ``ref_group`` > 1 means
    reference column ``pair // ref_group`` serves the pair (an n-best batch whose
    reference is not physically repeated, _string.py:1426/1439)."""
    _shapes(ref, hyp, batch_first, ref_group)
    ref, hyp = _as_tokens(ref), _as_tokens(hyp)
    args = (eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, norm, prefix, exclude_last,
            padding, return_mistakes, ref_group)
    plan = _host.block_plan(ref, hyp, batch_first, ref_group)
    if plan is not None:  # big host batch: blocks through three streams
        return _host.string_matching_blocks(
            plan, ref, hyp, lambda r, h: _string_matching_device(r, h, r.device, *args),
            batch_first, prefix, exclude_last, ref_group)
    pl = _host.Placement(ref, hyp)
    out, flags = _string_matching_device(pl.to_dev(ref), pl.to_dev(hyp), pl.dev, *args)
    return pl.back(out), pl.back(flags)


string_matching = torch.library.custom_op("b200lev::string_matching", string_matching_impl,
                                          mutates_args=())


@string_matching.register_fake
def _(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, norm, prefix,
      exclude_last, padding, return_mistakes, ref_group):
    if batch_first:
        n, H = hyp.shape
    else:
        H, n = hyp.shape
    flags = ref.new_empty((1,), dtype=torch.int32)
    if not prefix:
        return ref.new_empty((n,), dtype=torch.float32), flags
    hout = H + (0 if exclude_last else 1)
    shape = (n, hout) if batch_first else (hout, n)
    return ref.new_empty(shape, dtype=torch.float32), flags


# ---------------------------------------------------------------------------------------
# error counts: (C, S, D, I) per pair; error alignment: the ops along the same path
# ---------------------------------------------------------------------------------------
def error_path_impl(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool, batch_first: bool,
                ins_cost: float, del_cost: float, sub_cost: float, align: bool
                ) -> Tuple[Tensor, Tensor]:
    """The body of both ops below: one C call, ``b200lev_error_alignment`` if ``align`` else
    ``b200lev_error_counts``."""
    R, H, n = _shapes(ref, hyp, batch_first, 1)
    ref, hyp = _as_tokens(ref), _as_tokens(hyp)
    pl = _host.Placement(ref, hyp)
    ref, hyp, dev = pl.to_dev(ref), pl.to_dev(hyp), pl.dev
    L = _abi.lib()
    with _DeviceGuard(dev):
        rt, ht = _tok_struct(ref, batch_first), _tok_struct(hyp, batch_first)
        o = _opts(eos, include_eos, ins_cost, del_cost, sub_cost, False, False, 0, True, 1)
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        nbytes = L.b200lev_workspace_bytes(ctypes.byref(rt), ctypes.byref(ht), 3 if align else 0, 0)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        toks = (ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o))
        rest = (ws.data_ptr(), nbytes, flags.data_ptr(), _stream(dev))
        if not align:
            out = torch.empty((n, 4), dtype=torch.long, device=dev)
            _abi.check(L.b200lev_error_counts(*toks, out.data_ptr(), *rest))
        else:
            if batch_first:
                out = torch.empty((n, R + H), dtype=torch.int8, device=dev)
                sk, sn = 1, R + H
            else:
                out = torch.empty((R + H, n), dtype=torch.int8, device=dev)
                sk, sn = n, 1
            _abi.check(L.b200lev_error_alignment(*toks, out.data_ptr(), sk, sn, *rest))
    return pl.back(out), pl.back(flags)


def error_counts_impl(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool,
                      batch_first: bool, ins_cost: float, del_cost: float, sub_cost: float
                      ) -> Tuple[Tensor, Tensor]:
    """Per pair the correct, substitution, deletion and insertion counts along the path the
    count mode of ``error_rate`` takes (_string.py:292-314), ``(out, flags)``: int64 ``(N, 4)``
    and the int32[1] warning flags, on the device of ``ref``."""
    return error_path_impl(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, False)


error_counts = torch.library.custom_op("b200lev::error_counts", error_counts_impl, mutates_args=())


@error_counts.register_fake
def _(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost):
    n = hyp.shape[0] if batch_first else hyp.shape[1]
    return ref.new_empty((n, 4), dtype=torch.long), ref.new_empty((1,), dtype=torch.int32)


def error_alignment_impl(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool,
                         batch_first: bool, ins_cost: float, del_cost: float, sub_cost: float
                         ) -> Tuple[Tensor, Tensor]:
    """Per pair the edit operations along the path ``error_counts_impl`` counts, ``(out, flags)``:
    int8 ``(R + H, N)`` (``(N, R + H)`` with ``batch_first``; 0 correct, 1 substitution,
    2 deletion, 3 insertion, -1 past the path's end) and the int32[1] warning flags, on the device
    of ``ref``."""
    return error_path_impl(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, True)


error_alignment = torch.library.custom_op("b200lev::error_alignment", error_alignment_impl,
                                          mutates_args=())


@error_alignment.register_fake
def _(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost):
    if batch_first:
        (_, R), (n, H) = ref.shape, hyp.shape
    else:
        (R, _), (H, n) = ref.shape, hyp.shape
    shape = (n, R + H) if batch_first else (R + H, n)
    return ref.new_empty(shape, dtype=torch.int8), ref.new_empty((1,), dtype=torch.int32)


# ---------------------------------------------------------------------------------------
# infix: the cheapest match of each reference anywhere inside its hypothesis
# ---------------------------------------------------------------------------------------
def infix_impl(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool, batch_first: bool,
               ins_cost: float, del_cost: float, sub_cost: float, norm: bool, spans: bool
               ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """One ``b200lev_infix`` call, ``(dist, start, end, flags)``: fp32 ``(N,)``, the int64 ``(N,)``
    match bounds (``(0,)`` unless ``spans``) and the int32[1] warning flags, on the device of
    ``ref``."""
    _, _, n = _shapes(ref, hyp, batch_first, 1)
    ref, hyp = _as_tokens(ref), _as_tokens(hyp)
    pl = _host.Placement(ref, hyp)
    ref, hyp, dev = pl.to_dev(ref), pl.to_dev(hyp), pl.dev
    L = _abi.lib()
    with _DeviceGuard(dev):
        rt, ht = _tok_struct(ref, batch_first), _tok_struct(hyp, batch_first)
        o = _opts(eos, include_eos, ins_cost, del_cost, sub_cost, norm, False, 0, False, 1)
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        nbytes = L.b200lev_workspace_bytes(ctypes.byref(rt), ctypes.byref(ht), 0, 0)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        dist = torch.empty(n, dtype=torch.float32, device=dev)
        start = torch.empty(n if spans else 0, dtype=torch.long, device=dev)
        end = torch.empty(n if spans else 0, dtype=torch.long, device=dev)
        _abi.check(L.b200lev_infix(ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o), dist.data_ptr(),
                                   start.data_ptr() if spans else None, end.data_ptr() if spans else None,
                                   ws.data_ptr(), nbytes, flags.data_ptr(), _stream(dev)))
    return pl.back(dist), pl.back(start), pl.back(end), pl.back(flags)


infix = torch.library.custom_op("b200lev::infix", infix_impl, mutates_args=())


@infix.register_fake
def _(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, norm, spans):
    n = hyp.shape[0] if batch_first else hyp.shape[1]
    m = n if spans else 0
    return (ref.new_empty((n,), dtype=torch.float32), ref.new_empty((m,), dtype=torch.long),
            ref.new_empty((m,), dtype=torch.long), ref.new_empty((1,), dtype=torch.int32))


# ---------------------------------------------------------------------------------------
# pairwise: every reference of a group against every hypothesis of it; minimum Bayes risk
# ---------------------------------------------------------------------------------------
def _pairwise_shapes(ref: Tensor, hyp: Tensor, batch_first: bool) -> Tuple[int, int, int]:
    """``(G, A, B)`` of ``ref`` ``(R, G, A)`` and ``hyp`` ``(H, G, B)`` (``(G, A, R)`` and
    ``(G, B, H)`` with ``batch_first``)."""
    if ref.dim() != 3 or hyp.dim() != 3:
        raise RuntimeError("ref and hyp must be 3 dimensional")
    if batch_first:
        (G, A, _), (Gh, B, _) = ref.shape, hyp.shape
    else:
        (_, G, A), (_, Gh, B) = ref.shape, hyp.shape
    if G != Gh:
        raise RuntimeError("ref and hyp group dimensions must match")
    return G, A, B


def _flat_tokens(t: Tensor, batch_first: bool) -> Tensor:
    """The 3-D token tensor as the 2-D ``(T, G*K)`` (``(G*K, T)``) view the C ABI reads (a copy
    only when the group and member axes do not merge)."""
    if batch_first:
        return t.reshape(t.size(0) * t.size(1), t.size(2))
    return t.reshape(t.size(0), t.size(1) * t.size(2))


def _pairwise_device(ref: Tensor, hyp: Tensor, dev: torch.device, G: int, A: int, B: int,
                     eos: Optional[int], include_eos: bool, batch_first: bool, ins_cost: float,
                     del_cost: float, sub_cost: float, norm: bool, return_mistakes: bool
                     ) -> Tuple[Tensor, Tensor]:
    """Device tensors in, ``(out (G, A, B) fp32, flags)`` out: one ``b200lev_final_cross`` call."""
    out = torch.empty((G, A, B), dtype=torch.float32, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    if G * A * B == 0:
        return out, flags
    L = _abi.lib()
    # (the flattened tensors may be copies: held here until the kernels are enqueued, since the
    # token structs keep only their data pointers)
    ref2, hyp2 = _flat_tokens(ref, batch_first), _flat_tokens(hyp, batch_first)
    with _DeviceGuard(dev):
        rt = _tok_struct(ref2, batch_first)
        ht = _tok_struct(hyp2, batch_first)
        o = _opts(eos, include_eos, ins_cost, del_cost, sub_cost, norm, False, 0, return_mistakes, 1)
        nbytes = L.b200lev_final_cross_workspace_bytes(ctypes.byref(rt), ctypes.byref(ht), A, B,
                                                       ctypes.byref(o))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _abi.check(L.b200lev_final_cross(ctypes.byref(rt), ctypes.byref(ht), A, B, ctypes.byref(o),
                                         out.data_ptr(), ws.data_ptr(), nbytes, flags.data_ptr(),
                                         _stream(dev)))
    return out, flags


def pairwise_impl(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool, batch_first: bool,
                  ins_cost: float, del_cost: float, sub_cost: float, norm: bool, return_mistakes: bool
                  ) -> Tuple[Tensor, Tensor]:
    """``(out, flags)``: ``out[g, a, b]`` (fp32 ``(G, A, B)``) is ``string_matching`` of
    reference ``(g, a)`` against hypothesis ``(g, b)``, and the int32[1] warning flags, on the
    device of ``ref``."""
    G, A, B = _pairwise_shapes(ref, hyp, batch_first)
    ref, hyp = _as_tokens(ref), _as_tokens(hyp)
    pl = _host.Placement(ref, hyp)
    out, flags = _pairwise_device(pl.to_dev(ref), pl.to_dev(hyp), pl.dev, G, A, B, eos, include_eos,
                                  batch_first, ins_cost, del_cost, sub_cost, norm, return_mistakes)
    return pl.back(out), pl.back(flags)


pairwise = torch.library.custom_op("b200lev::pairwise", pairwise_impl, mutates_args=())


@pairwise.register_fake
def _(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, norm, return_mistakes):
    G, A, B = _pairwise_shapes(ref, hyp, batch_first)
    return ref.new_empty((G, A, B), dtype=torch.float32), ref.new_empty((1,), dtype=torch.int32)


def _mbr_shapes(log_probs: Tensor, hyp: Tensor, batch_first: bool) -> Tuple[int, int]:
    if log_probs.dim() != 2:
        raise RuntimeError("log_probs must be 2 dimensional")
    if hyp.dim() != 3:
        raise RuntimeError("hyp must be 3 dimensional")
    N, M = (hyp.size(0), hyp.size(1)) if batch_first else (hyp.size(1), hyp.size(2))
    if log_probs.size(0) != N or log_probs.size(1) != M:
        raise RuntimeError("ref and hyp batch_size and sample dimensions must match")
    if M < 1:
        raise RuntimeError(f"Batch must have at least one sample, got {M}")
    return N, M


def minimum_bayes_risk_impl(log_probs: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool,
                            batch_first: bool, norm: bool, ins_cost: float, del_cost: float,
                            sub_cost: float) -> Tuple[Tensor, Tensor, Tensor]:
    """``(best, risk, flags)``: int64 ``(N,)``, ``(N, M)`` in the dtype of ``log_probs`` and the
    int32[1] warning flags.  Two C calls: ``b200lev_final_cross`` of the hypotheses against
    themselves (error rates with ``norm``, edit distances without), then ``b200lev_mbr``."""
    N, M = _mbr_shapes(log_probs, hyp, batch_first)
    code = _float_code(log_probs)
    hyp = _as_tokens(hyp)
    pl = _host.Placement(log_probs, hyp)
    dev = pl.dev
    lp, hyp = pl.to_dev(log_probs.detach()), pl.to_dev(hyp)
    er, flags = _pairwise_device(hyp, hyp, dev, N, M, M, eos, include_eos, batch_first, ins_cost,
                                 del_cost, sub_cost, norm, norm)
    risk = torch.empty((N, M), dtype=lp.dtype, device=dev)
    best = torch.empty(N, dtype=torch.long, device=dev)
    if N > 0:
        with _DeviceGuard(dev):
            _abi.check(_abi.lib().b200lev_mbr(er.data_ptr(), lp.data_ptr(), code, N, M, lp.stride(0),
                                              lp.stride(1), risk.data_ptr(), best.data_ptr(), _stream(dev)))
    return pl.back(best), pl.back(risk), pl.back(flags)


minimum_bayes_risk = torch.library.custom_op("b200lev::minimum_bayes_risk", minimum_bayes_risk_impl,
                                             mutates_args=())


@minimum_bayes_risk.register_fake
def _(log_probs, hyp, eos, include_eos, batch_first, norm, ins_cost, del_cost, sub_cost):
    N, M = _mbr_shapes(log_probs, hyp, batch_first)
    return (log_probs.new_empty((N,), dtype=torch.long), log_probs.new_empty((N, M)),
            log_probs.new_empty((1,), dtype=torch.int32))


# ---------------------------------------------------------------------------------------
# optimal completion
# ---------------------------------------------------------------------------------------
def optimal_completion_impl(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool,
                            batch_first: bool, ins_cost: float, del_cost: float, sub_cost: float,
                            padding: int, exclude_last: bool) -> Tuple[Tensor, Tensor]:
    """``optimal_completion`` (_string.py:464-517): ``(targets, flags)`` with targets int64
    ``(H', N, U)`` or ``(N, H', U)``.  One host read of U, as the reference has at :511."""
    R, H, n = _shapes(ref, hyp, batch_first, 1)
    ref, hyp = _as_tokens(ref), _as_tokens(hyp)
    pl = _host.Placement(ref, hyp)
    ref, hyp, dev = pl.to_dev(ref), pl.to_dev(hyp), pl.dev
    L = _abi.lib()
    with _DeviceGuard(dev):
        rt, ht = _tok_struct(ref, batch_first), _tok_struct(hyp, batch_first)
        o = _opts(eos, include_eos, ins_cost, del_cost, sub_cost, False, exclude_last, padding,
                  False, 1)
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        umax = torch.zeros(1, dtype=torch.int32, device=dev)
        nbytes = L.b200lev_workspace_bytes(ctypes.byref(rt), ctypes.byref(ht), 1, int(exclude_last))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        st = _stream(dev)
        _abi.check(L.b200lev_completion_count(ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o),
                                              ws.data_ptr(), nbytes, umax.data_ptr(),
                                              flags.data_ptr(), st))
        U = int(umax.item())  # _string.py:511
        hout = max(H + (0 if exclude_last else 1), 1)  # _string.py:271-278
        if batch_first:  # _string.py:515-516
            out = torch.empty((n, hout, U), dtype=torch.long, device=dev)
            si, sn = U, hout * U
        else:
            out = torch.empty((hout, n, U), dtype=torch.long, device=dev)
            si, sn = n * U, U
        _abi.check(L.b200lev_completion_fill(ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o),
                                             ws.data_ptr(), nbytes, U, out.data_ptr(), si, sn, st))
    return pl.back(out), pl.back(flags)


optimal_completion = torch.library.custom_op("b200lev::optimal_completion", optimal_completion_impl,
                                             mutates_args=())


@optimal_completion.register_fake
def _(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, padding, exclude_last):
    if batch_first:
        n, H = hyp.shape
    else:
        H, n = hyp.shape
    U = torch.library.get_ctx().new_dynamic_size()
    hout = max(H + (0 if exclude_last else 1), 1)
    shape = (n, hout, U) if batch_first else (hout, n, U)
    return ref.new_empty(shape, dtype=torch.long), ref.new_empty((1,), dtype=torch.int32)


# ---------------------------------------------------------------------------------------
# OCD loss (forward / backward)
# ---------------------------------------------------------------------------------------
def _acc_dtype(t: Tensor) -> torch.dtype:
    return torch.float64 if t.dtype == torch.float64 else torch.float32


def _float_code(t: Tensor) -> int:
    try:
        return _FLOAT_CODES[t.dtype]
    except KeyError:
        raise RuntimeError(f"unsupported floating dtype {t.dtype}") from None


def _rowmajor_last(t: Tensor) -> Tensor:
    return t if t.stride(-1) == 1 or t.size(-1) <= 1 else t.contiguous()


def _check_weight(w: Optional[Tensor], V: int) -> None:
    # the kernels read weight[t] for every target t in [0, V)
    if w is not None and (w.dim() != 1 or w.size(0) != V):
        raise RuntimeError(f"weight tensor should be defined either for all {V} classes or no classes but "
                           f"got weight tensor of shape: {list(w.shape)}")


def _weight_on(w: Optional[Tensor], dev: torch.device, acc: torch.dtype) -> Optional[Tensor]:
    """The class weights as the kernels read them: in the accumulation dtype of the logits."""
    return None if w is None else w.detach().to(device=dev, dtype=acc).contiguous()


def ocd_loss_impl(logits: Tensor, targets: Tensor, weight: Optional[Tensor], ignore_index: int,
                  reduction: int, seq_axis: int) -> Tuple[Tensor, Tensor, Tensor]:
    """_string.py:1229-1251 given the optimal-completion targets.  Returns
    ``(loss, lse, denom)`` (lse/denom are saved for the backward).  A target outside [0, V)
    other than ``ignore_index`` raises IndexError, as cross_entropy does (_string.py:1232-1238):
    the kernel flags it, read back with one 4-byte D2H."""
    pl = _host.Placement(logits, targets)
    dev = pl.dev
    A, B, V = logits.shape
    U = targets.size(-1)
    _check_weight(weight, V)
    logits = _rowmajor_last(pl.to_dev(logits.detach()))
    targets = pl.to_dev(targets).contiguous()
    acc = _acc_dtype(logits)
    w = _weight_on(weight, dev, acc)
    per = torch.empty((A, B), dtype=acc, device=dev)
    lse = torch.empty((A, B), dtype=acc, device=dev)
    denom = torch.empty(max(B if seq_axis == 0 else A, 1), dtype=acc, device=dev)
    loss = torch.empty((), dtype=acc, device=dev)  # written by the reduction whenever it is returned
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_ocd_forward(
            logits.data_ptr(), _float_code(logits), A, B, V, logits.stride(0), logits.stride(1),
            targets.data_ptr(), U, targets.stride(0), targets.stride(1),
            None if w is None else w.data_ptr(), ignore_index, reduction, seq_axis,
            per.data_ptr(), lse.data_ptr(), denom.data_ptr(), loss.data_ptr(), flags.data_ptr(),
            _stream(dev)))
    if int(flags.item()) & _abi.FLAG_BAD_TARGET:
        bad = targets[(targets != ignore_index) & ((targets < 0) | (targets >= V))]
        raise IndexError(f"Target {int(bad[0])} is out of bounds.")
    out = per if reduction == 0 else loss
    return pl.back(out.to(logits.dtype)), pl.back(lse), pl.back(denom)


ocd_loss = torch.library.custom_op("b200lev::ocd_loss", ocd_loss_impl, mutates_args=())


@ocd_loss.register_fake
def _(logits, targets, weight, ignore_index, reduction, seq_axis):
    A, B, V = logits.shape
    _check_weight(weight, V)
    acc = _acc_dtype(logits)
    out = logits.new_empty((A, B) if reduction == 0 else ())
    return out, logits.new_empty((A, B), dtype=acc), logits.new_empty(
        (max(B if seq_axis == 0 else A, 1),), dtype=acc)


def ocd_loss_backward_impl(grad_out: Tensor, logits: Tensor, targets: Tensor, weight: Optional[Tensor],
                           ignore_index: int, reduction: int, seq_axis: int, lse: Tensor,
                           denom: Tensor) -> Tensor:
    pl = _host.Placement(logits, targets)
    dev = pl.dev
    A, B, V = logits.shape
    U = targets.size(-1)
    logits = _rowmajor_last(pl.to_dev(logits.detach()))
    targets = pl.to_dev(targets).contiguous()
    acc = _acc_dtype(logits)
    w = _weight_on(weight, dev, acc)
    go = grad_out.detach().to(device=dev, dtype=acc).contiguous()
    lse, denom = lse.to(dev), denom.to(dev)
    grad = torch.empty((A, B, V), dtype=logits.dtype, device=dev)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_ocd_backward(
            logits.data_ptr(), _float_code(logits), A, B, V, logits.stride(0), logits.stride(1),
            targets.data_ptr(), U, targets.stride(0), targets.stride(1),
            None if w is None else w.data_ptr(), ignore_index, reduction, seq_axis,
            lse.data_ptr(), denom.data_ptr(), go.data_ptr(), grad.data_ptr(), _stream(dev)))
    return pl.back(grad)


ocd_loss_backward = torch.library.custom_op("b200lev::ocd_loss_backward", ocd_loss_backward_impl,
                                            mutates_args=())


@ocd_loss_backward.register_fake
def _(grad_out, logits, targets, weight, ignore_index, reduction, seq_axis, lse, denom):
    return logits.new_empty(logits.shape)


def _ocd_setup(ctx, inputs, output):
    logits, targets, weight, ignore_index, reduction, seq_axis = inputs
    _, lse, denom = output
    ctx.save_for_backward(logits, targets, weight, lse, denom)
    ctx.args = (ignore_index, reduction, seq_axis)


def _ocd_backward(ctx, g_loss, g_lse, g_denom):
    logits, targets, weight, lse, denom = ctx.saved_tensors
    ignore_index, reduction, seq_axis = ctx.args
    grad = ocd_loss_backward(g_loss, logits, targets, weight, ignore_index, reduction, seq_axis,
                             lse, denom)
    return grad, None, None, None, None, None


ocd_loss.register_autograd(_ocd_backward, setup_context=_ocd_setup)


class _OcdEager(torch.autograd.Function):
    """Plain eager calls (see _MwerEager)."""

    @staticmethod
    def forward(ctx, logits, targets, weight, ignore_index, reduction, seq_axis):
        loss, lse, denom = ocd_loss_impl(logits, targets, weight, ignore_index, reduction, seq_axis)
        ctx.save_for_backward(logits, targets, weight, lse, denom)
        ctx.args = (ignore_index, reduction, seq_axis)
        return loss

    @staticmethod
    def backward(ctx, g):
        logits, targets, weight, lse, denom = ctx.saved_tensors
        ignore_index, reduction, seq_axis = ctx.args
        return (ocd_loss_backward_impl(g, logits, targets, weight, ignore_index, reduction, seq_axis, lse, denom),
                None, None, None, None, None)


def ocd_loss_eager(logits: Tensor, targets: Tensor, weight: Optional[Tensor], ignore_index: int,
                   reduction: int, seq_axis: int) -> Tensor:
    if wants_grad(logits):
        return _OcdEager.apply(logits, targets, weight, ignore_index, reduction, seq_axis)
    return ocd_loss_impl(logits, targets, weight, ignore_index, reduction, seq_axis)[0]


# ---------------------------------------------------------------------------------------
# sequence_log_probs, tensor path (_decoding.py:1516-1548)
# ---------------------------------------------------------------------------------------
def sequence_log_probs_impl(logits: Tensor, hyp: Tensor, eos: Optional[int]
                            ) -> Tuple[Tensor, Tensor, Tensor]:
    """``logits`` (outer, T, inner, V) float, ``hyp`` (outer, T, inner) int64, both contiguous.
    Returns ``(out (outer, inner), row_lse, len)``; the last two are saved for the backward."""
    pl = _host.Placement(logits, hyp)
    dev = pl.dev
    outer, T, inner, V = logits.shape
    logits, hyp = pl.to_dev(logits.detach()), pl.to_dev(hyp.detach())
    acc = _acc_dtype(logits)
    length = torch.empty(max(outer * inner, 1), dtype=torch.int32, device=dev)
    row_lp = torch.empty(max(outer * T * inner, 1), dtype=acc, device=dev)
    row_lse = torch.empty(max(outer * T * inner, 1), dtype=acc, device=dev)
    out = torch.zeros((outer, inner), dtype=logits.dtype, device=dev)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_seqlp_forward(
            logits.data_ptr(), _float_code(logits), outer, T, inner, V, hyp.data_ptr(),
            int(eos is not None), 0 if eos is None else int(eos), length.data_ptr(),
            row_lp.data_ptr(), row_lse.data_ptr(), out.data_ptr(), _stream(dev)))
    return pl.back(out), pl.back(row_lse), pl.back(length)


sequence_log_probs = torch.library.custom_op("b200lev::sequence_log_probs", sequence_log_probs_impl,
                                             mutates_args=())


@sequence_log_probs.register_fake
def _(logits, hyp, eos):
    outer, T, inner, _ = logits.shape
    acc = _acc_dtype(logits)
    return (logits.new_empty((outer, inner)),
            logits.new_empty((max(outer * T * inner, 1),), dtype=acc),
            logits.new_empty((max(outer * inner, 1),), dtype=torch.int32))


@torch.library.custom_op("b200lev::sequence_log_probs_backward", mutates_args=())
def sequence_log_probs_backward(grad_out: Tensor, logits: Tensor, hyp: Tensor, row_lse: Tensor,
                                length: Tensor) -> Tensor:
    pl = _host.Placement(logits, hyp)
    dev = pl.dev
    outer, T, inner, V = logits.shape
    logits, hyp = pl.to_dev(logits.detach()), pl.to_dev(hyp.detach())
    go = grad_out.detach().to(device=dev, dtype=logits.dtype).contiguous()
    row_lse, length = row_lse.to(dev), length.to(dev)
    grad = torch.empty_like(logits)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_seqlp_backward(
            logits.data_ptr(), _float_code(logits), outer, T, inner, V, hyp.data_ptr(),
            length.data_ptr(), row_lse.data_ptr(), go.data_ptr(), grad.data_ptr(), _stream(dev)))
    return pl.back(grad)


@sequence_log_probs_backward.register_fake
def _(grad_out, logits, hyp, row_lse, length):
    return logits.new_empty(logits.shape)


def _seqlp_setup(ctx, inputs, output):
    logits, hyp, _ = inputs
    _, row_lse, length = output
    ctx.save_for_backward(logits, hyp, row_lse, length)


def _seqlp_backward(ctx, g_out, g_lse, g_len):
    logits, hyp, row_lse, length = ctx.saved_tensors
    return sequence_log_probs_backward(g_out, logits, hyp, row_lse, length), None, None


sequence_log_probs.register_autograd(_seqlp_backward, setup_context=_seqlp_setup)


# ---------------------------------------------------------------------------------------
# ctc_greedy_search (_decoding.py:507-560)
# ---------------------------------------------------------------------------------------
def ctc_greedy_search_impl(logits: Tensor, in_lens: Optional[Tensor], blank: int, is_probs: bool
                           ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """``logits`` contiguous (outer, T, inner, V); ``in_lens`` int64 (outer*inner) or None.
    Returns ``(max_ (outer, inner), paths (outer, T, inner), out_lens (outer, inner), arg,
    row_lse, len)``; the last three are saved for the backward."""
    pl = _host.Placement(logits, in_lens)
    dev = pl.dev
    outer, T, inner, V = logits.shape
    logits = pl.to_dev(logits.detach())
    acc = _acc_dtype(logits)
    n, rows = max(outer * inner, 1), max(outer * T * inner, 1)
    arg = torch.empty(rows, dtype=torch.int64, device=dev)
    row_val = torch.empty(rows, dtype=acc, device=dev)
    row_lse = torch.empty(rows, dtype=acc, device=dev)
    length = torch.empty(n, dtype=torch.int32, device=dev)
    paths = torch.empty((outer, T, inner), dtype=torch.int64, device=dev)
    out_lens = torch.zeros((outer, inner), dtype=torch.int64, device=dev)
    max_ = torch.zeros((outer, inner), dtype=logits.dtype, device=dev)
    lens = None if in_lens is None else pl.to_dev(in_lens.detach()).to(torch.int64).contiguous()
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_ctc_greedy(
            logits.data_ptr(), _float_code(logits), outer, T, inner, V,
            0 if lens is None else lens.data_ptr(), int(blank), int(is_probs), arg.data_ptr(),
            row_val.data_ptr(), row_lse.data_ptr(), length.data_ptr(), paths.data_ptr(),
            out_lens.data_ptr(), max_.data_ptr(), _stream(dev)))
    return (pl.back(max_), pl.back(paths), pl.back(out_lens), pl.back(arg), pl.back(row_lse),
            pl.back(length))


ctc_greedy_search = torch.library.custom_op("b200lev::ctc_greedy_search", ctc_greedy_search_impl,
                                            mutates_args=())


@ctc_greedy_search.register_fake
def _(logits, in_lens, blank, is_probs):
    outer, T, inner, _ = logits.shape
    acc = _acc_dtype(logits)
    n, rows = max(outer * inner, 1), max(outer * T * inner, 1)
    return (logits.new_empty((outer, inner)), logits.new_empty((outer, T, inner), dtype=torch.int64),
            logits.new_empty((outer, inner), dtype=torch.int64), logits.new_empty((rows,), dtype=torch.int64),
            logits.new_empty((rows,), dtype=acc), logits.new_empty((n,), dtype=torch.int32))


def _ctc_setup(ctx, inputs, output):
    logits, _, _, is_probs = inputs
    _, _, _, arg, row_lse, length = output
    ctx.is_probs = is_probs
    ctx.save_for_backward(logits, arg, row_lse, length)


def _ctc_probs_backward(g_max: Tensor, probs: Tensor, arg: Tensor, length: Tensor) -> Tensor:
    """is_probs=True: max_ is the PRODUCT of the chosen probabilities over the valid steps
    (_decoding.py:527, 540-553).  Its gradient is torch's own, taken through that product on the
    chosen entries (zeros among them included) -- a handful of small torch ops, off the hot path."""
    outer, T, inner, V = probs.shape
    dev = probs.device
    with torch.enable_grad():
        x = probs.detach().requires_grad_(True)
        chosen = x.gather(3, arg.to(dev).view(outer, T, inner, 1)).squeeze(3)  # (outer, T, inner)
        steps = torch.arange(T, device=dev).view(1, T, 1)
        valid = steps < length.to(dev).view(outer, 1, inner)
        prod = chosen.masked_fill(~valid, 1.0).prod(1)  # (outer, inner)
        (grad,) = torch.autograd.grad(prod, x, g_max.to(device=dev, dtype=prod.dtype).view(outer, inner))
    return grad


def _ctc_backward(ctx, g_max, g_paths, g_lens, g_arg, g_lse, g_len):
    logits, arg, row_lse, length = ctx.saved_tensors
    outer, T, inner, _ = logits.shape
    if ctx.is_probs:
        return _ctc_probs_backward(g_max, logits, arg, length), None, None, None
    # d max_ / d logits = g * (onehot(arg max) - softmax) on the valid steps: the same kernel as
    # sequence_log_probs' backward with the greedy path as the hypothesis
    return (sequence_log_probs_backward(g_max, logits, arg.view(outer, T, inner), row_lse, length),
            None, None, None)


ctc_greedy_search.register_autograd(_ctc_backward, setup_context=_ctc_setup)


# ---------------------------------------------------------------------------------------
# MWER epilogue (forward / backward)
# ---------------------------------------------------------------------------------------
def mwer_loss_impl(er: Tensor, log_probs: Tensor, sub_avg: bool, reduction: int) -> Tensor:
    """_string.py:1463-1471 on the (N, M) error rates."""
    pl = _host.Placement(er, log_probs)
    dev = pl.dev
    N, M = log_probs.shape
    er = pl.to_dev(er.detach()).reshape(N, M).contiguous()
    lp = pl.to_dev(log_probs.detach())
    acc = _acc_dtype(lp)
    per = torch.empty((N, M), dtype=acc, device=dev)
    loss = torch.zeros((), dtype=acc, device=dev)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_mwer_forward(
            er.data_ptr(), lp.data_ptr(), _float_code(lp), N, M, lp.stride(0), lp.stride(1),
            int(sub_avg), reduction, per.data_ptr(), loss.data_ptr(), _stream(dev)))
    return pl.back(per if reduction == 0 else loss)


mwer_loss = torch.library.custom_op("b200lev::mwer_loss", mwer_loss_impl, mutates_args=())


@mwer_loss.register_fake
def _(er, log_probs, sub_avg, reduction):
    acc = _acc_dtype(log_probs)
    return log_probs.new_empty(log_probs.shape if reduction == 0 else (), dtype=acc)


def mwer_loss_backward_impl(grad_out: Tensor, er: Tensor, log_probs: Tensor, sub_avg: bool,
                            reduction: int) -> Tensor:
    pl = _host.Placement(er, log_probs)
    dev = pl.dev
    N, M = log_probs.shape
    er = pl.to_dev(er.detach()).reshape(N, M).contiguous()
    lp = pl.to_dev(log_probs.detach())
    acc = _acc_dtype(lp)
    go = grad_out.detach().to(device=dev, dtype=acc).contiguous()
    grad = torch.empty((N, M), dtype=lp.dtype, device=dev)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_mwer_backward(
            er.data_ptr(), lp.data_ptr(), _float_code(lp), N, M, lp.stride(0), lp.stride(1),
            int(sub_avg), reduction, go.data_ptr(), grad.data_ptr(), _stream(dev)))
    return pl.back(grad)


mwer_loss_backward = torch.library.custom_op("b200lev::mwer_loss_backward", mwer_loss_backward_impl,
                                             mutates_args=())


@mwer_loss_backward.register_fake
def _(grad_out, er, log_probs, sub_avg, reduction):
    return log_probs.new_empty(log_probs.shape)


def _mwer_setup(ctx, inputs, output):
    er, log_probs, sub_avg, reduction = inputs
    ctx.save_for_backward(er, log_probs)
    ctx.args = (sub_avg, reduction)


def _mwer_backward(ctx, g):
    er, log_probs = ctx.saved_tensors
    sub_avg, reduction = ctx.args
    # autograd flows only through log_probs: er is built from detached integers
    # (_string.py:186-187)
    return None, mwer_loss_backward(g, er, log_probs, sub_avg, reduction), None, None


mwer_loss.register_autograd(_mwer_backward, setup_context=_mwer_setup)


class _MwerEager(torch.autograd.Function):
    """The same forward / backward pair as the registered op, for plain eager calls: a
    registered op's autograd round trip costs ~150 us of host time per step, this ~30."""

    @staticmethod
    def forward(ctx, er, log_probs, sub_avg, reduction):
        ctx.save_for_backward(er, log_probs)
        ctx.args = (sub_avg, reduction)
        return mwer_loss_impl(er, log_probs, sub_avg, reduction)

    @staticmethod
    def backward(ctx, g):
        er, log_probs = ctx.saved_tensors
        return None, mwer_loss_backward_impl(g, er, log_probs, *ctx.args), None, None


def mwer_loss_eager(er: Tensor, log_probs: Tensor, sub_avg: bool, reduction: int) -> Tensor:
    if wants_grad(log_probs):
        return _MwerEager.apply(er, log_probs, sub_avg, reduction)
    return mwer_loss_impl(er, log_probs, sub_avg, reduction)


# ---------------------------------------------------------------------------------------
# fill_after_eos scan, bulk error sums, INT32 microbenchmark
# ---------------------------------------------------------------------------------------
def after_eos_mask_impl(tokens: Tensor, eos: int, dim: int) -> Tensor:
    """bool mask, True strictly after the first ``eos`` along ``dim`` (_string.py:41)."""
    pl = _host.Placement(tokens)
    dev = pl.dev
    nd = tokens.dim()
    if nd and not (-nd <= dim < nd):
        raise IndexError(f"Dimension out of range (expected to be in range of [{-nd}, {nd - 1}], "
                         f"but got {dim})")
    dim = dim % max(nd, 1)
    tok = pl.to_dev(tokens.detach())
    tok = tok.to(torch.long) if tok.dtype != torch.long else tok
    tok = tok.contiguous()
    shape = tok.shape
    T = shape[dim] if tok.dim() else 1
    outer = 1
    for s in shape[:dim]:
        outer *= s
    inner = 1
    for s in shape[dim + 1:]:
        inner *= s
    mask = torch.zeros(shape, dtype=torch.uint8, device=dev)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_after_eos_mask(tok.data_ptr(), outer, T, inner, int(eos),
                                                     mask.data_ptr(), _stream(dev)))
    return pl.back(mask.bool())


after_eos_mask = torch.library.custom_op("b200lev::after_eos_mask", after_eos_mask_impl,
                                         mutates_args=())


@after_eos_mask.register_fake
def _(tokens, eos, dim):
    return tokens.new_empty(tokens.shape, dtype=torch.bool)


def ragged_to_padded(flat: Tensor, offsets: Tensor, sel: Optional[Tensor], first: int, count: int, T: int,
                     eos: int, pad: int) -> Tensor:
    """``(count, T)`` token matrix: row u = utterance ``sel[u]`` (``first + u`` without
    ``sel``) of the flat corpus, then ``eos``, then ``pad`` (what command_line.py:1110-1121
    builds with pad_sequence).  ``flat`` int16/int32/int64, ``offsets`` int64, same device."""
    pl = _host.Placement(flat, offsets, sel)
    if pl.moved:
        raise _abi.B200LevError("ragged_to_padded: arguments must be CUDA tensors")
    dev = pl.dev
    if flat.dtype not in (torch.int16, torch.int32, torch.int64) or offsets.dtype != torch.int64:
        raise _abi.B200LevError("ragged_to_padded: flat must be int16/int32/int64 and offsets int64")
    if not (flat.is_contiguous() and offsets.is_contiguous() and (sel is None or sel.is_contiguous())):
        raise _abi.B200LevError("ragged_to_padded: arguments must be contiguous")
    if sel is not None and (sel.dtype != torch.int64 or sel.numel() != count):
        raise _abi.B200LevError("ragged_to_padded: sel must hold `count` int64 indices")
    if count < 0 or T < 1 or (sel is None and not (0 <= first and first + count <= offsets.numel() - 1)):
        raise _abi.B200LevError("ragged_to_padded: utterance range outside offsets")
    out = torch.empty((count, T), dtype=flat.dtype, device=dev)
    off_ptr = offsets.data_ptr() + (0 if sel is not None else 8 * first)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_ragged_to_padded(
            flat.data_ptr(), flat.element_size(), off_ptr, 0 if sel is None else sel.data_ptr(), count, T,
            int(eos), int(pad), out.data_ptr(), _stream(dev)))
    return out


def error_sums_impl(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool, batch_first: bool,
                    ins_cost: float, del_cost: float, sub_cost: float, norm: bool,
                    return_mistakes: bool, ref_group: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Bulk scoring (command_line.py:1124-1147 without the per-utterance host reads):
    ``(er, acc, flags)`` with ``er`` the per-pair values of ``string_matching`` and
    ``acc = [sum(er), sum(ref_lens), #pairs]`` in fp64 ON THE COMPUTE DEVICE, ready for a
    single all-reduce.  One C call (``b200lev_final_sums``); where the short-reference kernel
    serves it, one kernel."""
    R, H, n = _shapes(ref, hyp, batch_first, ref_group)
    ref, hyp = _as_tokens(ref), _as_tokens(hyp)
    pl = _host.Placement(ref, hyp)
    ref, hyp, dev = pl.to_dev(ref), pl.to_dev(hyp), pl.dev
    L = _abi.lib()
    with _DeviceGuard(dev):
        rt, ht = _tok_struct(ref, batch_first), _tok_struct(hyp, batch_first)
        o = _opts(eos, include_eos, ins_cost, del_cost, sub_cost, norm, False, 0,
                  return_mistakes, ref_group)
        # one zero fill for both: the totals, and behind them the warning flags (a step of a
        # strongly scaled scoring job is a few tens of microseconds: every launch counts)
        zeroed = torch.zeros(4, dtype=torch.float64, device=dev)
        acc = zeroed[:3]
        flags = zeroed[3:].view(torch.int32)[:1]
        nbytes = L.b200lev_workspace_bytes(ctypes.byref(rt), ctypes.byref(ht), 0, 0)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty(n, dtype=torch.float32, device=dev)
        st = _stream(dev)
        _abi.check(L.b200lev_final_sums(ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o),
                                        out.data_ptr(), ws.data_ptr(), nbytes, flags.data_ptr(),
                                        acc.data_ptr(), st))
    return pl.back(out), acc, pl.back(flags)


def _error_sums_op(ref: Tensor, hyp: Tensor, eos: Optional[int], include_eos: bool, batch_first: bool,
                   ins_cost: float, del_cost: float, sub_cost: float, norm: bool,
                   return_mistakes: bool, ref_group: int) -> Tuple[Tensor, Tensor, Tensor]:
    # (the returns of a registered op may not share storage: totals and flags are views of one
    # zero-filled block in the plain function)
    er, acc, flags = error_sums_impl(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                                     sub_cost, norm, return_mistakes, ref_group)
    return er, acc.clone(), flags.clone()


error_sums = torch.library.custom_op("b200lev::error_sums", _error_sums_op, mutates_args=())


@error_sums.register_fake
def _(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, norm,
      return_mistakes, ref_group):
    n = hyp.shape[0] if batch_first else hyp.shape[1]
    return (ref.new_empty((n,), dtype=torch.float32), ref.new_empty((3,), dtype=torch.float64),
            ref.new_empty((1,), dtype=torch.int32))


# ---------------------------------------------------------------------------------------
# N-best producers' step functions (_decoding.py:41-155, 1207-1283)
# ---------------------------------------------------------------------------------------
def _path_extend(pl, y_prev: Tensor, src: Optional[Tensor], lens_prev: Optional[Tensor], y_t: Tensor,
                 K: int, W: int) -> Tuple[Tensor, Tensor]:
    """Device tensors in and out: ``(y_next (S', N, W), lens_next (N, W))``."""
    dev = pl.dev
    S, N, Kp = y_prev.shape
    if S == 0:
        if lens_prev is not None and bool((lens_prev != 0).any()):
            raise RuntimeError("Invalid lengths for t=0")  # _decoding.py:135-136
        S_out = 1
    elif lens_prev is None:
        S_out = S + 1
    else:  # don't make y bigger unless we have to (_decoding.py:129-131): one host read
        S_out = S + 1 if int(lens_prev.max().item()) >= S else S
    y_next = torch.empty((S_out, N, W), dtype=torch.long, device=dev)
    lens_next = torch.empty((N, W), dtype=torch.long, device=dev)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_path_extend(
            y_prev.data_ptr() if S > 0 and y_prev.numel() else None, S, N, Kp,
            None if src is None else src.data_ptr(), None if lens_prev is None else lens_prev.data_ptr(),
            y_t.data_ptr(), K, W, S_out, y_next.data_ptr(), lens_next.data_ptr(), _stream(dev)))
    return y_next, lens_next


@torch.library.custom_op("b200lev::beam_search_advance", mutates_args=())
def beam_search_advance(log_probs_t: Tensor, width: int, log_probs_prev: Tensor, y_prev: Tensor,
                        y_prev_lens: Optional[Tensor]) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """``(y_next, y_next_lens, log_probs_next, next_src)`` of _decoding.py:41-155.  Shapes are
    checked by the caller (functional.beam_search_advance)."""
    pl = _host.Placement(log_probs_t, log_probs_prev, y_prev, y_prev_lens)
    dev = pl.dev
    N, Kp, V = log_probs_t.shape
    lpt = pl.to_dev(log_probs_t.detach())
    lpp = pl.to_dev(log_probs_prev.detach()).to(lpt.dtype)
    yp = pl.to_dev(y_prev.detach()).to(torch.long).contiguous()
    lens = None if y_prev_lens is None else pl.to_dev(y_prev_lens.detach()).to(torch.long).contiguous()
    K = min(width, Kp * V)
    lp_next = torch.empty((N, width), dtype=lpt.dtype, device=dev)
    next_src = torch.empty((N, width), dtype=torch.long, device=dev)
    y_t = torch.empty((N, width), dtype=torch.long, device=dev)
    with _DeviceGuard(dev):
        _abi.check(_abi.lib().b200lev_beam_topk(
            lpt.data_ptr(), _float_code(lpt), N, Kp, V, lpt.stride(0), lpt.stride(1), lpt.stride(2),
            lpp.data_ptr(), lpp.stride(0), lpp.stride(1), width, lp_next.data_ptr(), next_src.data_ptr(),
            y_t.data_ptr(), _stream(dev)))
    y_next, lens_next = _path_extend(pl, yp, next_src, lens, y_t, K, width)
    return pl.back(y_next), pl.back(lens_next), pl.back(lp_next), pl.back(next_src)


@beam_search_advance.register_fake
def _(log_probs_t, width, log_probs_prev, y_prev, y_prev_lens):
    N = log_probs_t.shape[0]
    S = y_prev.shape[0]
    S_out = S + 1 if y_prev_lens is None or S == 0 else torch.library.get_ctx().new_dynamic_size()
    return (y_prev.new_empty((S_out, N, width), dtype=torch.long), y_prev.new_empty((N, width), dtype=torch.long),
            log_probs_t.new_empty((N, width)), y_prev.new_empty((N, width), dtype=torch.long))


@torch.library.custom_op("b200lev::random_walk_advance", mutates_args=())
def random_walk_advance(log_probs_t: Tensor, log_probs_prev: Tensor, y_prev: Tensor,
                        y_prev_lens: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """``(y_next, log_probs_next)`` of _decoding.py:1207-1283.  The draw itself is torch's
    (``torch.multinomial`` on the compute device: the random stream is the reference's own, so a
    seeded run reproduces it); the path bookkeeping is the same kernel as the beam's."""
    pl = _host.Placement(log_probs_t, log_probs_prev, y_prev, y_prev_lens)
    dev = pl.dev
    N, V = log_probs_t.shape
    lpt = pl.to_dev(log_probs_t.detach())
    y_t = torch.multinomial(lpt.exp(), 1, True)  # (N, 1)   _decoding.py:1266
    lp_next = pl.to_dev(log_probs_prev.detach()) + lpt.gather(1, y_t).squeeze(1)
    yp = pl.to_dev(y_prev.detach()).to(torch.long).contiguous().unsqueeze(2)  # (S, N, 1)
    lens = None if y_prev_lens is None else pl.to_dev(y_prev_lens.detach()).to(torch.long).contiguous().unsqueeze(1)
    y_next, _ = _path_extend(pl, yp, None, lens, y_t.contiguous(), 1, 1)
    return pl.back(y_next.squeeze(2)), pl.back(lp_next)


@random_walk_advance.register_fake
def _(log_probs_t, log_probs_prev, y_prev, y_prev_lens):
    S, N = y_prev.shape
    S_out = S + 1 if y_prev_lens is None or S == 0 else torch.library.get_ctx().new_dynamic_size()
    return y_prev.new_empty((S_out, N), dtype=torch.long), log_probs_prev.new_empty((N,))


# ---------------------------------------------------------------------------------------
# eager fast path
# ---------------------------------------------------------------------------------------
def needs_dispatcher() -> bool:
    """The registered ops exist so that scripting / tracing / torch.compile see ONE opaque op
    per call.  In plain eager mode the dispatcher round trip (~20-30 us) is pure overhead next
    to kernels that take a few microseconds, so the ``*_impl`` bodies are called directly."""
    return torch.jit.is_tracing() or torch.compiler.is_compiling()


def wants_grad(t: Tensor) -> bool:
    return torch.is_grad_enabled() and t.requires_grad
