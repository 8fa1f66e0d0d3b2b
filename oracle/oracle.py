"""CPU oracle for the `pydrobert.torch._string` hot path -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product package
(``pydrobert-pytorch_b200/b200lev``) never does, and has no CPU fallback.

Parity status: PINNED -- see the header of ``lev_oracle.c`` and
``tests/test_oracle.py`` (golden fixtures generated from the unmodified reference by
``tests/golden/make_golden.py``, the reference's known-answer vectors, sclite).

"SM" below is ``/root/reference/src/pydrobert/torch/_string.py``.

The dynamic program lives in ``lev_oracle.c`` (plain C, fp32 where the reference is
fp32); this file is the ctypes binding plus numpy restatements of the thin wrappers
around it (SM:409-583) and of the two losses (SM:1188-1251, SM:1400-1472), the latter
in float64 so that they can referee two fp32 implementations.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from typing import Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "lev_oracle.c")
_SO = os.path.join(_HERE, "_build", "liblev_oracle.so")

FLAG_REF_NO_EOS = 1
FLAG_HYP_NO_EOS = 2
FLAG_EMPTY_REF = 4

MODE_FINAL, MODE_PREFIX, MODE_MASK = 0, 1, 2

INDEX_PAD_VALUE = -100  # config.py:55

_lib = None


def build(force: bool = False) -> str:
    """Compile lev_oracle.c -> oracle/_build/liblev_oracle.so (gcc, OpenMP, no fast-math)."""
    os.makedirs(os.path.dirname(_SO), exist_ok=True)
    if (
        not force
        and os.path.exists(_SO)
        and os.path.getmtime(_SO) >= os.path.getmtime(_SRC)
    ):
        return _SO
    cmd = [
        "gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off",
        "-fno-fast-math", "-std=c99", "-o", _SO, _SRC, "-lm",
    ]
    subprocess.run(cmd, check=True)
    return _SO


def lib():
    global _lib
    if _lib is None:
        so = _SO
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(_SRC):
            so = build()
        L = ctypes.CDLL(so)
        i64, p = ctypes.c_int64, ctypes.c_void_p
        L.lev_oracle_string_matching.restype = ctypes.c_int
        L.lev_oracle_string_matching.argtypes = [
            p, i64, i64, i64,  # ref, R, st, sn
            p, i64, i64, i64,  # hyp, H, st, sn
            i64, i64,  # N, ref_group
            ctypes.c_int, i64, ctypes.c_int,  # has_eos, eos, include_eos
            ctypes.c_float, ctypes.c_float, ctypes.c_float,
            ctypes.c_int, ctypes.c_int, ctypes.c_int, i64,  # norm, mode, exclude_last, padding
            ctypes.c_int, ctypes.c_int,  # return_mistakes, exact_del
            p, p, p, p, p,  # out, mask, ref_lens, hyp_lens, flags
        ]
        L.lev_oracle_completion.restype = i64
        L.lev_oracle_completion.argtypes = [p, i64, i64, i64, p, i64, i64, i64, i64, p]
        L.lev_oracle_num_threads.restype = ctypes.c_int
        _lib = L
    return _lib


def num_threads() -> int:
    return int(lib().lev_oracle_num_threads())


def use_all_cores() -> int:
    """Ask OpenMP for every core this process may run on (torchrun pins OMP_NUM_THREADS=1)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    lib().lev_oracle_set_threads(ctypes.c_int(n))
    return num_threads()


def _np_tokens(x) -> np.ndarray:
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    x = np.asarray(x)
    if x.dtype != np.int64:
        x = x.astype(np.int64)
    return x


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _is_integral(*costs) -> bool:
    return all(float(np.float32(c)) == round(float(np.float32(c))) for c in costs)


def string_matching(
    ref,
    hyp,
    eos: Optional[int],
    include_eos: bool,
    batch_first: bool,
    ins_cost: float,
    del_cost: float,
    sub_cost: float,
    norm: bool = False,
    return_mask: bool = False,
    return_prf_dsts: bool = False,
    exclude_last: bool = False,
    padding: int = INDEX_PAD_VALUE,
    return_mistakes: bool = False,
    ref_group: int = 1,
    exact_del: Optional[bool] = None,
):
    """SM:146-406.  Returns ``(out, flags, ref_lens, hyp_lens)``.

    ``out`` is float32 ``(N,)``, float32 ``(H', N)`` (``(N, H')`` if batch_first) or
    bool ``(H', R, N)``.  ``ref`` may hold ``N // ref_group`` columns.
    """
    assert not return_mask or not return_prf_dsts  # SM:164
    assert not exclude_last or (return_mask or return_prf_dsts)  # SM:165
    ref, hyp = _np_tokens(ref), _np_tokens(hyp)
    if ref.ndim != 2 or hyp.ndim != 2:
        raise RuntimeError("ref and hyp must be 2 dimensional")  # SM:166-167
    if batch_first:  # SM:181-183
        ref, hyp = ref.T, hyp.T
    R, Nr = ref.shape
    H, N = hyp.shape
    if Nr * ref_group != N:
        raise RuntimeError(f"ref has batch size {Nr * ref_group}, but hyp has {N}")  # SM:191-194
    if exact_del is None:
        exact_del = not _is_integral(ins_cost, del_cost, sub_cost)
    mode = MODE_MASK if return_mask else (MODE_PREFIX if return_prf_dsts else MODE_FINAL)
    Hout = 0 if mode == MODE_FINAL else H + (0 if exclude_last else 1)
    if mode == MODE_MASK:
        Hout = max(Hout, 1)  # SM:271-278: the prefix-0 mask is appended unconditionally
    out = mask = None
    if mode == MODE_FINAL:
        out = np.zeros((N,), np.float32)
    elif mode == MODE_PREFIX:
        out = np.zeros((Hout, N), np.float32)
    else:
        mask = np.zeros((Hout, R, N), np.uint8)
    ref_lens = np.zeros((N,), np.int64)
    hyp_lens = np.zeros((N,), np.int64)
    flags = ctypes.c_int(0)
    isz = ref.itemsize
    rc = lib().lev_oracle_string_matching(
        _ptr(ref), R, ref.strides[0] // isz if R else 0, ref.strides[1] // isz if Nr else 0,
        _ptr(hyp), H, hyp.strides[0] // isz if H else 0, hyp.strides[1] // isz if N else 0,
        N, ref_group,
        int(eos is not None), int(eos if eos is not None else 0), int(include_eos),
        float(ins_cost), float(del_cost), float(sub_cost),
        int(norm), mode, int(exclude_last), int(padding),
        int(return_mistakes), int(exact_del),
        _ptr(out), _ptr(mask), _ptr(ref_lens), _ptr(hyp_lens), ctypes.byref(flags),
    )
    if rc != 0:
        raise MemoryError("lev_oracle_string_matching failed")
    if mode == MODE_MASK:
        res = mask.astype(bool)
    elif mode == MODE_PREFIX and batch_first:
        res = np.ascontiguousarray(out.T)  # SM:387-388
    else:
        res = out
    return res, flags.value, ref_lens, hyp_lens


def error_rate(ref, hyp, eos=None, include_eos=False, norm=True, batch_first=False,
               ins_cost=1.0, del_cost=1.0, sub_cost=1.0, **kw):
    """SM:409-434"""
    return string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                           sub_cost, norm=norm, return_mistakes=True, **kw)[0]


def edit_distance(ref, hyp, eos=None, include_eos=False, norm=False, batch_first=False,
                  ins_cost=1.0, del_cost=1.0, sub_cost=1.0, **kw):
    """SM:437-461"""
    return string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                           sub_cost, norm=norm, **kw)[0]


def prefix_error_rates(ref, hyp, eos=None, include_eos=True, norm=True, batch_first=False,
                       ins_cost=1.0, del_cost=1.0, sub_cost=1.0,
                       padding=INDEX_PAD_VALUE, exclude_last=False, **kw):
    """SM:520-550"""
    return string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                           sub_cost, norm=norm, return_prf_dsts=True,
                           exclude_last=exclude_last, padding=padding,
                           return_mistakes=True, **kw)[0]


def prefix_edit_distances(ref, hyp, eos=None, include_eos=True, norm=False,
                          batch_first=False, ins_cost=1.0, del_cost=1.0, sub_cost=1.0,
                          padding=INDEX_PAD_VALUE, exclude_last=False, **kw):
    """SM:553-583"""
    return string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                           sub_cost, norm=norm, return_prf_dsts=True,
                           exclude_last=exclude_last, padding=padding,
                           return_mistakes=False, **kw)[0]


def completion_mask(ref, hyp, eos=None, include_eos=True, batch_first=False, ins_cost=1.0,
                    del_cost=1.0, sub_cost=1.0, exclude_last=False, **kw):
    """The `(H', R, N)` bool mask of SM:479-491 (never transposed, SM:348-355)."""
    return string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                           sub_cost, return_mask=True, exclude_last=exclude_last, **kw)[0]


def optimal_completion(ref, hyp, eos=None, include_eos=True, batch_first=False,
                       ins_cost=1.0, del_cost=1.0, sub_cost=1.0, padding=INDEX_PAD_VALUE,
                       exclude_last=False, **kw):
    """SM:464-517: `(H', N, U)` int64 (`(N, H', U)` if batch_first)."""
    mask = completion_mask(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                           sub_cost, exclude_last, **kw)
    ref = _np_tokens(ref)
    if batch_first:
        ref = ref.T
    Hout, R, N = mask.shape
    m8 = np.ascontiguousarray(mask.astype(np.uint8))
    isz = ref.itemsize
    st = ref.strides[0] // isz if R else 0
    sn = ref.strides[1] // isz if N else 0
    U = int(lib().lev_oracle_completion(_ptr(m8), Hout, R, N, _ptr(ref), st, sn,
                                        int(padding), 0, None))
    targets = np.full((Hout, N, U), padding, np.int64)
    if U > 0 and targets.size:
        lib().lev_oracle_completion(_ptr(m8), Hout, R, N, _ptr(ref), st, sn, int(padding),
                                    U, _ptr(targets))
    if batch_first:
        targets = np.ascontiguousarray(targets.transpose(1, 0, 2))
    return targets


def fill_after_eos(tokens, eos: int, dim: int = 0, fill=None, value=None):
    """SM:30-42: everything strictly after the first `eos` along `dim` becomes `fill`."""
    tokens = np.asarray(tokens.detach().cpu().numpy() if hasattr(tokens, "detach") else tokens)
    out = tokens if value is None else np.asarray(
        value.detach().cpu().numpy() if hasattr(value, "detach") else value)
    fill_ = float(eos) if fill is None else fill
    seen = np.cumsum((tokens == eos).astype(np.int64), axis=dim)
    seen = np.cumsum(np.minimum(seen, 1), axis=dim) > 1
    seen, out_b = np.broadcast_arrays(seen, out)
    res = out_b.copy()
    res[seen] = np.asarray(fill_).astype(res.dtype)
    return res


def _logsumexp(x: np.ndarray, axis: int) -> np.ndarray:
    m = np.max(x, axis=axis, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    return (m + np.log(np.sum(np.exp(x - m), axis=axis, keepdims=True))).squeeze(axis)


def hard_optimal_completion_distillation_loss(
    logits, ref, hyp, eos=None, include_eos=True, batch_first=False, ins_cost=1.0,
    del_cost=1.0, sub_cost=1.0, weight=None, reduction="mean", ignore_index=-2,
    grad_output=None,
) -> Tuple[np.ndarray, np.ndarray]:
    """SM:1188-1251 in float64.  Returns ``(loss, dloss/dlogits)``; for
    ``reduction='none'`` the gradient is taken for ``sum(loss * grad_output)``
    (``grad_output`` defaults to ones)."""
    lg = np.asarray(logits.detach().cpu().double().numpy() if hasattr(logits, "detach")
                    else logits).astype(np.float64)
    hyp_np = _np_tokens(hyp)
    if lg.ndim != 3:
        raise RuntimeError("logits must be 3 dimensional")  # SM:1205-1206
    if lg.shape[:-1] != hyp_np.shape:
        raise RuntimeError("first two dims of logits must match hyp shape")  # SM:1207-1208
    V = lg.shape[-1]
    if include_eos and eos is not None:  # SM:1209-1215
        if eos < 0 or eos >= V:
            raise RuntimeError(f"If include_eos=True, eos ({eos}) must be a class idx")
        if eos == ignore_index:
            raise RuntimeError(f"If include_eos=True, eos cannot equal ignore_index ({eos}")
    tg = optimal_completion(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                            sub_cost, padding=ignore_index, exclude_last=True)  # SM:1216-1228
    w = np.ones((V,), np.float64) if weight is None else np.asarray(
        weight.detach().cpu().numpy() if hasattr(weight, "detach") else weight
    ).astype(np.float64)
    valid = tg != ignore_index  # (A, B, U)
    cnt = valid.sum(2)  # (A, B)
    lse = _logsumexp(lg, 2)  # (A, B)
    tgc = np.where(valid, tg, 0)
    picked = np.take_along_axis(lg, tgc, axis=2)  # (A, B, U)
    wt = w[tgc] * valid
    # cross_entropy(reduction='none', weight) = w[t] * (lse - logit[t]), and 0 at ignore_index even
    # where the stand-in class 0 of an ignored slot has a -inf logit   SM:1232-1238
    per = np.where(valid, wt * (lse[..., None] - picked), 0.0).sum(2) / np.maximum(cnt, 1)  # SM:1239-1241
    seq_dim = 1 if batch_first else 0
    sm = np.exp(lg - lse[..., None])
    # d per / d logits = (sum_t w_t / cnt) * softmax - scatter(w_t / cnt)
    coef = wt.sum(2) / np.maximum(cnt, 1)
    gper = coef[..., None] * sm
    sc = np.zeros_like(lg)
    np.add.at(sc, (np.arange(lg.shape[0])[:, None, None], np.arange(lg.shape[1])[None, :, None],
                   tgc), wt / np.maximum(cnt, 1)[..., None])
    gper = gper - sc
    if reduction == "mean":  # SM:1242-1246
        denom = np.maximum((cnt > 0).sum(seq_dim), 1)
        nb = per.shape[1 - seq_dim]
        loss = (per.sum(seq_dim) / denom).mean()
        scale = np.expand_dims(1.0 / denom / nb, seq_dim)
        grad = gper * scale[..., None]
    elif reduction == "sum":
        loss = per.sum()
        grad = gper
    elif reduction == "none":
        loss = per
        go = np.ones_like(per) if grad_output is None else np.asarray(grad_output, np.float64)
        grad = gper * go[..., None]
    else:
        raise RuntimeError(f"'{reduction}' is not a valid value for reduction")  # SM:1250
    return loss, grad


def minimum_error_rate_loss(
    log_probs, ref, hyp, eos=None, include_eos=True, sub_avg=True, batch_first=False,
    norm=True, ins_cost=1.0, del_cost=1.0, sub_cost=1.0, reduction="mean",
    grad_output=None,
) -> Tuple[np.ndarray, np.ndarray]:
    """SM:1400-1472 with the softmax/reduction in float64.  Returns ``(loss, dloss/dlog_probs)``."""
    lp = np.asarray(log_probs.detach().cpu().double().numpy() if hasattr(log_probs, "detach")
                    else log_probs).astype(np.float64)
    ref, hyp = _np_tokens(ref), _np_tokens(hyp)
    if lp.ndim != 2:
        raise RuntimeError("log_probs must be 2 dimensional")
    if hyp.ndim != 3:
        raise RuntimeError("hyp must be 3 dimensional")
    if ref.ndim not in (2, 3):
        raise RuntimeError("ref must be 2 or 3 dimensional")
    if batch_first:  # SM:1423-1435
        N, M, H = hyp.shape
        if ref.ndim == 2:
            ref = np.repeat(ref[:, None, :], M, axis=1)
        if ref.shape[:2] != (N, M) or ref.shape[:2] != lp.shape:
            raise RuntimeError("ref and hyp batch_size and sample dimensions must match")
        ref2 = ref.reshape(N * M, -1)
        hyp2 = hyp.reshape(N * M, H)
    else:  # SM:1436-1448
        H, N, M = hyp.shape
        if ref.ndim == 2:
            ref = np.repeat(ref[:, :, None], M, axis=2)
        if ref.shape[1:] != (N, M) or ref.shape[1:] != lp.shape:
            raise RuntimeError("ref and hyp batch_size and sample dimensions must match")
        ref2 = ref.reshape(ref.shape[0], N * M)
        hyp2 = hyp.reshape(H, N * M)
    if M < 2:
        raise RuntimeError(f"Batch must have at least two samples, got {M}")
    er = error_rate(ref2, hyp2, eos, include_eos, norm, batch_first, ins_cost, del_cost,
                    sub_cost).astype(np.float64).reshape(N, M)  # SM:1451-1462
    if sub_avg:
        # the reference subtracts an fp32 mean; keep that rounding out of the referee
        er = er - er.mean(1, keepdims=True)
    z = lp - lp.max(1, keepdims=True)
    p = np.exp(z)
    p = p / p.sum(1, keepdims=True)
    per = er * p  # SM:1465
    if reduction == "mean":
        loss = per.mean()
        go = np.full_like(per, 1.0 / per.size)
    elif reduction == "sum":
        loss = per.sum()
        go = np.ones_like(per)
    elif reduction == "none":
        loss = per
        go = np.ones_like(per) if grad_output is None else np.asarray(grad_output, np.float64)
    else:
        raise RuntimeError(f"'{reduction}' is not a valid value for reduction")
    ge = go * er
    grad = p * (ge - (p * ge).sum(1, keepdims=True))
    return loss, grad


def sequence_log_probs(logits, hyp, dim=0, eos=None, grad_out=None):
    """float64 restatement of _sequence_log_probs_tensor (_decoding.py:1516-1548).

    ``logits`` (A*, T, B*, V), ``hyp`` (A*, T, B*) int.  A step counts if its token is in
    [0, V) (:1530) and it is not past the first eos (:1531-1544, the eos step counts).
    Returns the (A*, B*) sums (:1548); with ``grad_out`` also d(sum . grad_out)/d logits."""
    logits = np.asarray(logits, dtype=np.float64)
    hyp = np.asarray(hyp)
    nd = hyp.ndim
    if dim < -nd or dim > nd - 1:
        raise RuntimeError(
            "Dimension out of range (expected to be in range of [{}, {}], but "
            "got {})".format(-nd, nd - 1, dim))
    dim = (nd + dim) % nd
    V = logits.shape[-1]
    hyp_m = np.moveaxis(hyp, dim, 0)              # (T, rest...)
    z = np.moveaxis(logits, dim, 0)               # (T, rest..., V)
    T = hyp_m.shape[0]
    m = z.max(axis=-1, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    lse = m[..., 0] + np.log(np.exp(z - m).sum(axis=-1))
    ok = (hyp_m >= 0) & (hyp_m < V)
    if eos is not None:
        is_eos = hyp_m == eos
        seen_before = np.cumsum(is_eos, axis=0) - is_eos > 0   # an eos strictly before t
        ok &= ~seen_before
    tok = np.where(ok, hyp_m, 0)
    picked = np.take_along_axis(z, tok[..., None], axis=-1)[..., 0]
    lp = np.where(ok, picked - lse, 0.0)
    out = lp.sum(axis=0)
    if grad_out is None:
        return out
    g = np.asarray(grad_out, dtype=np.float64)
    soft = np.exp(z - lse[..., None])
    onehot = np.zeros_like(z)
    np.put_along_axis(onehot, tok[..., None], 1.0, axis=-1)
    gz = np.where(ok[..., None], g[None, ..., None] * (onehot - soft), 0.0)
    return out, np.moveaxis(gz, 0, dim)


def ctc_greedy_search(logits, in_lens=None, blank_idx=-1, batch_first=False, is_probs=False, grad_out=None):
    """float64 restatement of ctc_greedy_search (_decoding.py:507-560).

    Per step the arg max class (:531; first of equal maxima) of the log-softmax of ``logits``
    (``(T, N, V)``; ``(N, T, V)`` if ``batch_first``) -- of ``logits`` itself with ``is_probs``
    (:524-526); a step is kept unless it is blank or repeats the step before it (:532-534) or lies
    beyond ``in_lens`` (:536-540); kept classes are moved to the front of ``paths``, whose other
    positions keep the raw arg max (:546,555); ``max_`` = sum (product) of the maxima over the
    valid steps (:541-554).  With ``grad_out`` (logits only) also d(max_ . grad_out)/d logits =
    g (onehot(arg max) - softmax) on the valid steps -- the reference's own backward raises
    (its in-place masked_scatter_ invalidates the saved arg max)."""
    z = np.asarray(logits, dtype=np.float64)
    if z.ndim != 3:
        raise RuntimeError("logits must be 3-dimensional")
    V = z.shape[2]
    if blank_idx < -V or blank_idx > V - 1:
        raise RuntimeError(
            "Blank index out of range (expected to be in the range of "
            f"[-{V},{V-1}], but got {blank_idx})")
    blank = (blank_idx + V) % V
    if not batch_first:
        z = z.transpose(1, 0, 2)                       # (N, T, V)
    N, T, _ = z.shape
    arg = z.argmax(axis=2) if T else np.zeros((N, 0), dtype=np.int64)
    if is_probs:
        val = z.max(axis=2) if T else np.zeros((N, 0))
    else:
        m = z.max(axis=2, keepdims=True) if T else np.zeros((N, 0, 1))
        m = np.where(np.isfinite(m), m, 0.0)
        lse = m[..., 0] + np.log(np.exp(z - m).sum(axis=2))
        val = np.take_along_axis(z, arg[..., None], axis=2)[..., 0] - lse if T else np.zeros((N, 0))
    keep = arg != blank
    if T > 1:
        keep[:, 1:] &= arg[:, 1:] != arg[:, :-1]
    valid = np.ones((N, T), dtype=bool)
    if in_lens is not None:
        valid = np.arange(T)[None, :] < np.asarray(in_lens).reshape(N, 1)
        keep &= valid
    out_lens = keep.sum(axis=1).astype(np.int64)
    paths = arg.astype(np.int64).copy()
    for n in range(N):
        paths[n, :out_lens[n]] = arg[n][keep[n]]
    max_ = np.where(valid, val, 1.0).prod(axis=1) if is_probs else np.where(valid, val, 0.0).sum(axis=1)
    if not batch_first:
        paths = paths.T
    if grad_out is None:
        return max_, paths, out_lens
    if is_probs:
        raise RuntimeError("gradient restated for logits only")
    g = np.asarray(grad_out, dtype=np.float64).reshape(N, 1, 1)
    onehot = np.zeros_like(z)
    np.put_along_axis(onehot, arg[..., None], 1.0, axis=2)
    gz = np.where(valid[..., None], g * (onehot - np.exp(z - lse[..., None])), 0.0)
    if not batch_first:
        gz = gz.transpose(1, 0, 2)
    return max_, paths, out_lens, gz


def beam_search_advance(log_probs_t, width, log_probs_prev, y_prev, y_prev_lens=None):
    """_decoding.py:41-155 restated (numpy; test infrastructure).  Ties between equal candidate
    scores resolve to the lower flat index ``k * V + v`` (the reference leaves the order of ties
    to torch.topk).  The sum is formed in the arrays' dtype, as torch's add is.  Padding columns
    (fewer than ``width`` extensions) hold -inf / length 0 / source 0 / token 0."""
    lpt = np.asarray(log_probs_t)
    lpp = np.asarray(log_probs_prev).astype(lpt.dtype)
    y_prev = np.asarray(y_prev, dtype=np.int64)
    N, Kp, V = lpt.shape
    S = y_prev.shape[0]
    K = min(width, Kp * V)
    cand = (lpp[:, :, None] + lpt).astype(lpt.dtype).reshape(N, Kp * V)
    # descending by value (NaN greatest, as torch.topk), ascending by index among equals
    key = np.where(np.isnan(cand), np.inf, cand.astype(np.float64))
    isnan = np.isnan(cand)
    order = np.lexsort((np.arange(Kp * V)[None, :].repeat(N, 0), -key, ~isnan), axis=1)[:, :K]
    lp_next = np.take_along_axis(cand, order, 1)
    src = order // V
    y_t = order % V
    if y_prev_lens is None:
        lens = np.full((N, Kp), S, dtype=np.int64)
        S_out = S + 1
    else:
        lens = np.asarray(y_prev_lens, dtype=np.int64)
        if S == 0:
            if (lens != 0).any():
                raise RuntimeError("Invalid lengths for t=0")
            S_out = 1
        else:
            S_out = S + 1 if int(lens.max()) >= S else S
    y_next = np.zeros((S_out, N, width), dtype=np.int64)
    lens_next = np.zeros((N, width), dtype=np.int64)
    for n in range(N):
        for k in range(K):
            f = src[n, k]
            y_next[:S, n, k] = y_prev[:, n, f]
            if S_out > S:
                y_next[S, n, k] = y_t[n, k]  # cat([y_next, y_t]) leaves the token in the new row
            y_next[lens[n, f], n, k] = y_t[n, k]
            lens_next[n, k] = lens[n, f] + 1
    lp_out = np.full((N, width), -np.inf, dtype=lpt.dtype)
    lp_out[:, :K] = lp_next
    src_out = np.zeros((N, width), dtype=np.int64)
    src_out[:, :K] = src
    return y_next, lens_next, lp_out, src_out


def random_walk_advance(log_probs_t, log_probs_prev, y_prev, y_t, y_prev_lens=None):
    """_decoding.py:1207-1283 restated GIVEN the drawn tokens ``y_t`` (N,): the draw itself is
    torch.multinomial's."""
    lpt = np.asarray(log_probs_t)
    y_prev = np.asarray(y_prev, dtype=np.int64)
    y_t = np.asarray(y_t, dtype=np.int64)
    S, N = y_prev.shape
    lp_next = np.asarray(log_probs_prev) + lpt[np.arange(N), y_t]
    if S == 0:
        return y_t[None, :].copy(), lp_next
    if y_prev_lens is None:
        return np.concatenate([y_prev, y_t[None, :]], 0), lp_next
    lens = np.asarray(y_prev_lens, dtype=np.int64)
    y_next = np.concatenate([y_prev, y_t[None, :]], 0) if int(lens.max()) >= S else y_prev.copy()
    y_next[lens, np.arange(N)] = y_t
    return y_next, lp_next
