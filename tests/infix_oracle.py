"""CPU restatement of infix_edit_distance / infix_matches -- TEST INFRASTRUCTURE ONLY (tests/ and
__graft_entry__.smoke()).

The cost DP of ``oracle/lev_oracle.c::one_pair`` (SM:258-318, "SM" = src/pydrobert/torch/_string.py
of the reference) in its fp32 operation order, with one change: column 0 is 0 on every row, so an
alignment may leave it at any hypothesis position.  Per pair the minimum of column r over the rows
(row 0 included), the first row reaching it, and the start row carried along the path: column 0 of
row i starts at i, and among the predecessors that reach a cell's value exactly (diagonal, up,
deletion run origin) the largest start wins.  The fp32 deletion term min_k v[k] + (fl(j*d) -
fl(k*d)) of non-integral costs is kept by run origin, as the kernels keep it.  Uniform costs take
unit costs and a multiplier (SM:168-174); lengths and missing-eos flags as SM:195-228.

numpy, vectorised over the pairs (one step per DP cell); the identities that pin it to the
reference's edit_distance are in tests/test_infix.py.
"""
import numpy as np

from counts_oracle import FLAG_HYP_NO_EOS, FLAG_REF_NO_EOS, _lengths

FLAG_EMPTY_REF = 4


def _pick(a, sa, b, sb):
    """The start of min(a, b): the start of the smaller candidate, the larger start on a tie."""
    return np.where(a < b, sa, np.where(b < a, sb, np.maximum(sa, sb)))


def infix(ref, hyp, eos=None, include_eos=False, norm=False, batch_first=False, ins_cost=1.0,
          del_cost=1.0, sub_cost=1.0, return_flags=False):
    """``(dist, start, end)``: fp32 and int64 ``(N,)``; with ``return_flags`` also the OR of the
    missing-eos flags (only with include_eos, as SM:202-217) and FLAG_EMPTY_REF (norm and an
    empty reference)."""
    ref, hyp = np.asarray(ref).astype(np.int64), np.asarray(hyp).astype(np.int64)
    if ref.ndim != 2 or hyp.ndim != 2:
        raise RuntimeError("ref and hyp must be 2 dimensional")
    if batch_first:
        ref, hyp = ref.T, hyp.T
    R, N = ref.shape
    H, N2 = hyp.shape
    if N != N2:
        raise RuntimeError(f"ref has batch size {N}, but hyp has {N2}")
    ins, dl, sb = np.float32(ins_cost), np.float32(del_cost), np.float32(sub_cost)
    mult = np.float32(1)
    if ins == dl and dl == sb and sb > 0:  # SM:168-174
        mult = ins
        ins = dl = sb = np.float32(1)
    exact_del = not all(float(c).is_integer() for c in (ins, dl, sb))
    r, ref_miss = _lengths(ref, eos, include_eos)
    h, hyp_miss = _lengths(hyp, eos, include_eos)
    flags = (FLAG_REF_NO_EOS if ref_miss else 0) | (FLAG_HYP_NO_EOS if hyp_miss else 0)
    if norm and (r == 0).any():
        flags |= FLAG_EMPTY_REF
    cols = np.arange(N)
    jd = np.arange(R + 1, dtype=np.float32) * dl  # SM:258-263
    row = np.repeat(jd[:, None], N, axis=1)
    st = np.zeros((R + 1, N), np.int64)
    best = row[r, cols].copy()
    end = np.zeros(N, np.int64)
    start = np.zeros(N, np.int64)
    zero = np.zeros(N, np.float32)
    for i in range(1, H + 1):
        ht = hyp[i - 1]
        new = np.empty_like(row)
        nst = np.empty_like(st)
        new[0] = zero  # column 0: a match may start here
        nst[0] = i
        ob, oj, os = zero, np.float32(0), np.full(N, i, np.int64)  # the deletion run origin
        for j in range(1, R + 1):
            a = row[j] + ins  # SM:292
            b = row[j - 1] + np.where(ref[j - 1] != ht, sb, np.float32(0))  # SM:293
            t = np.where(a < b, a, b)
            ts = _pick(a, st[j], b, st[j - 1])
            if exact_del:  # SM:263-266, 317 by run origin
                cand = ob + (jd[j] - oj)
                fresh = ~(cand < t)
                new[j] = np.where(fresh, t, cand)
                nst[j] = _pick(cand, os, t, ts)
                ob = np.where(fresh, t, ob)
                oj = np.where(fresh, jd[j], oj)
                os = np.where(fresh, nst[j], os)
            else:
                left = new[j - 1] + dl
                new[j] = np.where(left < t, left, t)
                nst[j] = _pick(left, nst[j - 1], t, ts)
        row, st = new, nst
        val = row[r, cols]
        better = (i <= h) & (val < best)
        best = np.where(better, val, best)
        end = np.where(better, i, end)
        start = np.where(better, st[r, cols], start)
    dist = (best * mult).astype(np.float32)
    if norm:  # SM:390-405; an empty reference matches the empty stretch
        dist = np.where(r > 0, dist / np.where(r > 0, r, 1).astype(np.float32), np.float32(0))
    dist = dist.astype(np.float32)
    return (dist, start, end, flags) if return_flags else (dist, start, end)
