"""CPU restatement of error_alignment -- TEST INFRASTRUCTURE ONLY (tests/ and __graft_entry__.smoke()).

The loop of counts_oracle.error_counts with the op code of every cell's picked predecessor kept
instead of the counts carried (0 correct, 1 substitution, 2 deletion, 3 insertion; row 0 all
deletions, column 0 all insertions), then walked back from cell (h, r) of each pair.  The counts
oracle inherits the counts of the same predecessor the walk follows, so the op histogram of a
pair equals its error_counts by construction; tests/test_error_alignment.py checks that.

numpy, vectorised over the pairs (one step per DP cell, then one step per path position).
"""
import numpy as np

from counts_oracle import FLAG_HYP_NO_EOS, FLAG_REF_NO_EOS, _lengths

OPS = "CSDI"


def error_alignment(ref, hyp, eos=None, include_eos=False, batch_first=False, ins_cost=1.0,
                    del_cost=1.0, sub_cost=1.0, return_flags=False):
    """int8 (R + H, N) (or (N, R + H) with ``batch_first``): step k of pair n, -1 past the path's
    end; with ``return_flags`` also the missing-eos flags of counts_oracle.error_counts."""
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
    if ins == dl and dl == sb and sb > 0:  # SM:168-174
        ins = dl = sb = np.float32(1)
    r, ref_miss = _lengths(ref, eos, include_eos)
    h, hyp_miss = _lengths(hyp, eos, include_eos)
    flags = (FLAG_REF_NO_EOS if ref_miss else 0) | (FLAG_HYP_NO_EOS if hyp_miss else 0)
    code = np.empty((H + 1, R + 1, N), np.int8)
    code[0] = 2
    code[:, 0] = 3
    row = np.repeat((np.arange(R + 1, dtype=np.float32) * dl)[:, None], N, axis=1)
    for i in range(1, H + 1):
        ht = hyp[i - 1]
        new_row = np.empty_like(row)
        new_row[0] = row[0] + ins
        for j in range(1, R + 1):
            same = ref[j - 1] == ht
            ins_c = row[j] + ins  # SM:292
            sub_c = row[j - 1] + np.where(same, np.float32(0), sb)  # SM:293
            ps = ins_c >= sub_c  # SM:296
            c = np.where(ps, sub_c, ins_c)
            op = np.where(ps, np.where(same, 0, 1), 3)
            del_c = new_row[j - 1] + dl  # SM:308
            take = ~(del_c >= c)  # SM:309
            new_row[j] = np.where(take, del_c, c)
            code[i, j] = np.where(take, 2, op)
        row = new_row
    out = np.full((R + H, N), -1, np.int8)
    cols = np.arange(N)
    i, j = h.copy(), r.copy()
    steps = []  # the ops from (h, r) backwards
    while True:
        live = (i > 0) | (j > 0)
        if not live.any():
            break
        op = np.where(live, code[i, j, cols], -1)
        steps.append(op)
        i = i - ((op == 0) | (op == 1) | (op == 3))
        j = j - ((op == 0) | (op == 1) | (op == 2))
    if steps:
        back = np.stack(steps)  # back[t, n]: the op t steps before the end of pair n's path
        n_ops = (back >= 0).sum(0)
        for t in range(back.shape[0]):
            k = n_ops - 1 - t
            ok = k >= 0
            out[k[ok], cols[ok]] = back[t, ok]
    if batch_first:
        out = np.ascontiguousarray(out.T)
    return (out, flags) if return_flags else out


def histogram(ops, batch_first=False):
    """(N, 4) int64 counts of ops 0..3 per pair: what error_counts returns."""
    ops = np.asarray(ops)
    if not batch_first:
        ops = ops.T
    return np.stack([(ops == k).sum(1) for k in range(4)], 1).astype(np.int64)
