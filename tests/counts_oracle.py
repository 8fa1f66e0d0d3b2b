"""CPU restatement of error_counts -- TEST INFRASTRUCTURE ONLY (tests/ and __graft_entry__.smoke()).

Per pair the correct / substitution / deletion / insertion counts along the path the count mode
of ``_string_matching`` takes (SM:292-314, "SM" = src/pydrobert/torch/_string.py of the
reference): the loop of ``oracle/lev_oracle.c::one_pair``'s count mode, with the four counts of
the picked predecessor carried instead of the mistake count.  Uniform costs take the same cell
with unit costs (SM:168-174).  Lengths and missing-eos flags as SM:195-228.

numpy, vectorised over the pairs (one step per DP cell), fp32 where the reference is fp32; the
identities that pin it to the reference's stored outputs are in tests/test_error_counts.py.
"""
import numpy as np

FLAG_REF_NO_EOS, FLAG_HYP_NO_EOS = 1, 2
_E = np.eye(4, dtype=np.int64)  # one op: 0 correct, 1 substitution, 2 deletion, 3 insertion


def _lengths(tok, eos, include_eos):
    """SM:195-228: first eos (or T), +1 with include_eos when there is one; and 'some sequence
    has no eos' for the include_eos warning."""
    T, N = tok.shape
    if eos is None:
        return np.full(N, T, np.int64), False
    hit = tok == eos
    if T == 0:
        first = np.zeros(N, np.int64)
    else:
        first = np.where(hit.any(0), hit.argmax(0), T).astype(np.int64)
    if include_eos:
        return np.where(first < T, first + 1, first), bool((first == T).any())
    return first, False


def error_counts(ref, hyp, eos=None, include_eos=False, batch_first=False, ins_cost=1.0,
                 del_cost=1.0, sub_cost=1.0, return_flags=False):
    """(N, 4) int64 (correct, substitutions, deletions, insertions); with ``return_flags`` also
    the OR of FLAG_REF_NO_EOS / FLAG_HYP_NO_EOS (only raised with include_eos, as SM:202-217)."""
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
    cols = np.arange(N)
    # row 0: j deletions
    row = np.repeat((np.arange(R + 1, dtype=np.float32) * dl)[:, None], N, axis=1)
    cnt = np.zeros((R + 1, N, 4), np.int64)
    cnt[:, :, 2] = np.arange(R + 1)[:, None]
    out = cnt[r, cols].copy()  # pairs with h == 0
    for i in range(1, H + 1):
        ht = hyp[i - 1]
        new_row = np.empty_like(row)
        new_cnt = np.empty_like(cnt)
        new_row[0] = row[0] + ins  # column 0: an insertion
        new_cnt[0] = cnt[0] + _E[3]
        for j in range(1, R + 1):
            same = ref[j - 1] == ht
            neq = np.where(same, np.float32(0), np.float32(1))
            ins_c = row[j] + ins  # SM:292
            sub_c = row[j - 1] + sb * neq  # SM:293
            ps = ins_c >= sub_c  # SM:296-301: correct / substitution, else insertion
            c = np.where(ps, sub_c, ins_c)
            m = np.where(ps[:, None], cnt[j - 1] + np.where(same[:, None], _E[0], _E[1]), cnt[j] + _E[3])
            del_c = new_row[j - 1] + dl  # SM:308
            take = ~(del_c >= c)  # SM:309-313: deletion
            new_row[j] = np.where(take, del_c, c)
            new_cnt[j] = np.where(take[:, None], new_cnt[j - 1] + _E[2], m)
        row, cnt = new_row, new_cnt
        done = h == i
        out[done] = cnt[r[done], cols[done]]
    return (out, flags) if return_flags else out
