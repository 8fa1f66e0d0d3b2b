// lev_dp.cu -- K1: warp-per-pair anti-diagonal wavefront for the Levenshtein DP.
//
// Replaces the Python hot loop SM:258-318 and the epilogues SM:340-406 of the
// reference ("SM" = src/pydrobert/torch/_string.py).
//
// Geometry.  DP columns 0..r (r = valid reference length) are cut into strips of
// W = 32*C columns, RIGHT-aligned so the last strip ends exactly at column r; the
// columns of the first strip that fall left of column 0 are "virtual" and hold +BIG,
// which makes column 0 (value i*ins) an ordinary cell and leaves no boundary special
// case.  Inside a strip lane l owns C adjacent columns in registers and the warp is
// skewed over hypothesis rows: at step s lane l updates row s-l, so the cells touched
// in one step lie on an anti-diagonal (of C-wide column blocks).  The previous
// diagonal lives in registers; the values a lane needs from its left neighbour (row
// i, last column of lane l-1) move with __shfl_up_sync once per step, and the
// matching diagonal value is simply last step's shuffle result.  Between strips the
// boundary column is handed over through a per-warp shared-memory column (written by
// lane 31 for row i, read by lane 0 of the next strip 31 steps earlier in its own
// schedule, so one buffer per channel suffices).
//
// Per cell the integer path issues 3 ALU-pipe instructions and one on the FMA pipe:
//   VIADDMNMX.U32 (token + negated row token clamped to 0 / 1 = "differs"), IMAD (diag +
//   differs * sub), VIADDMNMX (min(up+ins, .)), VIADDMNMX (min(left+del, .))
//                                           -- the DPX fused add+min of sm_90+/sm_100.
//
// Modes: FINAL (one value per pair), PREFIX (value at column r after every row),
// MASK (row minima in pass A, equality bits in pass B; bits are set per DISTINCT
// reference token so the compaction of SM:492-517 becomes a bit enumeration).
// Arithmetic: int32 for integer costs (exact; converted to fp32 on store), fp32 for
// the rest, in the reference's operation order (including its deletion term
// min_k v[k] + (fl(j*d) - fl(k*d)), SM:263-266,317, tracked by run origin).
#include "lev_arith.cuh"
#include "lev_align.cuh"

// number of per-warp shared-memory columns (boundary channels + row minima)
template <typename V, bool COUNT, int MODE, bool OPS = false, bool SPAN = false>
struct LevBufs {
    static constexpr bool FLT_COST = !std::is_same<V, int>::value && !COUNT;
    // MASK: + row minima + the chained bitmap word handed from strip to strip; OPS: + insertions;
    // SPAN: + start rows of the cells (and, fp32, of the run origins)
    static constexpr int NB = (COUNT ? 2 : (FLT_COST ? 3 : 1)) + (MODE == LEV_MODE_MASK ? 2 : 0) + (OPS ? 1 : 0) +
                              (SPAN ? (FLT_COST ? 2 : 1) : 0);
};

// One pair on one warp.  PASS: 0 = the only pass (FINAL/PREFIX) or the row-minimum
// pass of MASK; 1 = the equality pass of MASK, one global atomicOr per flagged position;
// 2 = the equality pass for references with at most 32 distinct tokens: the row's bitmap is
// ONE word, OR-ed along the lane chain with the shuffle that also carries the boundary cell
// (and from strip to strip through a shared-memory column), and stored once per row by the
// last lane -- no atomics, no divergent branch per cell, and the largest set size (SM:510-511)
// falls out of the same word.  Returns that size (valid on lane 31).
// OPS (FINAL, COUNT only; b200lev_error_counts): one more int32 channel, the insertions along the
// path the count cell picks, carried like the count channel; the epilogue writes (C, S, D, I).
// TRACE (on top of OPS; b200lev_error_alignment, C = 8 or 4): every row's C choices of a lane as
// one uint16 / byte of 2-bit op codes (lev_align.cuh) into the pair's trace, and the epilogue
// writes the insertion count alone.
// INFIX (FINAL, cost cell; b200lev_infix): column 0 holds 0 on every row, so a path may leave it at
// any row; the owner of column r keeps the minimum of D[i][r] over the rows (row 0 included) and the
// first row reaching it, and the epilogue writes that minimum instead of D[h][r].
// SPAN (on top of INFIX): one more int32 channel, the start row of each cell's path (row i for column
// 0 of row i), carried like the insertions of OPS; among the predecessors that reach a cell's value
// exactly (diagonal, up, deletion run origin) the largest start wins.  The epilogue writes the start
// and end rows of the match.
// tokens that do not fit in int32 (B200LEV_FLAG_WIDE_TOKENS): read the caller's tensors
// directly and compare in 64 bits.  Slow (strided gathers) but exact; uniform per launch.
__device__ __forceinline__ int64_t lev_load_raw(const void* base, int elem_bytes, int64_t idx) {
    switch (elem_bytes) {
        case 8: return reinterpret_cast<const int64_t*>(base)[idx];
        case 4: return reinterpret_cast<const int32_t*>(base)[idx];
        case 2: return reinterpret_cast<const int16_t*>(base)[idx];
        default: return reinterpret_cast<const int8_t*>(base)[idx];
    }
}

// the start of a cell whose value min(a, b) comes from candidates with starts sa, sb (SPAN)
template <typename V>
__device__ __forceinline__ int lev_span_pick(V a, int sa, V b, int sb) {
    return a < b ? sa : (b < a ? sb : (sa > sb ? sa : sb));
}

template <typename V, bool COUNT, int MODE, int C, int PASS, bool WIDE, bool OPS, bool TRACE = false,
          bool INFIX = false, bool SPAN = false>
__device__ __forceinline__ int lev_warp_pair(const LevParams& p, const int pair, const int r,
                                              const int h, const int steps,
                                              const int* __restrict__ hyp_s_,
                                              V* __restrict__ bufs, const int Hs) {
    typedef typename std::conditional<WIDE, int64_t, int>::type Tok;
    const Tok* __restrict__ hyp_s = reinterpret_cast<const Tok*>(hyp_s_);
    constexpr bool IS_INT = std::is_same<V, int>::value;
    constexpr bool FLT_COST = !IS_INT && !COUNT;
    constexpr bool RMIN = (MODE == LEV_MODE_MASK && PASS == 0);
    constexpr bool EQ = (MODE == LEV_MODE_MASK && PASS == 1);
    constexpr bool EQC = (MODE == LEV_MODE_MASK && PASS == 2);
    constexpr int W = 32 * C;
    int set_max = 0;  // EQC: largest number of distinct next tokens over the rows (lane 31)
    const int lane = threadIdx.x & 31;
    const int S = (r + W) / W;  // ceil((r + 1) / W)
    const int refcol = pair / p.ref_group;
    const int32_t* __restrict__ rtok = p.ref_tok + (int64_t)refcol * p.Rp;
    const V BIG = LevArith<V>::big();
    const V insc = LevArith<V>::ins(p), delc = LevArith<V>::del(p), subc = LevArith<V>::sub(p);
    // shared-memory columns, all indexed [32 + row]
    V* __restrict__ bnd_v = bufs;
    V* __restrict__ bnd_a = bufs + Hs;      // COUNT: counts ; FLT_COST: run-origin value
    V* __restrict__ bnd_b = bufs + 2 * Hs;  // FLT_COST: fl(origin * del)
    V* __restrict__ rowmin = bufs + (LevBufs<V, COUNT, MODE>::NB - 2) * Hs;  // MASK only
    unsigned* __restrict__ bitcol = reinterpret_cast<unsigned*>(bufs + (LevBufs<V, COUNT, MODE>::NB - 1) * Hs);
    int* __restrict__ bnd_i = reinterpret_cast<int*>(bufs + 2 * Hs);  // OPS: insertions
    int* __restrict__ bnd_s = reinterpret_cast<int*>(bufs + (FLT_COST ? 3 : 1) * Hs);  // SPAN: starts
    int* __restrict__ bnd_os = reinterpret_cast<int*>(bufs + 4 * Hs);  // SPAN, fp32: run-origin starts
    (void)bnd_a; (void)bnd_b; (void)rowmin; (void)bitcol; (void)bnd_i; (void)bnd_s; (void)bnd_os;
    // INFIX: the minimum over the rows of column r, the first row reaching it and (SPAN) its start
    V best = (V)0;
    int best_end = 0, best_start = 0;
    (void)best; (void)best_end; (void)best_start;

    for (int k = 0; k < S; ++k) {
        const bool first = (k == 0), last = (k == S - 1);
        const int jb = r - (S - k) * W;    // boundary column left of lane 0 (< 0 iff first)
        const int j0 = jb + lane * C + 1;  // this lane's first column
        V v[C];
        V m[C];     // COUNT: mistake counts
        int ic[C];  // OPS: insertions
        int sc[C];  // SPAN: start rows
        V jd[C];    // FLT_COST: fl(j * del), SM:258-263
        Tok rt[C];  // reference token of column j (ref position j-1)
        int ud[C];  // EQ: distinct-token rank of ref position j, or -1
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int j = j0 + c;
            v[c] = (j >= 0) ? (V)j * delc : BIG;
            m[c] = (V)(j >= 0 ? j : 0);  // SM:260
            ic[c] = 0;                   // row 0: deletions only
            sc[c] = 0;
            jd[c] = (j >= 0) ? (V)j * delc : (V)0;
            if (WIDE)
                rt[c] = (j >= 1) ? (Tok)lev_load_raw(p.ref_raw, p.ref_eb,
                                                      (int64_t)(j - 1) * p.ref_st + (int64_t)refcol * p.ref_sn)
                                 : (Tok)0;
            else
                rt[c] = (j >= 1) ? (Tok)rtok[j - 1] : (Tok)0;
            ud[c] = -1;
            if (EQ) ud[c] = (j >= 0 && j < r) ? p.uid[(int64_t)refcol * p.Rp + j] : -1;
            // EQC: the bit of this column's token (ranks < 32), 0 for columns that are no target
            if (EQC) ud[c] = (j >= 0 && j < r) ? (int)(1u << (p.uid[(int64_t)refcol * p.Rp + j] & 31)) : 0;
        }
        (void)m; (void)jd; (void)ud; (void)ic; (void)sc;
        if (INFIX && last) best = v[C - 1];  // D[0][r] (lane 31)
        const int zc = -j0;  // INFIX: this lane's column c that is column 0, if any
        (void)zc;
        unsigned bitrun = 0u;  // EQC chain register
        (void)bitrun;
        // chain registers: what this lane publishes to lane+1 at the next step
        V ob = BIG, oj = (V)0, rmrun = BIG;
        int os = 0;  // SPAN, fp32: start of the run origin
        (void)ob; (void)oj; (void)rmrun; (void)os;
        // previous step's hand-in (the diagonal); lane 0 starts from row 0 of the
        // boundary column, the other lanes pick it up from the shuffle at step l
        V pl_v = first ? BIG : (V)jb * delc;
        V pl_m = (V)(first ? 0 : jb);
        int pl_i = 0, pl_s = 0;
        (void)pl_m; (void)pl_i; (void)pl_s;
        if (steps > 0) {
            const int nsteps = steps + 31;
            for (int s = 1; s <= nsteps; ++s) {
                // ---- hand-over from the left neighbour (all lanes, every step) ----
                const V sh_v = __shfl_up_sync(LEV_FULL_MASK, v[C - 1], 1);
                const V in_v = (lane == 0) ? (first ? BIG : bnd_v[32 + s]) : sh_v;
                const V diag_v = pl_v;
                pl_v = in_v;
                V in_m = (V)0, diag_m = (V)0, in_ob = BIG, in_oj = (V)0, in_rm = BIG;
                if (COUNT) {
                    const V sh_m = __shfl_up_sync(LEV_FULL_MASK, m[C - 1], 1);
                    in_m = (lane == 0) ? (first ? (V)0 : bnd_a[32 + s]) : sh_m;
                    diag_m = pl_m;
                    pl_m = in_m;
                }
                int in_i = 0, diag_i = 0;
                if (OPS) {
                    const int sh_i = __shfl_up_sync(LEV_FULL_MASK, ic[C - 1], 1);
                    in_i = (lane == 0) ? (first ? 0 : bnd_i[32 + s]) : sh_i;
                    diag_i = pl_i;
                    pl_i = in_i;
                }
                (void)in_i; (void)diag_i;
                int in_s = 0, diag_s = 0, in_os = 0;
                if constexpr (SPAN) {
                    const int sh_s = __shfl_up_sync(LEV_FULL_MASK, sc[C - 1], 1);
                    in_s = (lane == 0) ? (first ? 0 : bnd_s[32 + s]) : sh_s;
                    diag_s = pl_s;
                    pl_s = in_s;
                    if (FLT_COST) {
                        const int sh_os = __shfl_up_sync(LEV_FULL_MASK, os, 1);
                        in_os = (lane == 0) ? (first ? 0 : bnd_os[32 + s]) : sh_os;
                    }
                }
                (void)in_s; (void)diag_s; (void)in_os;
                if (FLT_COST) {
                    const V sh_ob = __shfl_up_sync(LEV_FULL_MASK, ob, 1);
                    const V sh_oj = __shfl_up_sync(LEV_FULL_MASK, oj, 1);
                    in_ob = (lane == 0) ? (first ? BIG : bnd_a[32 + s]) : sh_ob;
                    in_oj = (lane == 0) ? (first ? (V)0 : bnd_b[32 + s]) : sh_oj;
                }
                if (RMIN) {
                    const V sh_rm = __shfl_up_sync(LEV_FULL_MASK, rmrun, 1);
                    in_rm = (lane == 0) ? (first ? BIG : rowmin[32 + s]) : sh_rm;
                }
                unsigned in_bits = 0u;
                if (EQC) {
                    const unsigned sh_b = __shfl_up_sync(LEV_FULL_MASK, bitrun, 1);
                    in_bits = (lane == 0) ? (first ? 0u : bitcol[32 + s]) : sh_b;
                }
                (void)in_m; (void)diag_m; (void)in_ob; (void)in_oj; (void)in_rm; (void)in_bits;
                const int i = s - lane;  // the row this lane updates now
                if (i >= 1 && i <= steps) {
                    const Tok ht = hyp_s[32 + i - 1];
                    if (COUNT) {
                        // SM:292-314: (cost, count); ties: sub over ins over del
                        V dc = diag_v, dm = diag_m, lc = in_v, lm = in_m;
                        int di = diag_i, li = in_i;
                        (void)di; (void)li;
                        unsigned tr = 0u;  // TRACE: this row's C choices
                        (void)tr;
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            const V uc = v[c], um = m[c];
                            // (integer cells, 32-bit tokens: "differs" from one DPX add-and-clamp, the cost and count terms by
                            // multiply / add instead of two selects)
                            const V neq01 = (IS_INT && !WIDE) ? (V)(int)__viaddmin_u32((unsigned)rt[c], 0u - (unsigned)ht, 1u)
                                                   : (rt[c] != ht ? (V)1 : (V)0);
                            const V sub_c = IS_INT ? dc + neq01 * subc : dc + (neq01 != (V)0 ? subc : (V)0);  // SM:293
                            const V ins_c = uc + insc;                 // SM:292
                            const bool ps = ins_c >= sub_c;            // SM:296
                            V cc = ps ? sub_c : ins_c;
                            V mm = ps ? dm + neq01 : um + (V)1;  // SM:299-301
                            const V del_c = lc + delc;                          // SM:308
                            const bool keep = del_c >= cc;                      // SM:309
                            cc = keep ? cc : del_c;
                            mm = keep ? mm : lm + (V)1;  // SM:311-313
                            if (OPS) {  // the insertion count of the predecessor picked, +1 for ins
                                const int ui = ic[c];
                                int ii = ps ? di : ui + 1;
                                ii = keep ? ii : li;
                                di = ui;
                                li = ii;
                                ic[c] = ii;
                            }
                            if constexpr (TRACE)
                                tr |= (keep ? (ps ? (neq01 != (V)0 ? 1u : 0u) : 3u) : 2u) << (2 * c);
                            dc = uc;
                            dm = um;
                            lc = cc;
                            lm = mm;
                            v[c] = cc;
                            m[c] = mm;
                        }
                        if constexpr (TRACE) {
                            typedef typename LevTraceStrips<C>::Field Field;
                            reinterpret_cast<Field*>(p.trace + (int64_t)pair * p.trace_pair_bytes)
                                [((int64_t)k * p.trace_steps + (s - 1)) * 32 + lane] = (Field)tr;
                        }
                    } else if (FLT_COST) {
                        // SM:290-293,316-317 in fp32, deletion term by run origin:
                        // new[j] = min(t[j], t[k*] + (fl(j*d) - fl(k* * d)))
                        V dg = diag_v, obr = in_ob, ojr = in_oj;
                        int sdg = diag_s, sob = in_os;
                        (void)sdg; (void)sob;
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            const V up = v[c];
                            const V a = up + insc;
                            const V sb = dg + ((rt[c] != ht) ? subc : (V)0);
                            const V t = a < sb ? a : sb;
                            const V cand = obr + (jd[c] - ojr);
                            const bool fresh = !(cand < t);
                            v[c] = fresh ? t : cand;
                            obr = fresh ? t : obr;
                            ojr = fresh ? jd[c] : ojr;
                            if constexpr (SPAN) {
                                const int ns = lev_span_pick(cand, sob, t, lev_span_pick(a, sc[c], sb, sdg));
                                sdg = sc[c];
                                sc[c] = ns;
                                sob = fresh ? ns : sob;
                            }
                            if (INFIX && c == zc) {  // column 0: a match may start at this row
                                v[c] = (V)0;
                                obr = (V)0;
                                ojr = jd[c];
                                if (SPAN) sc[c] = sob = i;
                            }
                            dg = up;
                        }
                        ob = obr;
                        oj = ojr;
                        os = sob;
                    } else {
                        // integer costs: 4 INT32 instructions per cell
                        int dg = (int)diag_v, lf = (int)in_v;
                        // (32-bit tokens: "differs" as 0 / 1 from one DPX add-and-clamp, times the
                        // cost on the FMA pipe -- 3 ALU-pipe instructions per cell; 64-bit tokens
                        // keep the compare)
                        const unsigned nht = 0u - (unsigned)ht;
                        (void)nht;
                        int sdg = diag_s, slf = in_s;
                        (void)sdg; (void)slf;
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            const int up = (int)v[c];
                            const int sb = WIDE ? dg + ((rt[c] != ht) ? (int)subc : 0)
                                                : dg + (int)(__viaddmin_u32((unsigned)rt[c], nht, 1u) * (unsigned)subc);
                            const int t = __viaddmin_s32(up, (int)insc, sb);
                            if constexpr (SPAN) {
                                const int st = lev_span_pick(up + (int)insc, sc[c], sb, sdg);
                                const int l = lf + (int)delc;
                                slf = lev_span_pick(l, slf, t, st);
                                sdg = sc[c];
                                lf = l < t ? l : t;
                            } else {
                                lf = __viaddmin_s32(lf, (int)delc, t);
                            }
                            if (INFIX && c == zc) {  // column 0: a match may start at this row
                                lf = 0;
                                if (SPAN) slf = i;
                            }
                            if (SPAN) sc[c] = slf;
                            dg = up;
                            v[c] = (V)lf;
                        }
                    }
                    if (RMIN) {  // SM:332-333: running minimum of row i over columns <= mine
                        V rm = in_rm;
#pragma unroll
                        for (int c = 0; c < C; ++c) rm = v[c] < rm ? v[c] : rm;
                        rmrun = rm;
                    }
                    if (EQ) {  // SM:334, 349-354
                        const V mn = rowmin[32 + i];
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            if (ud[c] >= 0 && v[c] == mn)
                                atomicOr(p.dbits + ((int64_t)i * p.P + pair) * p.Wd + (ud[c] >> 5),
                                         1u << (ud[c] & 31));
                        }
                    }
                    if (EQC) {  // the same test, branch-free, into the row's one-word bitmap
                        const V mn = rowmin[32 + i];
                        unsigned bits = in_bits;
#pragma unroll
                        for (int c = 0; c < C; ++c) bits |= v[c] == mn ? (unsigned)ud[c] : 0u;
                        bitrun = bits;
                    }
                    if (lane == 31) {
                        if (EQC) {
                            if (!last) {
                                bitcol[32 + i] = bitrun;
                            } else {
                                p.dbits[((int64_t)i * p.P + pair) * p.Wd] = bitrun;
                                const int cnt = __popc(bitrun);
                                set_max = cnt > set_max ? cnt : set_max;
                            }
                        }
                        if (!last) {
                            bnd_v[32 + i] = v[C - 1];
                            if (COUNT) bnd_a[32 + i] = m[C - 1];
                            if (OPS) bnd_i[32 + i] = ic[C - 1];
                            if (SPAN) bnd_s[32 + i] = sc[C - 1];
                            if (SPAN && FLT_COST) bnd_os[32 + i] = os;
                            if (FLT_COST) {
                                bnd_a[32 + i] = ob;
                                bnd_b[32 + i] = oj;
                            }
                        } else if (MODE == LEV_MODE_PREFIX) {  // SM:340-346
                            p.out[(int64_t)i * p.out_si + (int64_t)pair * p.out_sn] =
                                lev_finalize((float)(COUNT ? m[C - 1] : v[C - 1]), p, r, true);
                        } else if (INFIX && v[C - 1] < best) {  // the first row reaching the minimum
                            best = v[C - 1];
                            best_end = i;
                            if (SPAN) best_start = sc[C - 1];
                        }
                        if (RMIN) rowmin[32 + i] = rmrun;
                    }
                }
            }
        }
        if (OPS && last && lane == 31) {
            if constexpr (TRACE) {
                p.align_ins[pair] = ic[C - 1];
            } else {
                // m = S + D + I; C + S + D = r and C + S + I = h
                const int ins = ic[C - 1], del = ins + r - h, sub = (int)m[C - 1] - ins - del;
                int64_t* __restrict__ o = p.counts + (int64_t)pair * 4;
                o[0] = h - sub - ins;
                o[1] = sub;
                o[2] = del;
                o[3] = ins;
            }
        } else if (INFIX && last && lane == 31) {  // an empty reference matches the empty stretch: 0
            p.out[pair] = lev_finalize((float)best, p, r, false);
            if (SPAN) {
                p.infix_start[pair] = best_start;
                p.infix_end[pair] = best_end;
            }
        } else if (MODE == LEV_MODE_FINAL && last && lane == 31) {  // SM:390-405
            p.out[pair] = lev_finalize((float)(COUNT ? m[C - 1] : v[C - 1]), p, r, h > 0);
        }
        __syncwarp();
    }
    return set_max;
}

// Returns -1 when the largest target set still has to be counted from the bitmaps in global
// memory (atomic pass), else that size as lane 31 saw it (chained pass).
template <typename V, bool COUNT, int MODE, int C, bool WIDE = false, bool OPS = false, bool TRACE = false,
          bool INFIX = false, bool SPAN = false>
__device__ __forceinline__ int lev_warp_pair_all(const LevParams& p, int pair, int r, int h,
                                                 int steps, const int* hyp_s, V* bufs, int Hs,
                                                 bool one_word) {
    lev_warp_pair<V, COUNT, MODE, C, 0, WIDE, OPS, TRACE, INFIX, SPAN>(p, pair, r, h, steps, hyp_s, bufs, Hs);
    if (MODE == LEV_MODE_MASK) {
        if (one_word) return lev_warp_pair<V, COUNT, MODE, C, 2, WIDE, false>(p, pair, r, h, steps, hyp_s, bufs, Hs);
        lev_warp_pair<V, COUNT, MODE, C, 1, WIDE, false>(p, pair, r, h, steps, hyp_s, bufs, Hs);
    }
    return -1;
}

// CMASK: bit c set => the kernel carries a C = 2^c variant (1, 2, 4, 8); each pair
// takes the smallest variant whose single strip covers its r + 1 columns, the largest
// one (multi-strip) otherwise.  OPS: the error-counts epilogue (FINAL, COUNT).  TRACE: the
// error-alignment trace (with OPS; one C only, CMASK 8 or 4).  INFIX / SPAN: b200lev_infix (FINAL,
// cost cell).
template <typename V, bool COUNT, int MODE, int CMASK, bool OPS = false, bool TRACE = false, bool INFIX = false,
          bool SPAN = false>
__global__ void __launch_bounds__(256) lev_warp_kernel(const LevParams p) {
    LEV_DYN_SMEM(int, smem);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int wpc = blockDim.x >> 5;
    // (even: every warp's slice starts 8-byte aligned, the 64-bit-token path stores int64)
    const int Hs = (p.H + 65) & ~1;
    constexpr int NB = LevBufs<V, COUNT, MODE, OPS, SPAN>::NB;
    int* hyp_s = smem + (size_t)warp * (2 + NB) * Hs;  // 2*Hs ints: room for int64 tokens
    V* bufs = reinterpret_cast<V*>(hyp_s + 2 * Hs);
    const bool wide = (*p.wide_flag & B200LEV_FLAG_WIDE_TOKENS) != 0;
    if (p.only_if_wide && !wide) return;  // the group kernel already did the work
    if (p.bv_check && lev_bv_took(p.wide_flag)) return;
    const bool mask16 = MODE == LEV_MODE_MASK && p.mask16 && lev_mask16_tokens_ok(p.wide_flag);
    for (int pair = blockIdx.x * wpc + warp; pair < p.P; pair += gridDim.x * wpc) {
        if (mask16 && lev_mask16_takes(p, pair)) continue;  // lev_mask16_kernel's pair
        const int r = p.ref_len[pair / p.ref_group];
        const int h = p.hyp_len[pair];
        const int steps = p.exclude_last ? (h > 0 ? h - 1 : 0) : h;  // SM:286-288
        if (MODE != LEV_MODE_MASK && lane == 0 && r == 0 && p.norm && p.flags != nullptr)
            atomicOr(p.flags, B200LEV_FLAG_EMPTY_REF);  // SM:360-366, 397-404
        const int32_t* __restrict__ htok = p.hyp_tok + (int64_t)pair * p.Hp;
        if (wide) {
            int64_t* h64 = reinterpret_cast<int64_t*>(hyp_s);
            for (int i = lane; i < steps; i += 32)
                h64[32 + i] = lev_load_raw(p.hyp_raw, p.hyp_eb, (int64_t)i * p.hyp_st + (int64_t)pair * p.hyp_sn);
        } else {
            for (int i = lane; i < steps; i += 32) hyp_s[32 + i] = htok[i];
        }
        __syncwarp();
        const int cols = r + 1;
        // MASK: a reference with at most 32 distinct tokens keeps a row's bitmap in one word
        const bool one_word = MODE == LEV_MODE_MASK && p.ndist[pair / p.ref_group] <= 32;
        int set_max = -1;
        if (wide)
            set_max = lev_warp_pair_all<V, COUNT, MODE, (CMASK & 8) ? 8 : ((CMASK & 4) ? 4 : ((CMASK & 2) ? 2 : 1)), true, OPS, TRACE, INFIX, SPAN>(
                p, pair, r, h, steps, hyp_s, bufs, Hs, one_word);
        else if ((CMASK & 1) && (cols <= 32 || !(CMASK & 14)))
            set_max = lev_warp_pair_all<V, COUNT, MODE, 1, false, OPS, TRACE, INFIX, SPAN>(p, pair, r, h, steps, hyp_s, bufs, Hs, one_word);
        else if ((CMASK & 2) && (cols <= 64 || !(CMASK & 12)))
            set_max = lev_warp_pair_all<V, COUNT, MODE, 2, false, OPS, TRACE, INFIX, SPAN>(p, pair, r, h, steps, hyp_s, bufs, Hs, one_word);
        else if ((CMASK & 4) && (cols <= 128 || !(CMASK & 8)))
            set_max = lev_warp_pair_all<V, COUNT, MODE, 4, false, OPS, TRACE, INFIX, SPAN>(p, pair, r, h, steps, hyp_s, bufs, Hs, one_word);
        else if (CMASK & 8)
            set_max = lev_warp_pair_all<V, COUNT, MODE, 8, false, OPS, TRACE, INFIX, SPAN>(p, pair, r, h, steps, hyp_s, bufs, Hs, one_word);

        if (MODE == LEV_MODE_PREFIX) {
            // SM:279-285 (row 0) and SM:379-386 (tail := padding)
            const int first_pad = h + (p.exclude_last ? 0 : 1);
            if (lane == 0 && first_pad > 0 && p.Hout > 0) {
                const float v0 = COUNT ? (float)r : (float)((V)r * LevArith<V>::del(p));
                p.out[(int64_t)pair * p.out_sn] = lev_finalize(v0, p, r, false);
            }
            for (int i = first_pad + lane; i < p.Hout; i += 32)
                p.out[(int64_t)i * p.out_si + (int64_t)pair * p.out_sn] = p.padding;
        }
        if (MODE == LEV_MODE_MASK) {
            // SM:271-278: prefix 0 points at ref position 0 whenever the ref is non-empty
            if (lane == 0 && r > 0 && p.Hout > 0) {
                const int u = p.uid[(int64_t)(pair / p.ref_group) * p.Rp];
                atomicOr(p.dbits + (int64_t)pair * p.Wd + (u >> 5), 1u << (u & 31));
            }
            // SM:510-511: largest target set of this pair -> global maximum U
            int mx = 0;
            if (one_word) {  // lane 31 counted the rows' words as it stored them; row 0 holds one token
                mx = __shfl_sync(LEV_FULL_MASK, set_max, 31);
                if (r > 0 && p.Hout > 0 && mx < 1) mx = 1;
            } else {
                __threadfence();
                __syncwarp();
                for (int i = lane; i <= steps && i < p.Hout; i += 32) {
                    const uint32_t* row = p.dbits + ((int64_t)i * p.P + pair) * p.Wd;
                    int cnt = 0;
                    for (int w = 0; w < p.Wd; ++w) cnt += __popc(__ldcg(row + w));
                    mx = cnt > mx ? cnt : mx;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const int other = __shfl_xor_sync(LEV_FULL_MASK, mx, o);
                mx = other > mx ? other : mx;
            }
            if (lane == 0 && mx > 0) atomicMax(p.umax, mx);
        }
        __syncwarp();
    }
}

template <typename V, bool COUNT, int MODE, int CMASK, bool OPS = false, bool TRACE = false, bool INFIX = false,
          bool SPAN = false>
static int lev_launch_variant(const LevParams& p, cudaStream_t st) {
    constexpr int NB = LevBufs<V, COUNT, MODE, OPS, SPAN>::NB;
    const size_t per_warp = (size_t)(2 + NB) * (size_t)((p.H + 65) & ~1) * sizeof(int);
    const size_t budget = 200 * 1024;
    if (per_warp > budget) {
        lev_set_error("hypothesis length %d needs %zu bytes of shared memory per warp (max %zu)",
                      p.H, per_warp, budget);
        return B200LEV_ERR_UNSUPPORTED;
    }
    int wpc = (int)(budget / per_warp);
    if (wpc > 8) wpc = 8;
    // keep at least two CTAs per SM resident when the rows are short
    while (wpc > 1 && per_warp * wpc > 100 * 1024) --wpc;
    const size_t smem = per_warp * wpc;
    auto kern = lev_warp_kernel<V, COUNT, MODE, CMASK, OPS, TRACE, INFIX, SPAN>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem);
        if (e != cudaSuccess) {
            lev_set_error("cudaFuncSetAttribute(smem=%zu): %s", smem, cudaGetErrorString(e));
            return B200LEV_ERR_CUDA;
        }
    }
    int64_t blocks = ((int64_t)p.P + wpc - 1) / wpc;
    // stand-by launch behind the group kernel (runs only for >32-bit tokens): keep the
    // grid small so that the usual immediate exit costs next to nothing
    const int64_t cap = p.only_if_wide ? 148 * 4 : 148 * 64;
    if (blocks > cap) blocks = cap;
    const int slot = p.only_if_wide ? LEV_PROF_STANDBY : LEV_PROF_DP;
    lev_prof_begin(slot, st);
    lev_launch(kern, dim3((unsigned)blocks), dim3((unsigned)(32 * wpc)), smem, st, p);
    lev_prof_end(slot, st);
    return lev_check_cuda("lev_warp_kernel");
}

int lev_launch_dp(const LevParams& p_, int mode, bool count_mode, bool float_path,
                  cudaStream_t st) {
    if (p_.P <= 0) return B200LEV_OK;
    LevParams p = p_;
    p.only_if_wide = 0;
    p.mask16 = 0;
    if (mode == LEV_MODE_MASK) {
        // integer costs, r <= 255: the packed two-pairs-per-warp kernel first; the warp kernel
        // below takes what it leaves (per pair, decided on the device)
        const int took = lev_launch_mask16(p, float_path || count_mode, st);
        if (took < 0) return took;
        p.mask16 = took;
    }
    if (!float_path) {
        // large batches of short/mid pairs: length-bucketed group kernel (lev_group.cu);
        // this kernel then only runs if K0 flagged tokens wider than 32 bits
        const int took = lev_launch_group(p, mode, count_mode, st);
        if (took < 0) return took;
        if (took == 1) p.only_if_wide = 1;
    }
    if (!p.only_if_wide) {
        // few pairs or long rows: one CTA per pair, strips pipelined across warps (lev_cta.cu)
        const int took = lev_launch_cta(p, mode, count_mode, float_path, st);
        if (took < 0) return took;
        if (took == 1) p.only_if_wide = 1;
    }
    // the stand-by launch exists for tokens wider than int32: impossible below 8-byte elements
    if (p.only_if_wide && p.ref_eb < 8 && p.hyp_eb < 8) return B200LEV_OK;
    if (!float_path) {
        if (!count_mode) {
            if (mode == LEV_MODE_FINAL) return lev_launch_variant<int, false, LEV_MODE_FINAL, 15>(p, st);
            if (mode == LEV_MODE_PREFIX) return lev_launch_variant<int, false, LEV_MODE_PREFIX, 15>(p, st);
            return lev_launch_variant<int, false, LEV_MODE_MASK, 14>(p, st);
        }
        if (mode == LEV_MODE_FINAL) return lev_launch_variant<int, true, LEV_MODE_FINAL, 10>(p, st);
        if (mode == LEV_MODE_PREFIX) return lev_launch_variant<int, true, LEV_MODE_PREFIX, 10>(p, st);
    } else {
        if (!count_mode) {
            if (mode == LEV_MODE_FINAL) return lev_launch_variant<float, false, LEV_MODE_FINAL, 4>(p, st);
            if (mode == LEV_MODE_PREFIX) return lev_launch_variant<float, false, LEV_MODE_PREFIX, 4>(p, st);
            return lev_launch_variant<float, false, LEV_MODE_MASK, 4>(p, st);
        }
        if (mode == LEV_MODE_FINAL) return lev_launch_variant<float, true, LEV_MODE_FINAL, 4>(p, st);
        if (mode == LEV_MODE_PREFIX) return lev_launch_variant<float, true, LEV_MODE_PREFIX, 4>(p, st);
    }
    lev_set_error("mask mode is defined on the cost row only (SM:479-491)");
    return B200LEV_ERR_ARG;
}

// b200lev_error_alignment, the long form: K1 with the count cell, the insertion channel and the
// choice trace at one strip width, then the walk, one thread per pair
template <typename V, int C>
static int lev_launch_align_t(const LevParams& p, cudaStream_t st) {
    int rc = lev_launch_variant<V, true, LEV_MODE_FINAL, C, true, true>(p, st);
    if (rc) return rc;
    int64_t blocks = ((int64_t)p.P + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    lev_launch(lev_align_walk_kernel<C>, dim3((unsigned)blocks), dim3(256), 0, st, p);
    return lev_check_cuda("lev_align_walk_kernel");
}

// b200lev_error_counts / b200lev_error_alignment, references longer than the short form takes
// (lev_counts.cuh): K1 with the count cell and the insertion channel, after K0.  No group, CTA or
// bit-vector kernel: they carry no path.
int lev_launch_counts_dp(const LevParams& p, bool float_path, cudaStream_t st) {
    if (p.P <= 0) return B200LEV_OK;
    if (p.ops != nullptr) {
        if (!float_path) return lev_launch_align_t<int, LEV_ALIGN_C_INT>(p, st);
        return lev_launch_align_t<float, LEV_ALIGN_C_FLT>(p, st);
    }
    if (!float_path) return lev_launch_variant<int, true, LEV_MODE_FINAL, 10, true>(p, st);
    return lev_launch_variant<float, true, LEV_MODE_FINAL, 4, true>(p, st);
}

// b200lev_infix, everything but the distance-only calls Ks serves: K1 with column 0 pinned to 0 and
// the minimum over the rows of column r, after K0; `spans` adds the start channel.  No group, CTA or
// bit-vector kernel: none of them has the pinned column.
int lev_launch_infix_dp(const LevParams& p, bool float_path, bool spans, cudaStream_t st) {
    if (p.P <= 0) return B200LEV_OK;
    if (!float_path)
        return spans ? lev_launch_variant<int, false, LEV_MODE_FINAL, 15, false, false, true, true>(p, st)
                     : lev_launch_variant<int, false, LEV_MODE_FINAL, 15, false, false, true, false>(p, st);
    return spans ? lev_launch_variant<float, false, LEV_MODE_FINAL, 4, false, false, true, true>(p, st)
                 : lev_launch_variant<float, false, LEV_MODE_FINAL, 4, false, false, true, false>(p, st);
}

// the short form (R <= 64): one lane per pair from the raw tokens
#include "lev_counts.cuh"
