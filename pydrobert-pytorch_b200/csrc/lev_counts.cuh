// lev_counts.cuh -- b200lev_error_counts, short form (padded reference length R <= 64): per pair
// the correct / substitution / deletion / insertion counts (sclite's C/S/D/I) along the path the
// count mode of error_rate picks (SM:292-314), one LANE per pair.
//
// The path.  Every cell takes one predecessor with the tie-breaks of SM:296 and SM:309: the
// substitution candidate (diag + sub * [ref != hyp]) unless the insertion candidate (up + ins) is
// smaller, then the deletion candidate (left + del) only if it is smaller still.  The cell
// inherits that predecessor's op counts plus one op.  Because C + S + D = j and C + S + I = i hold
// in cell (i, j), two numbers per cell are enough: the op word (I << 8) | S (S <= r <= 64, I <= h
// < 2^24), from which D = I + j - i and C = i - S - I.  A substitution adds [ref != hyp] to the
// word, an insertion 1 << 8, a deletion nothing.
//
// Layout as in lev_bvshort.cu: lane l of a warp serves pair 32 w + l, reads its reference column
// into registers (the low words of the tokens; positions past R repeat R - 1) and its hypothesis
// one coalesced row at a time, straight from the raw (T, N) tensors -- no K0, no bucketing, no
// workspace.  Costs and DP row live in registers (int32 cells for integer costs, fp32 in the
// count-mode operation order otherwise).  A reference token outside int32 anywhere in the warp
// sends the warp to an exact 64-bit compare against the (cached) column, one match mask per
// hypothesis token; a hypothesis token outside int32 equals no reference token of a warp that
// takes the fast path.
//
// TRACE (b200lev_error_alignment): each row also packs its cells' choices as 2-bit op codes
// (lev_align.cuh) into RM / 16 words, stored [row][word][pair]; after the last row the lane walks
// its own trace back from (h, r) and writes the ops instead of the counts.
//
// Compiled as part of lev_dp.cu (included once, at its end), next to the long form.
#pragma once
#include "lev_arith.cuh"

constexpr int LEV_CNT_WARPS = 4;

struct LevCountsArgs {
    const void* ref;
    const void* hyp;
    int64_t ref_st, ref_sn, hyp_st, hyp_sn;
    int64_t P;
    int R, H;
    int has_eos, include_eos;
    int64_t eos;
    int ins_i, del_i, sub_i;
    float ins_f, del_f, sub_f;
    int64_t* out;   // [P][4]
    int32_t* flags;  // may be NULL
};
// TRACE: the choice rows ([H][RM / 16][P] words) and the ops (step k of pair n at
// ops[k*ops_sk + n*ops_sn], k < Tout = R + H)
struct LevAlignArgs : LevCountsArgs {
    uint32_t* trace;
    int8_t* ops;
    int64_t ops_sk, ops_sn;
    int Tout;
};

template <typename V>
struct LevCountCost;
template <>
struct LevCountCost<int> {
    static __device__ __forceinline__ int ins(const LevCountsArgs& a) { return a.ins_i; }
    static __device__ __forceinline__ int del(const LevCountsArgs& a) { return a.del_i; }
    static __device__ __forceinline__ int sub(const LevCountsArgs& a) { return a.sub_i; }
};
template <>
struct LevCountCost<float> {
    static __device__ __forceinline__ float ins(const LevCountsArgs& a) { return a.ins_f; }
    static __device__ __forceinline__ float del(const LevCountsArgs& a) { return a.del_f; }
    static __device__ __forceinline__ float sub(const LevCountsArgs& a) { return a.sub_f; }
};

template <bool EXACT>
struct LevCntPath {
    static constexpr bool value = EXACT;
};
// TRACE: the path tag also carries where the next row's choice words go (the lambdas below name
// no other state for the trace, so the instantiations without it stay as they were)
template <bool EXACT>
struct LevCntTracePath {
    static constexpr bool value = EXACT;
    uint32_t* row;  // word 0 of the next row; word k at row[k * P]
};
template <bool TRACE, int NW>
struct LevRowTrace {
    unsigned w[NW] = {};
};
template <int NW>
struct LevRowTrace<false, NW> {};

template <typename TT, typename V, int RM, bool TRACE = false>
__global__ void __launch_bounds__(32 * LEV_CNT_WARPS)
    lev_counts_short_kernel(const typename std::conditional<TRACE, LevAlignArgs, LevCountsArgs>::type a) {
    constexpr int NW = RM / 16;  // TRACE: words per row
    constexpr bool IS_INT = std::is_same<V, int>::value;
    const int lane = threadIdx.x & 31;
    const int64_t nblocks = (a.P + 31) / 32;
    const int R = a.R, H = a.H;
    const V ins = LevCountCost<V>::ins(a), del = LevCountCost<V>::del(a), sub = LevCountCost<V>::sub(a);
    for (int64_t block = (int64_t)blockIdx.x * LEV_CNT_WARPS + (threadIdx.x >> 5); block < nblocks;
         block += (int64_t)gridDim.x * LEV_CNT_WARPS) {
        // lanes past the batch shadow its last pair (they compute the same values, store nothing)
        const int64_t pair = block * 32 + lane;
        const int64_t pc = pair < a.P ? pair : a.P - 1;
        const TT* __restrict__ rsrc = reinterpret_cast<const TT*>(a.ref) + pc * a.ref_sn;
        const TT* __restrict__ hsrc = reinterpret_cast<const TT*>(a.hyp) + pc * a.hyp_sn;

        // ---- reference column -> registers, its first eos, does it leave int32 --------------
        int rt[RM];
        int first_eos = R;
        bool wide = false;
        {
            constexpr int RB = 8;  // loads issued back to back, then consumed
            const TT* __restrict__ rp = rsrc;
#pragma unroll
            for (int j0 = 0; j0 < RM; j0 += RB) {
                if (j0 < R) {  // (warp-uniform)
                    TT raw[RB];
#pragma unroll
                    for (int k = 0; k < RB; ++k) {
                        raw[k] = *rp;
                        if (j0 + k < R - 1) rp += a.ref_st;
                    }
#pragma unroll
                    for (int k = 0; k < RB; ++k) {
                        const int64_t x = (int64_t)raw[k];
                        rt[j0 + k] = (int)x;
                        if (sizeof(TT) == 8) wide |= x != (int64_t)(int)x;
                        if (a.has_eos && x == a.eos && first_eos == R) first_eos = j0 + k;
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < RB; ++k) rt[j0 + k] = 0;
                }
            }
        }
        // SM:195-228
        const int rlen = first_eos < R ? first_eos + (a.include_eos ? 1 : 0) : R;
        int myflags = (a.has_eos && a.include_eos && first_eos == R) ? B200LEV_FLAG_REF_NO_EOS : 0;

        // ---- row 0: j deletions --------------------------------------------------------------
        V v[RM + 1];
        unsigned w[RM + 1];  // (I << 8) | S
#pragma unroll
        for (int j = 0; j <= RM; ++j) {
            v[j] = (V)j * del;
            w[j] = 0u;
        }
        int hlen = 0;
        bool live = true;  // no eos seen yet

        // one hypothesis row: SM:292-314 for every column, the op word alongside
        auto row = [&](auto path, const int64_t x) {
            constexpr bool EXACT = decltype(path)::value;
            const unsigned nlo = 0u - (unsigned)(int)x;
            // (fast path, 64-bit tokens: a hypothesis token outside int32 matches nothing)
            const unsigned bad = (sizeof(TT) == 8 && !EXACT && x != (int64_t)(int)x) ? 1u : 0u;
            // exact path: the positions of the column that hold x, compared in 64 bits (a rolled
            // loop: nothing of the column stays in registers)
            unsigned long long eqm = 0ull;
            if (EXACT) {
                const TT* __restrict__ rp = rsrc;
#pragma unroll 1
                for (int j = 0; j < R; ++j) {
                    eqm |= (int64_t)*rp == x ? 1ull << j : 0ull;
                    rp += a.ref_st;
                }
            }
            V diag = v[0];
            unsigned dw = w[0];
            v[0] = v[0] + ins;  // column 0: one more insertion
            w[0] = w[0] + 256u;
            V left = v[0];
            unsigned lw = w[0];
            LevRowTrace<TRACE, NW> tr;  // TRACE: this row's choices
            (void)tr;
#pragma unroll
            for (int j = 1; j <= RM; ++j) {
                unsigned neq;
                if (EXACT)
                    neq = (unsigned)(~eqm >> (j - 1)) & 1u;
                else
                    neq = __viaddmin_u32((unsigned)rt[j - 1], nlo, 1u) | bad;
                const V up = v[j];
                const unsigned uw = w[j];
                const V sub_c = IS_INT ? diag + (V)(int)neq * sub : diag + (neq ? sub : (V)0);  // SM:293
                const V ins_c = up + ins;                                                       // SM:292
                const bool ps = ins_c >= sub_c;                                                 // SM:296
                V c = ps ? sub_c : ins_c;
                unsigned cw = ps ? dw + neq : uw + 256u;
                const V del_c = left + del;  // SM:308
                const bool keep = del_c >= c;  // SM:309
                c = keep ? c : del_c;
                cw = keep ? cw : lw;
                if constexpr (TRACE) tr.w[(j - 1) >> 4] |= (keep ? (ps ? neq : 3u) : 2u) << (2 * ((j - 1) & 15));
                diag = up;
                dw = uw;
                left = c;
                lw = cw;
                v[j] = c;
                w[j] = cw;
            }
            if constexpr (TRACE) {
                if (path.row != nullptr) {  // (NULL: a lane past the batch)
#pragma unroll
                    for (int k = 0; k < NW; ++k) path.row[(int64_t)k * a.P] = tr.w[k];
                }
            }
        };
        // the hypothesis, CH rows per trip: the CH loads go out together
        auto hypothesis = [&](auto path) {
            constexpr int CH = 4;
            const TT* __restrict__ hp = hsrc;
            for (int t0 = 0; t0 < H; t0 += CH) {  // (warp-uniform)
                TT buf[CH];
#pragma unroll
                for (int k = 0; k < CH; ++k) {
                    buf[k] = (TT)0;
                    if (t0 + k < H) {
                        // (1-byte tokens: a plain load; the streaming one costs this kernel a spill)
                        buf[k] = sizeof(TT) == 1 ? *hp : lev_ldg_stream(hp);
                        hp += a.hyp_st;
                    }
                }
#pragma unroll
                for (int k = 0; k < CH; ++k) {
                    const int64_t x = (int64_t)buf[k];
                    const bool is_eos = a.has_eos && x == a.eos;
                    const bool in = t0 + k < H && live && (!is_eos || a.include_eos);
                    live = live && !(t0 + k < H && is_eos);
                    if (in) {
                        ++hlen;
                        row(path, x);
                        if constexpr (TRACE) {
                            if (path.row != nullptr) path.row += (int64_t)NW * a.P;
                        }
                    }
                }
                if (!__any_sync(LEV_FULL_MASK, live)) break;  // every hypothesis of the warp ended
            }
        };
        bool exact = false;
        if (sizeof(TT) == 8) exact = __any_sync(LEV_FULL_MASK, wide);
        if constexpr (TRACE) {
            uint32_t* const row0 = pair < a.P ? a.trace + pair : nullptr;
            if (exact)
                hypothesis(LevCntTracePath<true>{row0});
            else
                hypothesis(LevCntTracePath<false>{row0});
        } else {
            if (exact)
                hypothesis(LevCntPath<true>{});
            else
                hypothesis(LevCntPath<false>{});
        }
        if (a.has_eos && a.include_eos && live) myflags |= B200LEV_FLAG_HYP_NO_EOS;

        // ---- cell (h, r) ---------------------------------------------------------------------
        unsigned wf = 0u;
#pragma unroll
        for (int j = 0; j <= RM; ++j) wf = j == rlen ? w[j] : wf;
        const int ni = (int)(wf >> 8), ns = (int)(wf & 255u);
        const int nd = ni + rlen - hlen;
        if constexpr (TRACE) {
            if (pair < a.P) {
                LevTraceRows t;
                t.base = a.trace + pair;
                t.row_stride = (int64_t)NW * a.P;
                t.word_stride = a.P;
                lev_align_walk(t, hlen, rlen, rlen + ni, a.Tout, a.ops + pair * a.ops_sn, a.ops_sk);
            }
        } else if (pair < a.P) {
            int64_t* __restrict__ o = a.out + pair * 4;
            o[0] = hlen - ns - ni;
            o[1] = ns;
            o[2] = nd;
            o[3] = ni;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) myflags |= __shfl_xor_sync(LEV_FULL_MASK, myflags, d);
        if (lane == 0 && myflags != 0 && a.flags != nullptr) atomicOr(a.flags, myflags);
    }
}

// ---- host side ---------------------------------------------------------------------------------
template <typename TT, typename V, bool TRACE>
static void lev_counts_launch_t(const LevAlignArgs& a_, cudaStream_t st) {
    const typename std::conditional<TRACE, LevAlignArgs, LevCountsArgs>::type& a = a_;
    const int64_t n = (a.P + 32 * LEV_CNT_WARPS - 1) / (32 * LEV_CNT_WARPS);
    const int64_t cap = (int64_t)148 * 16;
    const dim3 grid((unsigned)(n < cap ? n : cap)), block(32 * LEV_CNT_WARPS);
    if (a.R <= 32)
        lev_launch(lev_counts_short_kernel<TT, V, 32, TRACE>, grid, block, 0, st, a);
    else
        lev_launch(lev_counts_short_kernel<TT, V, 64, TRACE>, grid, block, 0, st, a);
}

template <typename TT>
static void lev_counts_launch_tt(const LevAlignArgs& a, bool float_path, bool trace, cudaStream_t st) {
    if (trace) {
        if (float_path)
            lev_counts_launch_t<TT, float, true>(a, st);
        else
            lev_counts_launch_t<TT, int, true>(a, st);
    } else {
        if (float_path)
            lev_counts_launch_t<TT, float, false>(a, st);
        else
            lev_counts_launch_t<TT, int, false>(a, st);
    }
}

// both entry points: the counts to p.counts, or (p.ops set) the choice rows to p.trace and the ops
int lev_counts_short_launch(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                            const b200lev_opts_t* o, const LevParams& p, bool float_path,
                            cudaStream_t st) {
    if (ref->T > 64) {
        lev_set_error("short error-counts form: R = %lld > 64", (long long)ref->T);
        return B200LEV_ERR_ARG;
    }
    if (ref->elem_bytes != hyp->elem_bytes) {  // (the long form takes those)
        lev_set_error("short error-counts form: token widths differ (%d, %d bytes)", ref->elem_bytes,
                      hyp->elem_bytes);
        return B200LEV_ERR_ARG;
    }
    LevAlignArgs a;
    memset(&a, 0, sizeof(a));
    a.ref = ref->data;
    a.hyp = hyp->data;
    a.ref_st = ref->stride_t;
    a.ref_sn = ref->stride_n;
    a.hyp_st = hyp->stride_t;
    a.hyp_sn = hyp->stride_n;
    a.P = hyp->N;
    a.R = (int)ref->T;
    a.H = (int)hyp->T;
    a.has_eos = o->has_eos;
    a.include_eos = o->include_eos;
    a.eos = o->eos;
    a.ins_i = p.ins_i;
    a.del_i = p.del_i;
    a.sub_i = p.sub_i;
    a.ins_f = p.ins_f;
    a.del_f = p.del_f;
    a.sub_f = p.sub_f;
    a.flags = p.flags;
    a.out = p.counts;
    a.trace = reinterpret_cast<uint32_t*>(p.trace);
    a.ops = p.ops;
    a.ops_sk = p.ops_sk;
    a.ops_sn = p.ops_sn;
    a.Tout = p.ops_steps;
    const bool trace = p.ops != nullptr;
    lev_prof_begin(LEV_PROF_DP, st);
    switch (ref->elem_bytes) {
        case 8: lev_counts_launch_tt<int64_t>(a, float_path, trace, st); break;
        case 4: lev_counts_launch_tt<int32_t>(a, float_path, trace, st); break;
        case 2: lev_counts_launch_tt<int16_t>(a, float_path, trace, st); break;
        case 1: lev_counts_launch_tt<int8_t>(a, float_path, trace, st); break;
        default:
            lev_set_error("token width %d bytes", ref->elem_bytes);
            return B200LEV_ERR_ARG;
    }
    lev_prof_end(LEV_PROF_DP, st);
    return lev_check_cuda("lev_counts_short_kernel");
}
